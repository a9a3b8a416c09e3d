"""The fused detect path with cross-check matching (cvg_detect_params.method | CVG_MATCH_CROSS_CHECK): the correspondences
of every pair are BFMatcher(NORM_L2, crossCheck=True).match's, each view its own query matrix, then the geometric check of
the method, the gates and the inlier gather as with the ratio test.

Against cv2 4.13.0 on the 890 real (view, scaled scene) pairs of features_small.npz (golden_detect_crosscheck.npz, written
by tests/golden/make_golden_detect_crosscheck.py): status, counts, the bytes of H, det and the inlier scene points exactly.
Against the standalone calls (match_cross_check, then the batch estimators) on the same correspondences: iterations, masks
and found exactly, H / M bit-equal wherever both pick the same finish block size or at most 128 inliers are refined (the
rule of test_gpu_detect_verify.py), else within 4e-8 relative."""
import os

import numpy as np
import pytest

from affine_partial_cases import same_bytes

from computervision_objectdetection_featurematching_b200 import synth

pytestmark = pytest.mark.gpu

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
METHODS = ("homography", "affine", "partial")
UNPINNED_REL = 4e-8
EXACT_MAX_INLIERS = 128
# status histograms [accept, lt4 matches, H empty, lt4 inliers, det reject] of the 890 real pairs under cv2, cross-check
HIST = {"homography": [117, 0, 0, 41, 732], "affine": [609, 0, 0, 20, 261], "partial": [473, 0, 0, 268, 149]}
# findHomography's H on three real pairs (2, 3 and 6 RANSAC inliers; all rejected by the gates) is not cv2's bit for bit:
# the refit / LM on so few points is ill-conditioned and differs from cv2 by at most 8.4e-11 relative (B200)
HOMOGRAPHY_MAX_UNPINNED = 3
HOMOGRAPHY_REL = 1e-9


@pytest.fixture(scope="module")
def api():
    from computervision_objectdetection_featurematching_b200 import api as _api
    return _api


def _method(api, name):
    return {"homography": api.VERIFY_HOMOGRAPHY, "affine": api.VERIFY_AFFINE, "partial": api.VERIFY_AFFINE_PARTIAL}[name]


def _params(api, name, cross_check=True, **kw):
    """the goldens' parameters: the reference's for homography, (3.0, 2000, 0.99, refineIters 10) for the affine methods"""
    if name == "homography":
        return api.detect_params(cross_check=cross_check, **kw)
    return api.detect_params(ransac=api.ransac_params(3.0, 2000, 0.99), method=_method(api, name), refine_iters=10,
                             cross_check=cross_check, **kw)


def _open_gates(api, name):
    return _params(api, name, min_inliers=0, det_lo=0.0, det_hi=float("inf"))


def _block(max_n):
    return 64 if max_n <= 512 else 128              # the finish kernels' block size (ransac.cu)


def _standalone(ctx, name, src, dst, off):
    """-> found [P], model [P, 9] (M promoted to 3x3), mask, iters"""
    if name == "homography":
        r = ctx.find_homography_batch(src, dst, off)
        return r["found"], r["H"].reshape(-1, 9), r["mask"], r["iters"]
    fn = ctx.estimate_affine2d_batch if name == "affine" else ctx.estimate_affine_partial2d_batch
    r = fn(src, dst, off, threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10)
    P = len(off) - 1
    H = np.zeros((P, 9)); H[:, :6] = r["M"].reshape(P, 6); H[r["found"], 8] = 1.0     # as the fused path promotes M
    return r["found"], H, r["mask"], r["iters"]


class Real:
    """features_small.npz on one context: the model views, the ten scaled scenes resident, their scales."""

    def __init__(self, ctx, feats):
        self.feats = feats
        self.so = feats["scene_offsets"]; self.vo = feats["view_offsets"]
        self.scales = np.tile(feats["scales"], (len(self.so) - 1) // len(feats["scales"])).astype(np.float32)
        self.models = ctx.upload_models(feats["model_desc"].astype(np.float32), feats["model_kpt"], self.vo,
                                        feats["view_model"])
        self.scenes = ctx.upload_scenes(feats["scene_desc"].astype(np.float32), feats["scene_kpt"], self.so)

    def scene(self, s):
        a, b = self.so[s], self.so[s + 1]
        return self.feats["scene_desc"][a:b].astype(np.float32), self.feats["scene_kpt"][a:b].astype(np.float32)

    def free(self):
        self.scenes.free(); self.models.free()


@pytest.fixture(scope="module")
def ctx(api):
    with api.Context(0) as c:
        yield c


@pytest.fixture(scope="module")
def real(ctx, feats):
    r = Real(ctx, feats)
    yield r
    r.free()


@pytest.fixture(scope="module")
def golden():
    return dict(np.load(os.path.join(GOLDEN_DIR, "golden_detect_crosscheck.npz")))


def _sets(feats, idx_of_pair):
    """(src, dst, offsets) of the mutual matches, pair after pair (scene-major); idx_of_pair(s, v) -> train index per row"""
    mk = feats["model_kpt"].astype(np.float32); sk = feats["scene_kpt"].astype(np.float32)
    vo = feats["view_offsets"]; so = feats["scene_offsets"]
    src, dst, off = [], [], [0]
    for s in range(len(so) - 1):
        for v in range(len(vo) - 1):
            idx = idx_of_pair(s, v)
            sel = np.nonzero(idx >= 0)[0]
            src.append(mk[vo[v]:vo[v + 1]][sel]); dst.append(sk[so[s]:so[s + 1]][idx[sel]]); off.append(off[-1] + len(sel))
    return np.concatenate(src), np.concatenate(dst), np.asarray(off, np.int64)


@pytest.fixture(scope="module")
def cv2_sets(feats):
    """cv2's cross-check correspondences of the real pairs (golden_crosscheck.npz, real group)"""
    G = np.load(os.path.join(GOLDEN_DIR, "golden_crosscheck.npz"))
    ro, ri = G["real_offsets"], G["real_idx"]
    V = len(feats["view_offsets"]) - 1
    return _sets(feats, lambda s, v: ri[ro[s * V + v]:ro[s * V + v + 1]])


@pytest.fixture(scope="module")
def gpu_sets(ctx, real, feats):
    """the same from the standalone call, match_cross_check(view = -1) per scene"""
    per_scene = [ctx.match_cross_check(real.models, real.scene(s)[0], view=-1)[0] for s in range(len(real.so) - 1)]
    vo = feats["view_offsets"]
    return _sets(feats, lambda s, v: per_scene[s][vo[v]:vo[v + 1]])


# ---------------------------------------------------------------- against cv2
@pytest.mark.parametrize("name", METHODS)
def test_real_pairs_against_cv2(api, ctx, real, golden, cv2_sets, name):
    _, dst, soff = cv2_sets
    assert np.array_equal(soff, golden["offsets"])
    n = np.diff(soff)
    found = golden[f"{name}_found"]; model = golden[f"{name}_model"]; det = golden[f"{name}_det"]
    mask = np.unpackbits(golden[f"{name}_mask"], count=int(soff[-1])).astype(bool)
    P = len(n)
    H = np.zeros((P, 9)); status = np.zeros(P, np.int32); n_inl = np.zeros(P, np.int32)
    lo, hi = float(np.float32(0.1)), float(np.float32(10.0))
    for k in range(P):
        if found[k]:
            H[k, :model.shape[1]] = model[k]
            if model.shape[1] == 6:
                H[k, 8] = 1.0                                   # M promoted to 3x3 (findHomography's H[2,2] is its own)
            n_inl[k] = mask[soff[k]:soff[k + 1]].sum()
        status[k] = 1 if n[k] < 4 else (2 if not found[k] else (3 if n_inl[k] < 4 else (4 if not lo <= abs(det[k]) <= hi else 0)))
    assert np.bincount(status, minlength=5).tolist() == HIST[name]
    res, xy, off = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=_params(api, name))
    assert ctx.last_match_path == api.PATH_TENSOR
    r = res.ravel()
    assert np.bincount(r["status"], minlength=5).tolist() == HIST[name]
    assert np.array_equal(r["status"], status)
    assert np.array_equal(r["n_good"], n)
    assert np.array_equal(r["n_inliers"], n_inl)
    if name == "homography":
        # findHomography's LM accepts or rejects a step on rounding noise near convergence (DESIGN.md 3, 6): H is cv2's bit
        # for bit on all but a few pairs, and within HOMOGRAPHY_REL elsewhere; the masks above are exact all the same
        same = np.all(r["H"] == H, axis=1)
        rel = np.max(np.abs(r["H"] - H) / np.maximum(np.abs(H), 1e-12), axis=1)
        odd = [(k, int(n_inl[k]), float(rel[k])) for k in np.nonzero(~same)[0]]
        assert len(odd) <= HOMOGRAPHY_MAX_UNPINNED and rel.max() < HOMOGRAPHY_REL, odd
        assert np.array_equal(r["det"][found & same], det[found & same])
        assert np.allclose(r["det"][found], det[found], rtol=1e-7, atol=0)
    else:
        assert r["H"].tobytes() == H.tobytes()
        assert np.array_equal(r["det"][found], det[found])
    scale = np.repeat(real.scales, len(real.vo) - 1)
    for k in range(P):
        got = xy[off[k]:off[k + 1]]
        if r["status"][k] != api.ACCEPT:
            assert len(got) == 0, k
            continue
        pts = dst[soff[k]:soff[k + 1]][mask[soff[k]:soff[k + 1]]]
        sc = np.float32(scale[k])
        if sc != np.float32(1.0):
            pts = pts / sc
        assert np.array_equal(got, pts.astype(np.float32)), k


# ---------------------------------------------------------------- against the standalone calls
def _check_vs_standalone(api, res, xy, off, std, dst, soff, fused_block):
    """a fused call with open gates and no scales against the standalone batch on the same sets; -> refined inlier counts"""
    found_s, H_s, mask_s, iters_s = std
    n = np.diff(soff)
    std_block = _block(int(n.max()) if len(n) else 0)
    assert np.array_equal(res["n_good"], n)
    found = res["H"].any(axis=1)                                # zeros when no model came back
    assert np.array_equal(found, found_s)
    assert np.array_equal(res["ransac_iters"], iters_s)
    n_refined = []
    for k in range(len(n)):
        a, b = soff[k], soff[k + 1]
        m = mask_s[a:b].astype(bool)
        if not found[k]:
            assert res["status"][k] == api.H_EMPTY and res["n_inliers"][k] == 0 and not res["H"][k].any(), k
            assert off[k + 1] == off[k], k
            continue
        assert res["status"][k] == api.ACCEPT, k
        assert res["n_inliers"][k] == m.sum(), k
        assert np.array_equal(xy[off[k]:off[k + 1]], dst[a:b][m]), k
        if fused_block == std_block or m.sum() <= EXACT_MAX_INLIERS:
            assert same_bytes(res["H"][k], H_s[k]), (k, int(m.sum()))
        else:
            rel = np.abs(res["H"][k] - H_s[k]) / np.maximum(np.abs(H_s[k]), 1e-12)
            assert np.max(rel) < UNPINNED_REL, k
        n_refined.append(int(m.sum()))
    return n_refined


def test_standalone_match_is_cv2s(cv2_sets, gpu_sets):
    for a, b in zip(cv2_sets, gpu_sets):
        assert np.array_equal(a, b)


@pytest.mark.parametrize("name", METHODS)
def test_real_pairs_equal_standalone(api, ctx, real, gpu_sets, name):
    src, dst, soff = gpu_sets
    std = _standalone(ctx, name, src, dst, soff)
    res, xy, off = ctx.detect_scenes_inliers(real.models, real.scenes, params=_open_gates(api, name))
    _check_vs_standalone(api, res.ravel(), xy, off, std, dst, soff, _block(int(np.diff(real.vo).max())))


def _synthetic_8192(n_scenes=4, n=8192, seed=78):
    """one model view of n SIFT-like rows against n_scenes scenes of n rows: half the queries planted in every scene, 40 %
    of those placed by a homography-like map (0.7 px noise)"""
    rng = np.random.default_rng(seed)
    q = synth.sift_like(rng, n)
    qk = rng.uniform([0, 0], [640, 480], size=(n, 2)).astype(np.float32)
    descs, kpts = [], []
    for s in range(n_scenes):
        t = synth.sift_like(rng, n)
        tk = rng.uniform([0, 0], [640, 480], size=(n, 2)).astype(np.float32)
        k = n // 2
        rq = rng.permutation(n)[:k]; rt = rng.permutation(n)[:k]
        t[rt] = np.clip(q[rq] + np.round(rng.normal(0, 12.0, size=(k, 128))).astype(np.float32), 0, 255)
        A = np.array([[1 + rng.normal(0, .1), rng.normal(0, .1), rng.normal(0, 30)],
                      [rng.normal(0, .1), 1 + rng.normal(0, .1), rng.normal(0, 30)]])
        geo = rng.random(k) < 0.4
        tk[rt[geo]] = (np.c_[qk[rq[geo]], np.ones(int(geo.sum()))] @ A.T
                       + rng.normal(0, 0.7, size=(int(geo.sum()), 2))).astype(np.float32)
        descs.append(t); kpts.append(tk)
    return q, qk, np.concatenate(descs), np.concatenate(kpts), np.arange(n_scenes + 1, dtype=np.int64) * n


@pytest.fixture(scope="module")
def synth8192(ctx):
    q, qk, d, k, so = _synthetic_8192()
    models = ctx.upload_models(q, qk, [0, len(q)], [0])
    scenes = ctx.upload_scenes(d, k, so)
    src, dst, offs = [], [], [0]
    for s in range(len(so) - 1):
        idx, _ = ctx.match_cross_check(models, d[so[s]:so[s + 1]], view=0)
        sel = np.nonzero(idx >= 0)[0]
        src.append(qk[sel]); dst.append(k[so[s]:so[s + 1]][idx[sel]]); offs.append(offs[-1] + len(sel))
    yield models, scenes, np.concatenate(src), np.concatenate(dst), np.asarray(offs, np.int64)
    scenes.free(); models.free()


@pytest.mark.parametrize("name", METHODS)
def test_synthetic_8192_equals_standalone(api, ctx, synth8192, name):
    models, scenes, src, dst, soff = synth8192
    res, xy, off = ctx.detect_scenes_inliers(models, scenes, params=_open_gates(api, name))
    res = res.ravel()
    assert np.diff(soff).min() > 512                            # the block-reduction refine of the finish kernels
    std = _standalone(ctx, name, src, dst, soff)
    n_refined = _check_vs_standalone(api, res, xy, off, std, dst, soff, _block(8192))
    assert len(n_refined) == len(soff) - 1 and max(n_refined) > EXACT_MAX_INLIERS


# ---------------------------------------------------------------- every path, the same bytes
def _run_paths(api, ctx, feats, p, n_devices_visible):
    real = Real(ctx, feats)
    try:
        ref = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=p)
        outs = {"detect_scenes": (ctx.detect_scenes(real.models, real.scenes, scales=real.scales, params=p), None, None)}
        rs, xs, cnt = [], [], []
        for s in range(len(real.so) - 1):
            t, k = real.scene(s)
            r, x, o = ctx.detect_pairs(real.models, t, k, scale=float(real.scales[s]), params=p)
            rs.append(r); xs.append(x); cnt.append(np.diff(o))
        outs["detect_pairs"] = (np.stack(rs), np.concatenate(xs), np.r_[0, np.cumsum(np.concatenate(cnt))])
        jobs = [ctx.submit_scenes(real.models, real.scenes, scales=real.scales, params=p) for _ in range(3)]
        for i, j in enumerate(jobs):
            outs[f"submit_{i}"] = j.wait()
        ctx.set_lanes(1)
        outs["lanes_1"] = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=p)
        ctx.set_lanes(0)
        u8 = ctx.upload_scenes_u8_async(feats["scene_desc"], feats["scene_kpt"], real.so)
        outs["u8"] = ctx.detect_scenes_inliers(real.models, u8, scales=real.scales, params=p)
        u8.free()
    finally:
        real.free()
    devs = [[0, 0], [0, 0, 0]] + ([[0, 1]] if n_devices_visible >= 2 else [])
    for d in devs:
        with api.Context(d) as mc:
            r = Real(mc, feats)
            outs[f"multi_{d}"] = mc.detect_scenes_inliers(r.models, r.scenes, scales=real.scales, params=p)
            outs[f"multi_submit_{d}"] = mc.submit_scenes(r.models, r.scenes, scales=real.scales, params=p).wait()
            r.free()
    return ref, outs


@pytest.mark.parametrize("name", METHODS)
def test_every_path_same_bytes(api, feats, name):
    import torch
    with api.Context(0) as c:
        ref, outs = _run_paths(api, c, feats, _params(api, name), torch.cuda.device_count())
    r0, x0, o0 = ref
    assert np.bincount(r0["status"].ravel(), minlength=5).tolist() == HIST[name]
    for key, (r, x, o) in outs.items():
        assert r.tobytes() == r0.tobytes(), key
        if x is not None:
            assert np.array_equal(x, x0) and np.array_equal(np.asarray(o, np.int64), o0), key


# ---------------------------------------------------------------- guard and paths
def test_guard_rows_on_saturated_rows(api, ctx):
    """golden_sat.npz's u8 rows: every distance is above 2048, so the tensor path redoes rows and columns exactly"""
    Z = np.load(os.path.join(GOLDEN_DIR, "golden_sat.npz"))
    G = np.load(os.path.join(GOLDEN_DIR, "golden_crosscheck.npz"))
    q, t = Z["q"].astype(np.float32), Z["t"].astype(np.float32)
    rng = np.random.default_rng(5)
    qk = rng.uniform(0, 640, (len(q), 2)).astype(np.float32); tk = rng.uniform(0, 640, (len(t), 2)).astype(np.float32)
    models = ctx.upload_models(q, qk, [0, len(q)], [0])
    res, _, _ = ctx.detect_pairs(models, t, tk, params=api.detect_params(cross_check=True))
    assert ctx.last_match_path == api.PATH_TENSOR and ctx.last_match_guard_rows > 0
    assert res["n_good"][0] == int((G["sat_idx"] >= 0).sum())
    models.free()


def test_float_rows_and_forced_exact_path(api, ctx, real, feats):
    rng = np.random.default_rng(11)
    q = synth.float_desc(rng, 400); t = synth.float_desc(rng, 900)
    qk = rng.uniform(0, 640, (400, 2)).astype(np.float32); tk = rng.uniform(0, 640, (900, 2)).astype(np.float32)
    t[rng.permutation(900)[:300]] = q[:300] + rng.normal(0, 3, (300, 128)).astype(np.float32)
    vo = [0, 150, 400]
    models = ctx.upload_models(q, qk, vo, [0, 0])
    for name in METHODS:
        res, xy, off = ctx.detect_pairs(models, t, tk, params=_open_gates(api, name))
        assert ctx.last_match_path == api.PATH_EXACT
        src, dst, soff = [], [], [0]
        for v in range(2):
            idx, _ = ctx.match_cross_check(models, t, view=v)
            sel = np.nonzero(idx >= 0)[0]
            src.append(qk[vo[v]:vo[v + 1]][sel]); dst.append(tk[idx[sel]]); soff.append(soff[-1] + len(sel))
        src, dst, soff = np.concatenate(src), np.concatenate(dst), np.asarray(soff, np.int64)
        assert soff[-1] > 0
        std = _standalone(ctx, name, src, dst, soff)
        _check_vs_standalone(api, res, xy, off, std, dst, soff, _block(250))
    models.free()
    # CVG_FORCE_EXACT_MATCH on SIFT rows: the SIMT kernel, cv2's bytes all the same
    ref = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=_params(api, "affine"))
    with api.Context(0, flags=api.FORCE_EXACT_MATCH) as fc:
        fc.set_lanes(1)
        r = Real(fc, feats)
        got = fc.detect_scenes_inliers(r.models, r.scenes, scales=r.scales, params=_params(api, "affine"))
        assert fc.last_match_path == api.PATH_EXACT
        r.free()
    assert got[0].tobytes() == ref[0].tobytes() and np.array_equal(got[1], ref[1])


def test_empty_views_empty_and_tiny_scenes(api, ctx):
    rng = np.random.default_rng(21)
    q = synth.sift_like(rng, 300); qk = rng.uniform(0, 640, (300, 2)).astype(np.float32)
    t = synth.sift_like(rng, 700); tk = rng.uniform(0, 640, (700, 2)).astype(np.float32)
    t[:200] = q[100:300]
    vo = [0, 0, 120, 120, 300]                                   # views 0 and 2 have no rows
    so = np.array([0, 0, 1, 2, 700], np.int64)                  # an empty scene, two 1-row scenes, a full one
    models = ctx.upload_models(q, qk, vo, [0, 0, 0, 0])
    scenes = ctx.upload_scenes(t, tk, so)
    for name in METHODS:
        p = _params(api, name)
        res = ctx.detect_scenes(models, scenes, params=p)
        for s in range(len(so) - 1):
            ts, ks = t[so[s]:so[s + 1]], tk[so[s]:so[s + 1]]
            for v in range(len(vo) - 1):
                if vo[v + 1] > vo[v]:
                    idx, _ = ctx.match_cross_check(models, ts, view=v)
                    assert res["n_good"][s, v] == int((idx >= 0).sum()), (name, s, v)
                else:
                    assert res["n_good"][s, v] == 0 and res["status"][s, v] == api.LT4_MATCHES
            if len(ts):
                one, _, _ = ctx.detect_pairs(models, ts, ks, params=p)
                assert one.tobytes() == res[s].tobytes(), (name, s)
        assert res["n_good"][0].sum() == 0 and res["n_good"][3, 3] == 180 and res["n_good"][1, 1] == 1
    scenes.free(); models.free()


def test_views_of_exactly_the_model_points(api, ctx):
    """views with exactly 4 / 3 / 2 mutual matches: the smallest sets each method fits"""
    rng = np.random.default_rng(31)
    t = synth.sift_like(rng, 600)
    tk = rng.uniform([0, 0], [640, 480], size=(600, 2)).astype(np.float32)
    rows = rng.permutation(600)[:9]
    q = t[rows].copy()                                          # exact copies: mutual nearest neighbours
    qk = rng.uniform([0, 0], [640, 480], size=(9, 2)).astype(np.float32)
    vo = [0, 4, 7, 9]                                           # 4, 3 and 2 mutual matches
    models = ctx.upload_models(q, qk, vo, [0, 0, 0])
    for name, mp in (("homography", 4), ("affine", 3), ("partial", 2)):
        res, xy, off = ctx.detect_pairs(models, t, tk, params=_params(api, name, min_inliers=mp, det_lo=0.0,
                                                                      det_hi=float("inf")))
        assert res["n_good"].tolist() == [4, 3, 2]
        for v in range(3):
            a, b = vo[v], vo[v + 1]
            if b - a < mp:
                assert res["status"][v] == api.LT4_MATCHES and not res["H"][v].any()
                continue
            if name == "homography":
                M, mask = ctx.find_homography(qk[a:b], tk[rows[a:b]])
            else:
                fn = ctx.estimate_affine2d if name == "affine" else ctx.estimate_affine_partial2d
                M, mask = fn(qk[a:b], tk[rows[a:b]], threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10)
            assert M is not None and res["status"][v] == api.ACCEPT and res["n_inliers"][v] == mask.sum()
            assert same_bytes(res["H"][v][:M.size], M) and (M.size == 9 or res["H"][v][8] == 1.0)
            assert np.array_equal(xy[off[v]:off[v + 1]], tk[rows[a:b]][mask.astype(bool)])
            if b - a == mp:
                assert mask.all()
    models.free()


# ---------------------------------------------------------------- interleaving and the cached match plan
def test_interleaved_with_ratio_on_one_context(api, feats):
    """ratio -> cross-check -> ratio -> cross-check on one context and the same scene shapes, on the context's own engine
    and across a lane split: no call is served the other mode's match plan"""
    seq = ("ratio", "xc", "ratio", "xc")
    p = {"ratio": _params(api, "affine", cross_check=False), "xc": _params(api, "affine")}
    fresh = {}
    for mode in ("ratio", "xc"):
        with api.Context(0) as c:
            r = Real(c, feats)
            fresh[mode] = c.detect_scenes_inliers(r.models, r.scenes, scales=r.scales, params=p[mode])
            r.free()
    assert fresh["ratio"][0].tobytes() != fresh["xc"][0].tobytes()
    with api.Context(0) as c:
        r = Real(c, feats)
        for lanes in (1, 0, 1):
            c.set_lanes(lanes)
            got = [c.detect_scenes_inliers(r.models, r.scenes, scales=r.scales, params=p[m]) for m in seq]
            for g, m in zip(got, seq):
                assert g[0].tobytes() == fresh[m][0].tobytes() and np.array_equal(g[1], fresh[m][1]), (lanes, m)
        r.free()


# ---------------------------------------------------------------- parameters and timing
def test_invalid_flags_and_ignored_ratio(api, ctx, real):
    t, k = real.scene(0)
    for method in (0x200, 0x100 | 3, 0x100 | 0xFF, 0x300, -1, 3, 0x1000):
        p = api.detect_params()
        p.method = method
        for call in (lambda: ctx.detect_scenes(real.models, real.scenes, params=p),
                     lambda: ctx.submit_scenes(real.models, real.scenes, params=p),
                     lambda: ctx.detect_pairs(real.models, t, k, params=p)):
            with pytest.raises(api.CvgError) as e:
                call()
            assert e.value.code == 1, hex(method)
    ref = ctx.detect_scenes(real.models, real.scenes, scales=real.scales, params=_params(api, "homography"))
    for ratio in (0.0, 0.5, 1.0, 7.0, -1.0, float("nan")):
        got = ctx.detect_scenes(real.models, real.scenes, scales=real.scales, params=_params(api, "homography", ratio=ratio))
        assert got.tobytes() == ref.tobytes(), ratio


def test_timing_and_path(api, feats):
    with api.Context(0) as c:
        c.set_lanes(1)
        r = Real(c, feats)
        c.set_timing(True)
        for name in METHODS:
            c.detect_scenes(r.models, r.scenes, scales=r.scales, params=_params(api, name))
            t = c.last_timing()
            assert c.last_match_path == api.PATH_TENSOR
            assert t["match_ms"] > 0 and t["total_ms"] >= t["match_ms"], name
        r.free()
