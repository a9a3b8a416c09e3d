"""The fused detect path with estimateAffine2D / estimateAffinePartial2D as its geometric check (cvg_detect_params.method).

Against cv2 4.13.0 on the 890 real (view, scaled scene) pairs of features_small.npz: the per-pair records are composed from
the committed goldens (golden_affine*.npz for M and the mask, golden_pairs.npz for the good-match counts) with the gates of
src/TestsDetector.cpp:74-94 applied in numpy, and must come back exactly: status, counts, the bytes of H (M promoted to
3x3) and the inlier scene points.  Against the standalone batch calls on the same correspondences: iterations, masks and
found exactly, M bit-equal wherever both pick the same finish block size (and at <= 128 refined inliers, where the refine
sums in one fixed order whatever the block size), else within 4e-8 relative."""
import ctypes as C
import os

import numpy as np
import pytest

import affine_cases
import affine_partial_cases
from affine_partial_cases import same_bytes

from computervision_objectdetection_featurematching_b200 import synth
from computervision_objectdetection_featurematching_b200._lib import DetectParams, RansacParams

pytestmark = pytest.mark.gpu

UNPINNED_REL = 4e-8
EXACT_MAX_INLIERS = 128                 # refines on at most this many inliers sum in one order at any block size
METHODS = ("affine", "partial")
# status histograms [accept, lt4 matches, H empty, lt4 inliers, det reject] of the 890 real pairs under cv2
HIST = {"homography": [96, 6, 9, 77, 702], "affine": [515, 6, 0, 129, 240], "partial": [219, 6, 0, 411, 254]}


@pytest.fixture(scope="module")
def api():
    from computervision_objectdetection_featurematching_b200 import api as _api
    return _api


def _method(api, name):
    return {"homography": api.VERIFY_HOMOGRAPHY, "affine": api.VERIFY_AFFINE, "partial": api.VERIFY_AFFINE_PARTIAL}[name]


def _params(api, name, **kw):
    """the goldens' parameters (3.0, 2000, 0.99, refineIters 10) for the affine methods; the reference's for homography"""
    if name == "homography":
        return api.detect_params(**kw)
    return api.detect_params(ransac=api.ransac_params(3.0, 2000, 0.99), method=_method(api, name), refine_iters=10, **kw)


def _open_gates(api, name):
    """every found model accepted: the inlier points of every pair with a model expose its whole mask"""
    return _params(api, name, min_inliers=0, det_lo=0.0, det_hi=float("inf"))


def _standalone(ctx, name, src, dst, off):
    fn = ctx.estimate_affine2d_batch if name == "affine" else ctx.estimate_affine_partial2d_batch
    return fn(src, dst, off, threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10)


def _block(max_n):
    return 64 if max_n <= 512 else 128              # the finish kernel's block size (ransac.cu, launch_affine_model)


class Real:
    """features_small.npz on one context: the model views, the ten scaled scenes resident, their scales."""

    def __init__(self, ctx, feats):
        self.feats = feats
        self.so = feats["scene_offsets"]; self.vo = feats["view_offsets"]
        self.scales = np.tile(feats["scales"], (len(self.so) - 1) // len(feats["scales"])).astype(np.float32)
        self.models = ctx.upload_models(feats["model_desc"].astype(np.float32), feats["model_kpt"], self.vo,
                                        feats["view_model"])
        self.scenes = ctx.upload_scenes(feats["scene_desc"].astype(np.float32), feats["scene_kpt"], self.so)

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
def real_sets():
    """the correspondences the fused path compacts, pair after pair (scene-major): ratio-accepted rows in query order"""
    return affine_cases.pack(affine_cases.real_sets())


def _expected(name, gpairs, scales, V):
    """cv2's record of every real pair: the goldens with the gates of :74-94 (float32 thresholds promoted to double)"""
    Z = np.load(os.path.join(affine_cases.GOLDEN_DIR, "golden_affine.npz") if name == "affine" else affine_partial_cases.GOLDEN)
    off = Z["real_offsets"]; found = Z["real_found"]; M = Z["real_M"]
    mask = np.unpackbits(Z["real_mask"], count=int(off[-1])).astype(bool)
    n = np.diff(off)
    assert np.array_equal(n, gpairs["n_good"].ravel())
    P = len(n)
    status = np.zeros(P, np.int32); n_inl = np.zeros(P, np.int32); H = np.zeros((P, 9))
    lo, hi = float(np.float32(0.1)), float(np.float32(10.0))
    for k in range(P):
        cnt = int(mask[off[k]:off[k + 1]].sum()) if found[k] else 0
        if found[k]:
            H[k, :6] = M[k]; H[k, 8] = 1.0; n_inl[k] = cnt
        if n[k] < 4:
            status[k] = 1
        elif not found[k]:
            status[k] = 2
        elif cnt < 4:
            status[k] = 3
        else:
            ad = abs(M[k, 0] * M[k, 4] - M[k, 1] * M[k, 3])
            status[k] = 4 if (ad < lo or ad > hi) else 0
    return {"status": status, "n_good": n.astype(np.int32), "n_inliers": n_inl, "H": H, "mask": mask, "off": off,
            "scale": np.repeat(scales, V)}


# ---------------------------------------------------------------- against cv2
@pytest.mark.parametrize("name", METHODS)
def test_real_pairs_against_cv2(api, ctx, real, real_sets, gpairs, name):
    V = len(real.vo) - 1
    exp = _expected(name, gpairs, real.scales, V)
    assert np.bincount(exp["status"], minlength=5).tolist() == HIST[name]
    res, xy, off = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=_params(api, name))
    r = res.ravel()
    assert np.bincount(r["status"], minlength=5).tolist() == HIST[name]
    assert np.array_equal(r["status"], exp["status"])
    assert np.array_equal(r["n_good"], exp["n_good"])
    assert np.array_equal(r["n_inliers"], exp["n_inliers"])
    assert r["H"].tobytes() == exp["H"].tobytes()
    has = exp["H"][:, 8] == 1.0
    assert np.array_equal(r["det"][has], exp["H"][has, 0] * exp["H"][has, 4] - exp["H"][has, 1] * exp["H"][has, 3])
    _, dst, soff = real_sets
    assert np.array_equal(soff, exp["off"])
    for k in range(len(r)):
        got = xy[off[k]:off[k + 1]]
        if r["status"][k] != api.ACCEPT:
            assert len(got) == 0, k
            continue
        pts = dst[soff[k]:soff[k + 1]][exp["mask"][soff[k]:soff[k + 1]]]
        sc = np.float32(exp["scale"][k])
        if sc != np.float32(1.0):
            pts = pts / sc
        assert np.array_equal(got, pts.astype(np.float32)), k
    assert (r["status"] == api.ACCEPT).sum() > 0


def test_real_pairs_homography_histogram(api, ctx, real, gpairs):
    res = ctx.detect_scenes(real.models, real.scenes, scales=real.scales)
    assert np.array_equal(res["status"], gpairs["status"].astype(np.int32))
    assert np.bincount(res["status"].ravel(), minlength=5).tolist() == HIST["homography"]


# ---------------------------------------------------------------- against the standalone batch calls
def _check_vs_standalone(api, res, xy, off, std, dst, soff, fused_block):
    """res / xy / off of a fused call with open gates and no scales against the standalone batch on the same sets"""
    n = np.diff(soff)
    std_block = _block(int(n.max()) if len(n) else 0)
    assert np.array_equal(res["n_good"], n)
    found = res["H"][:, 8] == 1.0
    assert np.array_equal(found, std["found"])
    assert np.array_equal(res["ransac_iters"], std["iters"])
    n_refined = []
    for k in range(len(n)):
        a, b = soff[k], soff[k + 1]
        m = std["mask"][a:b].astype(bool)
        if not found[k]:
            assert res["status"][k] == api.H_EMPTY and res["n_inliers"][k] == 0 and not res["H"][k].any(), k
            assert off[k + 1] == off[k], k
            continue
        assert res["status"][k] == api.ACCEPT, k
        assert res["n_inliers"][k] == m.sum(), k
        assert np.array_equal(xy[off[k]:off[k + 1]], dst[a:b][m]), k
        assert res["H"][k][6:].tolist() == [0.0, 0.0, 1.0]
        M, Ms = res["H"][k][:6], std["M"][k].ravel()
        if fused_block == std_block or m.sum() <= EXACT_MAX_INLIERS:
            assert same_bytes(M, Ms), (k, int(m.sum()))
        else:
            assert np.max(np.abs(M - Ms) / np.maximum(np.abs(Ms), 1e-12)) < UNPINNED_REL, k
        n_refined.append(int(m.sum()))
    return n_refined


@pytest.mark.parametrize("name", METHODS)
def test_real_pairs_equal_standalone_batch(api, ctx, real, real_sets, name):
    src, dst, soff = real_sets
    std = _standalone(ctx, name, src, dst, soff)
    res, xy, off = ctx.detect_scenes_inliers(real.models, real.scenes, params=_open_gates(api, name))
    _check_vs_standalone(api, res.ravel(), xy, off, std, dst, soff, _block(int(np.diff(real.vo).max())))
    # the same gates as cv2's record: what the standalone call gives, with the gates applied on the host
    res2 = ctx.detect_scenes(real.models, real.scenes, scales=real.scales, params=_params(api, name)).ravel()
    assert np.array_equal(res2["ransac_iters"], std["iters"])


def _similarity(rng):
    th = rng.uniform(-0.5, 0.5); s = np.exp(rng.normal(0, .15))
    return np.array([[s * np.cos(th), -s * np.sin(th), rng.normal(40, 20)], [s * np.sin(th), s * np.cos(th), rng.normal(30, 20)]])


def _affine(rng):
    return np.array([[1 + rng.normal(0, .1), rng.normal(0, .1), rng.normal(0, 30)],
                     [rng.normal(0, .1), 1 + rng.normal(0, .1), rng.normal(0, 30)]])


def _synthetic_8192(n_scenes=4, n=8192, seed=77):
    """one model view of n SIFT-like rows against n_scenes scenes of n rows: half the queries planted in every scene, 40 %
    of those placed by a random affine map (even scenes) or similarity (odd scenes) plus 0.7 px noise"""
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
        A = _affine(rng) if s % 2 == 0 else _similarity(rng)
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
        idx, _, acc = ctx.match_knn2(models, d[so[s]:so[s + 1]])
        sel = np.nonzero(acc)[0]
        src.append(qk[sel]); dst.append(k[so[s]:so[s + 1]][idx[sel, 0]]); offs.append(offs[-1] + len(sel))
    yield models, scenes, np.concatenate(src), np.concatenate(dst), np.asarray(offs, np.int64)
    scenes.free(); models.free()


@pytest.mark.parametrize("name", METHODS)
def test_synthetic_8192_equals_standalone_and_match(api, ctx, synth8192, name):
    models, scenes, src, dst, soff = synth8192
    res, xy, off = ctx.detect_scenes_inliers(models, scenes, params=_open_gates(api, name))
    res = res.ravel()
    assert np.array_equal(res["n_good"], np.diff(soff))          # the fused compaction keeps what match_knn2 accepts
    assert np.diff(soff).min() > 512                            # the block-reduction refine of the finish kernel
    std = _standalone(ctx, name, src, dst, soff)
    n_refined = _check_vs_standalone(api, res, xy, off, std, dst, soff, _block(8192))
    assert len(n_refined) == len(soff) - 1 and max(n_refined) > EXACT_MAX_INLIERS


# ---------------------------------------------------------------- every path, the same bytes
def _run_paths(api, ctx, feats, name, n_devices_visible):
    p = _params(api, name)
    real = Real(ctx, feats)
    try:
        ref = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=p)
        outs = {"detect_scenes": (ctx.detect_scenes(real.models, real.scenes, scales=real.scales, params=p), None, None)}
        # one scene at a time
        so = real.so; rs, xs, cnt = [], [], []
        for s in range(len(so) - 1):
            r, x, o = ctx.detect_pairs(real.models, feats["scene_desc"][so[s]:so[s + 1]].astype(np.float32),
                                       feats["scene_kpt"][so[s]:so[s + 1]], scale=float(real.scales[s]), params=p)
            rs.append(r); xs.append(x); cnt.append(np.diff(o))
        outs["detect_pairs"] = (np.stack(rs), np.concatenate(xs), np.r_[0, np.cumsum(np.concatenate(cnt))])
        jobs = [ctx.submit_scenes(real.models, real.scenes, scales=real.scales, params=p) for _ in range(3)]
        for i, j in enumerate(jobs):
            outs[f"submit_{i}"] = j.wait()
        ctx.set_lanes(1)
        outs["lanes_1"] = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales, params=p)
        ctx.set_lanes(0)
        u8 = ctx.upload_scenes_u8_async(feats["scene_desc"], feats["scene_kpt"], so)
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
        ref, outs = _run_paths(api, c, feats, name, torch.cuda.device_count())
    r0, x0, o0 = ref
    assert (r0["status"] == api.ACCEPT).sum() > 0
    for key, (r, x, o) in outs.items():
        assert r.tobytes() == r0.tobytes(), key
        if x is not None:
            assert np.array_equal(x, x0) and np.array_equal(np.asarray(o, np.int64), o0), key


def test_interleaved_methods(api, feats):
    """homography -> affine -> partial -> homography on one context (one engine, one niters table keyed on the model
    points): the two homography results are the same bytes, each affine result is a fresh context's"""
    seq = ("homography", "affine", "partial", "homography")
    with api.Context(0) as c:
        r = Real(c, feats)
        got = [c.detect_scenes_inliers(r.models, r.scenes, scales=r.scales, params=_params(api, nm)) for nm in seq]
        r.free()
    assert got[0][0].tobytes() == got[3][0].tobytes() and np.array_equal(got[0][1], got[3][1])
    for i, nm in ((1, "affine"), (2, "partial")):
        with api.Context(0) as c:
            r = Real(c, feats)
            fresh = c.detect_scenes_inliers(r.models, r.scenes, scales=r.scales, params=_params(api, nm))
            r.free()
        assert got[i][0].tobytes() == fresh[0].tobytes() and np.array_equal(got[i][1], fresh[1]), nm
        assert got[i][0].tobytes() != got[0][0].tobytes()


# ---------------------------------------------------------------- edge cases
def test_model_point_count_sets_found_by_the_closed_form(api, ctx):
    """views with exactly 3 (affine) and 2 (partial) good matches: the closed form, mask all ones, no refine"""
    rng = np.random.default_rng(31)
    t = synth.sift_like(rng, 600)
    tk = rng.uniform([0, 0], [640, 480], size=(600, 2)).astype(np.float32)
    rows = rng.permutation(600)[:10]
    q = t[rows].copy()                                          # exact copies: distance 0, accepted by the ratio test
    qk = rng.uniform([0, 0], [640, 480], size=(10, 2)).astype(np.float32)
    vo = [0, 3, 5, 10]                                          # views of 3, 2 and 5 good matches
    models = ctx.upload_models(q, qk, vo, [0, 0, 0])
    for name, mp in (("affine", 3), ("partial", 2)):
        p = _params(api, name, min_inliers=mp, det_lo=0.0, det_hi=float("inf"))
        res, xy, off = ctx.detect_pairs(models, t, tk, params=p)
        assert res["n_good"].tolist() == [3, 2, 5]
        fn = ctx.estimate_affine2d if name == "affine" else ctx.estimate_affine_partial2d
        for v in range(3):
            a, b = vo[v], vo[v + 1]
            M, mask = fn(qk[a:b], tk[rows[a:b]], threshold=3.0, max_iters=2000, confidence=0.99, refine_iters=10)
            if b - a < mp:
                assert M is None and res["status"][v] == api.LT4_MATCHES and not res["H"][v].any()
                continue
            assert res["status"][v] == api.ACCEPT and res["n_inliers"][v] == mask.sum()
            assert same_bytes(res["H"][v][:6], M) and res["H"][v][8] == 1.0
            assert np.array_equal(xy[off[v]:off[v + 1]], tk[rows[a:b]][mask.astype(bool)])
            if b - a == mp:
                assert mask.all() and res["n_inliers"][v] == mp
    models.free()


def test_invalid_parameters(api, ctx, real):
    cases = [(dict(method=3), 1), (dict(method=-1), 1)]
    for nm in METHODS:
        cases += [(dict(method=_method(api, nm), flags=api.RANSAC_NO_REFINE), 1),
                  (dict(method=_method(api, nm), flags=4), 1),
                  (dict(method=_method(api, nm), refine_iters=-1), 5),
                  (dict(method=_method(api, nm), refine_iters=1001), 5)]
    for kw, code in cases:
        p = api.detect_params(method=kw["method"], refine_iters=kw.get("refine_iters", 10))
        p.ransac.flags = kw.get("flags", 0)
        for call in (lambda: ctx.detect_scenes(real.models, real.scenes, params=p),
                     lambda: ctx.submit_scenes(real.models, real.scenes, params=p),
                     lambda: ctx.detect_pairs(real.models, real.feats["scene_desc"][:500].astype(np.float32),
                                              real.feats["scene_kpt"][:500], params=p)):
            with pytest.raises(api.CvgError) as e:
                call()
            assert e.value.code == code, kw
    p = api.detect_params(); p.size = 60
    with pytest.raises(api.CvgError) as e:
        ctx.detect_scenes(real.models, real.scenes, params=p)
    assert e.value.code == 1
    # homography ignores refine_iters; the affine methods accept 0 and 1000
    ref = ctx.detect_scenes(real.models, real.scenes, scales=real.scales)
    p = api.detect_params(refine_iters=5000)
    assert ctx.detect_scenes(real.models, real.scenes, scales=real.scales, params=p).tobytes() == ref.tobytes()
    for nm in METHODS:
        for ri in (0, 1000):
            ctx.detect_scenes(real.models, real.scenes, params=api.detect_params(
                ransac=api.ransac_params(3.0, 2000, 0.99), method=_method(api, nm), refine_iters=ri))


class OldDetectParams(C.Structure):
    """cvg_detect_params as it was before `method` and `refine_iters`: 56 bytes"""
    _fields_ = [("size", C.c_uint32), ("ratio", C.c_float), ("min_inliers", C.c_int32), ("det_lo", C.c_float),
                ("det_hi", C.c_float), ("reserved", C.c_int32), ("ransac", RansacParams)]


def test_old_layout_and_explicit_homography_same_bytes(api, ctx, real):
    assert C.sizeof(OldDetectParams) == 56
    lib, ptr = ctx.lib, (lambda a: a.ctypes.data_as(C.c_void_p))
    default = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales)
    explicit = ctx.detect_scenes_inliers(real.models, real.scenes, scales=real.scales,
                                         params=api.detect_params(method=api.VERIFY_HOMOGRAPHY))
    assert explicit[0].tobytes() == default[0].tobytes() and np.array_equal(explicit[1], default[1])
    d = api.detect_params()
    old = OldDetectParams()
    old.size = 56; old.ratio = d.ratio; old.min_inliers = d.min_inliers; old.det_lo = d.det_lo; old.det_hi = d.det_hi
    old.reserved = 12345; old.ransac = d.ransac
    # a 64-byte struct that says 56: the tail (method 2, refine_iters -5) is not the caller's and must not be read
    tail = api.detect_params(method=api.VERIFY_AFFINE_PARTIAL, refine_iters=-5); tail.size = 56; tail.reserved = -1
    S, V = real.scenes.n_scenes, real.models.n_views
    sc = np.ascontiguousarray(real.scales, np.float32)
    for p in (C.cast(C.pointer(old), C.POINTER(DetectParams)), C.pointer(tail)):
        res = np.zeros(S * V, api.PAIR_DTYPE)
        ctx._check(lib.cvg_detect_scenes(ctx.handle, real.models.handle, real.scenes.handle, ptr(sc), p, ptr(res)))
        assert res.tobytes() == default[0].tobytes()
        res = np.zeros(S * V, api.PAIR_DTYPE); inl = np.zeros((S * real.models.n_rows, 2), np.float32)
        off = np.zeros(S * V + 1, np.int64); h = C.c_void_p()
        ctx._check(lib.cvg_detect_scenes_submit(ctx.handle, real.models.handle, real.scenes.handle, ptr(sc), p, ptr(res),
                                                ptr(inl), ptr(off), C.byref(h)))
        ctx._check(lib.cvg_job_wait(ctx.handle, h))
        assert res.tobytes() == default[0].tobytes() and np.array_equal(inl[:off[-1]], default[1])
        so = real.so
        res = np.zeros(V, api.PAIR_DTYPE)
        t = np.ascontiguousarray(real.feats["scene_desc"][so[2]:so[3]], np.float32)
        k = np.ascontiguousarray(real.feats["scene_kpt"][so[2]:so[3]], np.float32)
        ctx._check(lib.cvg_detect_pairs(ctx.handle, real.models.handle, ptr(t), ptr(k), len(t), float(real.scales[2]), p,
                                        ptr(res), None, None))
        assert res.tobytes() == default[0][2].tobytes()


def test_timing_reports_no_stale_solve_and_score_times(api, feats):
    with api.Context(0) as c:
        c.set_lanes(1)                                           # every call on the context's own engine
        r = Real(c, feats)
        c.set_timing(True)
        c.detect_scenes(r.models, r.scenes, scales=r.scales)
        t = c.last_timing()
        assert t["hyp_launches"] > 0 and t["hyp_ms"] > 0 and t["score_ms"] > 0 and t["scored_points"] > 0
        for nm in METHODS:
            c.detect_scenes(r.models, r.scenes, scales=r.scales, params=_params(api, nm))
            t = c.last_timing()
            assert t["hyp_launches"] == 0 and t["hyp_ms"] == 0 and t["score_ms"] == 0 and t["scored_points"] == 0, nm
            assert t["ransac_ms"] > 0 and t["match_ms"] > 0 and t["total_ms"] >= t["ransac_ms"], nm
        r.free()
