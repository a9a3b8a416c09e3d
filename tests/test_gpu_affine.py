"""cv::estimateAffine2D(RANSAC) on the GPU (cvg_estimate_affine2d / _batch) against cv2 4.13.0's outputs
(tests/golden/golden_affine.npz) and the CPU oracle.  Masks and found are exact on every set; M is bit-equal where the
refine runs on fewer than 50 inliers (below that cv2's every sum is pinned) and within 4e-8 relative above, where cv2's
gemm goes through OpenBLAS in an unpinned order.  Against the oracle the RANSAC iteration count is exact everywhere."""
import numpy as np
import pytest

import affine_cases
import affine_oracle

from computervision_objectdetection_featurematching_b200 import synth

pytestmark = pytest.mark.gpu

UNPINNED_REL = 4e-8


@pytest.fixture(scope="module")
def api():
    from computervision_objectdetection_featurematching_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def ctx(api):
    with api.Context(0) as c:
        yield c


@pytest.fixture(scope="module")
def gaff():
    return affine_cases.load_golden()


@pytest.fixture(scope="module")
def aff_oracle():
    return affine_oracle


def _check_golden(g, tag, out):
    off = g[f"{tag}_offsets"]
    assert np.array_equal(out["mask"], g[f"{tag}_mask"])
    assert np.array_equal(out["found"], g[f"{tag}_found"])
    for k in range(len(off) - 1):
        M = out["M"][k].ravel(); Mg = g[f"{tag}_M"][k]
        n_inl = int(g[f"{tag}_mask"][off[k]:off[k + 1]].sum())
        if not g[f"{tag}_found"][k] or n_inl < 50:
            assert np.array_equal(M, Mg), (tag, k, n_inl)
        else:
            assert np.max(np.abs(M - Mg) / np.maximum(np.abs(Mg), 1e-12)) < UNPINNED_REL, (tag, k)


def _oracle_batch(aff_oracle, src, dst, off, **kw):
    Ms, masks, founds, iters = [], [], [], []
    for k in range(len(off) - 1):
        a, b = off[k], off[k + 1]
        if b == a:
            Ms.append(np.zeros(6)); founds.append(False); iters.append(0)
            continue
        r = aff_oracle.estimate_affine2d(src[a:b], dst[a:b], **kw)
        Ms.append(r["M"].ravel()); masks.append(r["mask"]); founds.append(r["found"]); iters.append(r["info"]["iters_run"])
    return np.stack(Ms), np.concatenate(masks) if masks else np.zeros(0, np.uint8), np.array(founds), np.array(iters)


def test_golden_synthetic_and_real(ctx, gaff, aff_oracle):
    for tag in ("syn", "real"):
        out = ctx.estimate_affine2d_batch(gaff[f"{tag}_src"], gaff[f"{tag}_dst"], gaff[f"{tag}_offsets"])
        _check_golden(gaff, tag, out)
        _, _, _, it = _oracle_batch(aff_oracle, gaff[f"{tag}_src"], gaff[f"{tag}_dst"], gaff[f"{tag}_offsets"])
        assert np.array_equal(out["iters"], it)
    assert (np.diff(gaff["syn_offsets"]) == 8192).any()


def test_single_call_equals_batch(ctx, gaff):
    off = gaff["syn_offsets"]
    out = ctx.estimate_affine2d_batch(gaff["syn_src"], gaff["syn_dst"], off)
    for k in range(len(off) - 1):
        a, b = off[k], off[k + 1]
        M, mask = ctx.estimate_affine2d(gaff["syn_src"][a:b], gaff["syn_dst"][a:b])
        assert (M is not None) == out["found"][k]
        assert np.array_equal(mask, out["mask"][a:b])
        if M is not None:
            assert np.array_equal(M, out["M"][k])


def test_parameter_variants(ctx, gaff, aff_oracle):
    s, d = gaff["par_src"], gaff["par_dst"]
    for (thr, it, conf, ref), Mg, maskg in zip(gaff["par_params"], gaff["par_M"], gaff["par_mask"]):
        M, mask = ctx.estimate_affine2d(s, d, threshold=float(thr), max_iters=int(it), confidence=float(conf),
                                        refine_iters=int(ref))
        assert np.array_equal(mask, maskg)
        if int(maskg.sum()) < 50:
            assert np.array_equal(M.ravel(), Mg)
        else:
            assert np.max(np.abs(M.ravel() - Mg) / np.maximum(np.abs(Mg), 1e-12)) < UNPINNED_REL
    rng = np.random.default_rng(11)
    src, dst, _ = synth.correspondences(rng, 40, 0.6)
    for ref in range(13):                                        # refine_iters 0..12 against the CPU restatement, bit for bit
        M, mask = ctx.estimate_affine2d(src, dst, refine_iters=ref)
        r = aff_oracle.estimate_affine2d(src, dst, refine_iters=ref)
        assert np.array_equal(M, r["M"]) and np.array_equal(mask, r["mask"]), ref


def test_small_n_and_invalid_params(ctx, api):
    tri = np.array([[0, 0], [10, 0], [0, 10]], np.float32)
    for n in (1, 2):
        M, mask = ctx.estimate_affine2d(tri[:n], tri[:n] + 3)
        assert M is None and not mask.any()
    M, mask = ctx.estimate_affine2d(tri, tri * 2 + 1)
    assert np.array_equal(M, [[2, 0, 1], [0, 2, 1]]) and mask.all()
    with pytest.raises(api.CvgError) as e:
        ctx.estimate_affine2d(np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32))
    assert e.value.code == 3
    for kw, code in ((dict(flags=2), 1), (dict(flags=4), 1), (dict(refine_iters=-1), 5), (dict(refine_iters=1001), 5),
                     (dict(confidence=1.0), 1), (dict(max_iters=0), 5)):
        with pytest.raises(api.CvgError) as e:
            ctx.estimate_affine2d(tri, tri, **kw)
        assert e.value.code == code, kw
    out = ctx.estimate_affine2d_batch(np.r_[tri, tri], np.r_[tri, tri], [0, 2, 2, 5, 6])
    assert list(out["found"]) == [False, False, True, False]


def test_no_early_stop_against_oracle_iterations(ctx, api, aff_oracle):
    """5 % inlier sets: the adaptive niters never falls below max_iters, so cv2's loop runs exactly the iterations the
    no-early-stop mode scores; up to 30 000 iterations, all on the round sampler."""
    rng = np.random.default_rng(12)
    sets = [synth.correspondences(rng, n, 0.05)[:2] for n in (300, 2000, 5000)]
    src = np.concatenate([s for s, _ in sets]); dst = np.concatenate([d for _, d in sets])
    off = np.cumsum([0] + [len(s) for s, _ in sets])
    for it in (2000, 30000):
        out = ctx.estimate_affine2d_batch(src, dst, off, max_iters=it, flags=api.RANSAC_NO_EARLY_STOP)
        assert ctx.last_sampler_serial_sets == -1                # the chunked sampler is for 4-point draws only
        Ms, masks, founds, iters = _oracle_batch(aff_oracle, src, dst, off, max_iters=it)
        assert np.array_equal(iters, np.full(len(off) - 1, it))
        assert np.array_equal(out["iters"], iters)
        assert np.array_equal(out["mask"], masks) and np.array_equal(out["found"], founds)
        for k in range(len(off) - 1):
            assert np.max(np.abs(out["M"][k].ravel() - Ms[k]) / np.maximum(np.abs(Ms[k]), 1e-12)) < UNPINNED_REL


def test_rng_table_regrowth(api, aff_oracle, gaff):
    """A set with one point off a line and random targets: every iteration spends ~n draws on rejected attempts and the
    loop runs all 2000 iterations, 3 M draws, beyond a fresh context's table, which is grown and the stage repeated.
    Then the rejection-heavy goldens, one of which exhausts getSubset's 10000 attempts."""
    rng = np.random.default_rng(14)
    n = 1500
    x = rng.integers(0, 20000, n).astype(np.float32)
    src = np.c_[x, 2 * x + 3].astype(np.float32); src[7] = (300, 50)
    dst = rng.uniform(0, 640, (n, 2)).astype(np.float32)
    r = aff_oracle.estimate_affine2d(src, dst)
    assert r["info"]["draws"] > (1 << 21)
    with api.Context(0) as fresh:
        M, mask = fresh.estimate_affine2d(src, dst)
        out = fresh.estimate_affine2d_batch(src, dst, [0, n])
    assert np.array_equal(M, r["M"]) and np.array_equal(mask, r["mask"]) and out["iters"][0] == r["info"]["iters_run"]
    off = gaff["syn_offsets"]
    for k in [k for k in range(len(off) - 1) if off[k + 1] - off[k] in (4000, 9000, 15000)]:
        a, b = off[k], off[k + 1]
        with api.Context(0) as fresh:
            M, mask = fresh.estimate_affine2d(gaff["syn_src"][a:b], gaff["syn_dst"][a:b])
        assert (M is not None) == gaff["syn_found"][k] and np.array_equal(mask, gaff["syn_mask"][a:b])


def test_niters_all_on_host_same_bytes(ctx, api, gaff):
    ref = ctx.estimate_affine2d_batch(gaff["real_src"], gaff["real_dst"], gaff["real_offsets"])
    with api.Context(0, flags=api.NITERS_ALL_ON_HOST) as c:
        out = c.estimate_affine2d_batch(gaff["real_src"], gaff["real_dst"], gaff["real_offsets"])
    for key in ("M", "mask", "found", "iters"):
        assert np.array_equal(out[key], ref[key]), key


def test_interleaved_with_homography(api, gaff):
    """Both verify methods on one context share its host-verified niters table, keyed on the model points: the homography
    outputs equal those of a context that never ran an affine call (with every niters entry answered on the host)."""
    rng = np.random.default_rng(13)
    sets = [synth.correspondences(rng, n, r)[:2] for n, r in ((60, 0.5), (200, 0.3), (1000, 0.2))]
    src = np.concatenate([s for s, _ in sets]); dst = np.concatenate([d for _, d in sets])
    off = np.cumsum([0] + [len(s) for s, _ in sets])
    with api.Context(0, flags=api.NITERS_ALL_ON_HOST) as c:
        h_ref = c.find_homography_batch(src, dst, off, want_ransac_mask=True)
        a_ref = c.estimate_affine2d_batch(src, dst, off)
    with api.Context(0, flags=api.NITERS_ALL_ON_HOST) as c:
        for _ in range(2):
            a = c.estimate_affine2d_batch(src, dst, off)
            h = c.find_homography_batch(src, dst, off, want_ransac_mask=True)
            for key in h_ref:
                assert np.array_equal(h[key], h_ref[key]), key
            for key in a_ref:
                assert np.array_equal(a[key], a_ref[key]), key


def test_multi_device_and_lanes_same_bytes(api, gaff):
    ref = None
    for dev, lanes in ((0, 1), (0, 3), ([0, 0], 0)):
        with api.Context(dev) as c:
            if lanes:
                c.set_lanes(lanes)
            out = c.estimate_affine2d_batch(gaff["syn_src"], gaff["syn_dst"], gaff["syn_offsets"])
        if ref is None:
            ref = out
        for key in ref:
            assert np.array_equal(out[key], ref[key]), (dev, lanes, key)
