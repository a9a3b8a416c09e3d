"""cv::estimateAffinePartial2D(RANSAC) on the GPU (cvg_estimate_affine_partial2d / _batch) against cv2 4.13.0's outputs
(tests/golden/golden_affine_partial.npz) and the CPU oracle.  Masks and found are exact on every set; M is bit-equal
(NaN positions for the coincident pair) where the refine runs on fewer than 50 inliers and within 4e-8 relative above,
where cv2's gemm goes through OpenBLAS in an unpinned order.  Against the oracle the RANSAC iteration count is exact."""
import numpy as np
import pytest

import affine_partial_oracle
import affine_partial_cases as cases
from affine_partial_cases import same_bytes

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
def gp():
    return cases.load_golden()


def _same_outputs(a, b):
    return all(same_bytes(a[k], b[k]) if k == "M" else np.array_equal(a[k], b[k]) for k in a)


def _check_M(M, Mg, n_inl, found, what):
    if not found or n_inl < 50:
        assert same_bytes(M, Mg), what
    else:
        assert np.max(np.abs(M.ravel() - Mg) / np.maximum(np.abs(Mg), 1e-12)) < UNPINNED_REL, what


def _oracle_batch(src, dst, off, **kw):
    Ms, masks, founds, iters = [], [], [], []
    for k in range(len(off) - 1):
        a, b = off[k], off[k + 1]
        if b == a:
            Ms.append(np.zeros(6)); founds.append(False); iters.append(0)
            continue
        r = affine_partial_oracle.estimate_affine_partial2d(src[a:b], dst[a:b], **kw)
        Ms.append(r["M"].ravel()); masks.append(r["mask"]); founds.append(r["found"]); iters.append(r["info"]["iters_run"])
    return np.stack(Ms), np.concatenate(masks) if masks else np.zeros(0, np.uint8), np.array(founds), np.array(iters)


def test_golden_synthetic_and_real(ctx, gp):
    for tag in ("syn", "real"):
        off = gp[f"{tag}_offsets"]
        out = ctx.estimate_affine_partial2d_batch(gp[f"{tag}_src"], gp[f"{tag}_dst"], off)
        assert np.array_equal(out["mask"], gp[f"{tag}_mask"])
        assert np.array_equal(out["found"], gp[f"{tag}_found"])
        for k in range(len(off) - 1):
            n_inl = int(gp[f"{tag}_mask"][off[k]:off[k + 1]].sum())
            _check_M(out["M"][k], gp[f"{tag}_M"][k], n_inl, gp[f"{tag}_found"][k], (tag, k, n_inl))
        _, _, _, it = _oracle_batch(gp[f"{tag}_src"], gp[f"{tag}_dst"], off)
        assert np.array_equal(out["iters"], it)
    assert (np.diff(gp["syn_offsets"]) == 8192).any()


def test_single_call_equals_batch(ctx, gp):
    off = gp["syn_offsets"]
    out = ctx.estimate_affine_partial2d_batch(gp["syn_src"], gp["syn_dst"], off)
    for k in range(len(off) - 1):
        a, b = off[k], off[k + 1]
        M, mask = ctx.estimate_affine_partial2d(gp["syn_src"][a:b], gp["syn_dst"][a:b])
        assert (M is not None) == out["found"][k]
        assert np.array_equal(mask, out["mask"][a:b])
        if M is not None:
            assert same_bytes(M, out["M"][k])


def test_parameter_variants(ctx, gp):
    s, d = gp["par_src"], gp["par_dst"]
    for (thr, it, conf, ref), Mg, maskg in zip(gp["par_params"], gp["par_M"], gp["par_mask"]):
        M, mask = ctx.estimate_affine_partial2d(s, d, threshold=float(thr), max_iters=int(it), confidence=float(conf),
                                                refine_iters=int(ref))
        assert np.array_equal(mask, maskg)
        _check_M(M, Mg, int(maskg.sum()), True, (thr, it, conf, ref))
    rng = np.random.default_rng(21)
    src, dst = cases.similarity_correspondences(rng, 40, 0.6)
    for ref in range(13):                                        # refine_iters 0..12 against the CPU restatement, bit for bit
        M, mask = ctx.estimate_affine_partial2d(src, dst, refine_iters=ref)
        r = affine_partial_oracle.estimate_affine_partial2d(src, dst, refine_iters=ref)
        assert M.tobytes() == r["M"].tobytes() and np.array_equal(mask, r["mask"]), ref


def test_small_n_and_invalid_params(ctx, api):
    tri = np.array([[0, 0], [10, 0], [0, 10]], np.float32)
    M, mask = ctx.estimate_affine_partial2d(tri[:1], tri[:1] + 3)
    assert M is None and not mask.any()
    M, mask = ctx.estimate_affine_partial2d(tri[:2], tri[:2] * 2 + 1)
    assert np.array_equal(M, [[2, 0, 1], [0, 2, 1]]) and mask.all()
    assert np.signbit(M[0, 1]) and not np.signbit(M[1, 0])      # -S1 with S1 == +0, as cv2 returns it
    M, mask = ctx.estimate_affine_partial2d(tri[[0, 0]], tri[[1, 2]])
    assert M is not None and np.isnan(M).all() and mask.all()   # coincident source points: NaN, found, mask 1,1
    M, mask = ctx.estimate_affine_partial2d(np.full((4, 2), 7, np.float32), np.full((4, 2), 9, np.float32))
    assert M is None and not mask.any()
    with pytest.raises(api.CvgError) as e:
        ctx.estimate_affine_partial2d(np.zeros((0, 2), np.float32), np.zeros((0, 2), np.float32))
    assert e.value.code == 3
    for kw, code in ((dict(flags=2), 1), (dict(flags=4), 1), (dict(refine_iters=-1), 5), (dict(refine_iters=1001), 5),
                     (dict(confidence=1.0), 1), (dict(max_iters=0), 5)):
        with pytest.raises(api.CvgError) as e:
            ctx.estimate_affine_partial2d(tri, tri, **kw)
        assert e.value.code == code, kw
    out = ctx.estimate_affine_partial2d_batch(np.r_[tri, tri], np.r_[tri, tri], [0, 1, 1, 3, 6])
    assert list(out["found"]) == [False, False, True, True]


def test_collinear_set_found_where_affine2d_is_not(ctx):
    xs = np.linspace(0, 100, 12).astype(np.float32)
    src, dst = np.c_[xs, 2 * xs].astype(np.float32), np.c_[xs + 5, 2 * xs + 1].astype(np.float32)
    M, mask = ctx.estimate_affine_partial2d(src, dst)
    r = affine_partial_oracle.estimate_affine_partial2d(src, dst)
    assert M is not None and mask.all() and M.tobytes() == r["M"].tobytes()
    M6, mask6 = ctx.estimate_affine2d(src, dst)
    assert M6 is None and not mask6.any()


def test_no_early_stop_against_oracle_iterations(ctx, api):
    """1 % inlier sets (a 2-point model needs far fewer inliers than 5 % to stop early): the adaptive niters never falls
    below max_iters, so cv2's loop runs exactly the iterations the no-early-stop mode scores; up to 30 000 iterations, all
    on the round sampler."""
    rng = np.random.default_rng(22)
    sets = [cases.similarity_correspondences(rng, n, 0.01) for n in (1000, 2000, 5000)]
    src, dst, off = cases.pack(sets)
    for it in (2000, 30000):
        out = ctx.estimate_affine_partial2d_batch(src, dst, off, max_iters=it, flags=api.RANSAC_NO_EARLY_STOP)
        assert ctx.last_sampler_serial_sets == -1                # the chunked sampler is for 4-point draws only
        Ms, masks, founds, iters = _oracle_batch(src, dst, off, max_iters=it)
        assert np.array_equal(iters, np.full(len(off) - 1, it))
        assert np.array_equal(out["iters"], iters)
        assert np.array_equal(out["mask"], masks) and np.array_equal(out["found"], founds)
        for k in range(len(off) - 1):
            assert np.max(np.abs(out["M"][k].ravel() - Ms[k]) / np.maximum(np.abs(Ms[k]), 1e-12)) < UNPINNED_REL


def test_niters_all_on_host_same_bytes(ctx, api, gp):
    ref = ctx.estimate_affine_partial2d_batch(gp["real_src"], gp["real_dst"], gp["real_offsets"])
    with api.Context(0, flags=api.NITERS_ALL_ON_HOST) as c:
        out = c.estimate_affine_partial2d_batch(gp["real_src"], gp["real_dst"], gp["real_offsets"])
    assert _same_outputs(out, ref)


def test_interleaved_with_homography_and_affine(api):
    """The three verify methods on one context share its host-verified niters table, keyed on the model points 2/3/4:
    interleaved, each gives the bytes it gives on a context that runs it alone."""
    rng = np.random.default_rng(23)
    sets = [synth.correspondences(rng, n, r)[:2] for n, r in ((60, 0.5), (200, 0.3), (1000, 0.2))]
    src, dst, off = cases.pack(sets)
    runs = {"h": lambda c: c.find_homography_batch(src, dst, off, want_ransac_mask=True),
            "a": lambda c: c.estimate_affine2d_batch(src, dst, off),
            "p": lambda c: c.estimate_affine_partial2d_batch(src, dst, off)}
    ref = {}
    for key, run in runs.items():
        with api.Context(0, flags=api.NITERS_ALL_ON_HOST) as c:
            ref[key] = run(c)
    with api.Context(0, flags=api.NITERS_ALL_ON_HOST) as c:
        for _ in range(2):
            for key in ("p", "h", "a", "p"):
                assert _same_outputs(runs[key](c), ref[key]), key


def test_multi_device_and_lanes_same_bytes(api, gp):
    ref = None
    for dev, lanes in ((0, 1), (0, 3), ([0, 0], 0)):
        with api.Context(dev) as c:
            if lanes:
                c.set_lanes(lanes)
            out = c.estimate_affine_partial2d_batch(gp["syn_src"], gp["syn_dst"], gp["syn_offsets"])
        if ref is None:
            ref = out
        assert _same_outputs(out, ref), (dev, lanes)
