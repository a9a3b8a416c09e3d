"""GPU parity tests: libcvgraft (through its C ABI) against the CPU oracle and the cv2 goldens.
Bit-exact for indices / accept masks / inlier masks, tolerances (stated per test) for floating point."""
import numpy as np
import pytest

from computervision_objectdetection_featurematching_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def api():
    from computervision_objectdetection_featurematching_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def ctx(api):
    c = api.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ctx_exact(api):
    c = api.Context(0, api.FORCE_EXACT_MATCH)
    yield c
    c.close()


def _assert_match(got, want, check_dist_exact=True):
    idx, dist, acc = got
    widx, wdist, wacc = want
    assert np.array_equal(idx, widx)
    valid = widx >= 0
    if check_dist_exact:
        assert np.array_equal(dist[valid], wdist[valid])
    else:
        assert np.allclose(dist[valid], wdist[valid], rtol=1e-4, atol=0)      # north_star: 1e-4 relative
    assert np.array_equal(acc, wacc)


# ---------------------------------------------------------------- match stage
def test_match_tensor_path_integer_descriptors(ctx, api, oracle):
    rng = np.random.default_rng(101)
    for nq, nt in [(300, 700), (128, 256), (1, 2), (129, 257), (500, 3000), (77, 5)]:
        q, t, _ = synth.planted_pair(rng, nq, nt)
        got = ctx.match_knn2(q, t)
        assert ctx.last_match_path == api.PATH_TENSOR
        oi, od = oracle.knn2(q, t, nthreads=8)
        _assert_match(got, (oi, od, oracle.ratio(oi, od)))


def test_match_ties_and_duplicates(ctx, api, gsynth):
    q, t = gsynth["knn_int_q"], gsynth["knn_int_t"]
    idx, dist, acc = ctx.match_knn2(q, t)
    assert ctx.last_match_path == api.PATH_TENSOR
    assert np.array_equal(idx, gsynth["knn_int_idx"])          # cv2 golden incl. exact distance ties
    assert np.array_equal(dist, gsynth["knn_int_dist"])


def test_match_float_descriptors_candidate_path_and_exact_path(ctx, ctx_exact, api, gsynth):
    """Non-integer descriptors: tensor-core candidates + fp32 re-rank with proof (+ exact fallback rows) must give
    cv2's indices and distances bit for bit, like the exact SIMT kernel (cv::batchDistance summation order)."""
    for c, path in ((ctx, api.PATH_TENSOR_RERANK), (ctx_exact, api.PATH_EXACT)):
        idx, dist, acc = c.match_knn2(gsynth["knn_float_q"], gsynth["knn_float_t"])
        assert c.last_match_path == path
        assert np.array_equal(idx, gsynth["knn_float_idx"])
        assert np.array_equal(dist, gsynth["knn_float_dist"])


def test_match_float_candidate_path_stress(ctx, ctx_exact, api, oracle):
    """Shapes and data that stress the candidate path's proof: near-duplicate train rows (distance gaps far below the
    bf16 error bound -> fallback rows), exact duplicates (ties -> lower index), tiny and ragged sizes, mixed integer
    query vs float train, large dynamic range, unit-norm (RootSIFT-like) rows."""
    rng = np.random.default_rng(1103)
    cases = []
    q = synth.float_desc(rng, 300, 128); t = synth.float_desc(rng, 2000, 128)
    t[500:700] = t[0:200] + rng.normal(0, 1e-3, size=(200, 128)).astype(np.float32)     # near duplicates
    t[900] = t[17]; t[1500] = t[17]                                                     # exact duplicates
    q[:50] = t[rng.integers(0, 2000, 50)] + rng.normal(0, 0.5, size=(50, 128)).astype(np.float32)
    q[7] = t[17]
    cases.append((q, t))
    for nq, nt in [(1, 3), (5, 4), (129, 5), (77, 257), (260, 1000)]:
        cases.append((synth.float_desc(rng, nq, 128), synth.float_desc(rng, nt, 128)))
    qi, ti, _ = synth.planted_pair(rng, 200, 900)
    cases.append((qi, ti + np.float32(0.25)))                                           # integer queries, float train
    cases.append((qi + np.float32(0.5), ti))
    u = np.abs(rng.standard_normal((400, 128))).astype(np.float32); u /= np.linalg.norm(u, axis=1, keepdims=True)
    cases.append((np.sqrt(u[:100]).astype(np.float32), np.sqrt(u[100:]).astype(np.float32)))
    big = (synth.float_desc(rng, 150, 128) * np.float32(1e4)).astype(np.float32)
    cases.append((big[:50], big[50:]))
    n_fallback = 0
    for q, t in cases:
        got = ctx.match_knn2(q, t)
        assert ctx.last_match_path == api.PATH_TENSOR_RERANK
        n_fallback += ctx.last_match_fallback_rows
        oi, od = oracle.knn2(q, t, nthreads=8)
        _assert_match(got, (oi, od, oracle.ratio(oi, od)))
        ref = ctx_exact.match_knn2(q, t)
        for x, y in zip(got, ref):
            assert np.array_equal(x, y)
    assert n_fallback > 0                                    # the near-duplicate rows cannot be proven: fallback exercised


def test_match_float_8k_candidate_path(ctx, api, oracle):
    """8192 x 8192 non-integer descriptors (BASELINE config 3 shape, 'float' generator of SURVEY 8d) through the
    candidate path: bit-equal to the CPU oracle on 1024 sampled rows."""
    rng = np.random.default_rng(3103)
    q = synth.float_desc(rng, 8192, 128); t = synth.float_desc(rng, 8192, 128)
    rows = rng.permutation(8192)[:4096]
    t[rows[:2048]] = q[rows[2048:]] + rng.normal(0, 6.0, size=(2048, 128)).astype(np.float32)   # planted neighbours
    idx, dist, acc = ctx.match_knn2(q, t)
    assert ctx.last_match_path == api.PATH_TENSOR_RERANK
    assert ctx.last_match_fallback_rows < 82                 # < 1 % of the rows need the exact fallback
    chk = rng.permutation(8192)[:1024]
    oi, od = oracle.knn2(q[chk], t, nthreads=8)
    assert np.array_equal(idx[chk], oi) and np.array_equal(dist[chk], od)
    assert np.array_equal(acc[chk], oracle.ratio(oi, od))


def test_match_both_paths_agree(ctx, ctx_exact, api):
    q, t, _ = synth.planted_pair(np.random.default_rng(102), 1000, 4000)
    a = ctx.match_knn2(q, t)
    b = ctx_exact.match_knn2(q, t)
    assert ctx.last_match_path == api.PATH_TENSOR and ctx_exact.last_match_path == api.PATH_EXACT
    for x, y in zip(a, b):
        assert np.array_equal(x, y)


def test_match_pair_mode_cta_group_2(api, oracle):
    """The cta_group::2 form of the match kernel (clusters of two CTAs, one M256 N256 MMA on two query tiles, each CTA
    holding half of every train stage; opt-in, CVG_MATCH_PAIR_MODE) gives the one-CTA form's results bit for bit:
    even number of query row blocks -> pairs; odd -> the one-CTA kernel serves the call."""
    rng = np.random.default_rng(4242)
    with api.Context(0, api.MATCH_PAIR_MODE) as cp, api.Context(0) as c1:
        for nq, nt in ((512, 3000), (1024, 700), (256, 255), (2048, 8192), (384, 1000)):
            q = synth.sift_like(rng, nq); t = synth.sift_like(rng, nt)
            t[rng.permutation(nt)[: nt // 3]] = q[rng.integers(0, nq, size=nt // 3)]       # exact duplicates: ties
            a = cp.match_knn2(q, t); b = c1.match_knn2(q, t)
            assert cp.last_match_path == api.PATH_TENSOR
            for x, y in zip(a, b):
                assert np.array_equal(x, y), (nq, nt)
        q = synth.sift_like(rng, 640); t = synth.sift_like(rng, 2100)
        oi, od = oracle.knn2(q, t, nthreads=4)
        i, d, acc = cp.match_knn2(q, t)
        assert np.array_equal(i, oi) and np.array_equal(d, od) and np.array_equal(acc, oracle.ratio(oi, od))


def test_match_tiny_train_sets(ctx, gsynth):
    q, t = gsynth["knn_int_q"][:9], gsynth["knn_int_t"]
    for nt in (1, 2):
        idx, dist, acc = ctx.match_knn2(q, t[:nt])
        gi, gd = gsynth[f"knn_nt{nt}_idx"], gsynth[f"knn_nt{nt}_dist"]
        assert np.array_equal(idx, gi)
        assert np.array_equal(dist[gi >= 0], gd[gi >= 0])
        if nt == 1:
            assert not acc.any()                            # m.size()==2 fails, src/TestsDetector.cpp:67
    idx, dist, acc = ctx.match_knn2(q, t[:0])
    assert (idx == -1).all() and not acc.any()
    qf = q + np.float32(0.5)                                 # non-integer queries: candidate path, same contract
    for nt in (0, 1, 2, 3):
        idx, dist, acc = ctx.match_knn2(qf, t[:nt])
        assert (idx[:, min(nt, 2):] == -1).all() and (idx[:, :min(nt, 2)] >= 0).all()
        if nt < 2:
            assert not acc.any()


def test_match_resident_models_per_view_and_all(ctx, oracle, feats, gpairs):
    md = feats["model_desc"].astype(np.float32)
    models = ctx.upload_models(md, feats["model_kpt"], feats["view_offsets"], feats["view_model"])
    so = feats["scene_offsets"]
    for s in (0, 4, 7):
        t = feats["scene_desc"][so[s]:so[s + 1]].astype(np.float32)
        idx, dist, acc = ctx.match_knn2(models, t)
        assert np.array_equal(idx, gpairs["idx"][s].astype(np.int32))
        assert np.array_equal(dist, gpairs["dist"][s])
        assert np.array_equal(acc, gpairs["accept"][s])
    vo = feats["view_offsets"]
    t = feats["scene_desc"][so[2]:so[3]].astype(np.float32)
    for v in (0, 17, 88):
        idx, dist, acc = ctx.match_knn2(models, t, view=v)
        assert np.array_equal(idx, gpairs["idx"][2][vo[v]:vo[v + 1]].astype(np.int32))
        assert np.array_equal(acc, gpairs["accept"][2][vo[v]:vo[v + 1]])
    models.free()


def test_match_8k_round_trip_properties(ctx, api):
    """Full-size case (BASELINE config 3 shape): planted matches must be found, self-match is exact."""
    rng = np.random.default_rng(3000)
    q, t, truth = synth.planted_pair(rng, 8192, 8192)
    idx, dist, acc = ctx.match_knn2(q, t)
    assert ctx.last_match_path == api.PATH_TENSOR
    planted = truth >= 0
    assert (idx[planted, 0] == truth[planted]).mean() > 0.999
    assert np.all(dist[:, 0] <= dist[:, 1])
    idx2, dist2, _ = ctx.match_knn2(t, t)                    # every row is its own nearest neighbour
    assert np.array_equal(idx2[:, 0] * 0, np.zeros(8192, np.int32)) and np.all(dist2[:, 0] == 0)
    d0 = np.sqrt(((q[:64, None, :] - t[None, idx[:64, 0], :][0]) ** 2).sum(-1)) if False else None
    # spot-check distances against a direct fp64 evaluation
    for i in range(0, 8192, 517):
        d = np.sqrt(((q[i].astype(np.float64) - t[idx[i, 0]].astype(np.float64)) ** 2).sum())
        assert abs(d - dist[i, 0]) <= 1e-4 * max(d, 1.0)


# ---------------------------------------------------------------- verify stage
def _check_fh(got_H, got_mask, ref, rtol=1e-5):
    assert (got_H is not None) == ref["found"]
    assert np.array_equal(got_mask, ref["mask"])             # bit-exact inlier mask
    if ref["found"]:
        rel = np.max(np.abs(got_H - ref["H"]) / np.maximum(np.abs(ref["H"]), 1e-12))
        assert rel < rtol, rel                               # north_star: 1e-5 relative


def test_find_homography_vs_cv2_goldens(ctx, gsynth):
    off = gsynth["fh_offsets"]
    exact = 0; total = 0
    for k in range(len(off) - 1):
        a, b = off[k], off[k + 1]
        H, mask = ctx.find_homography(gsynth["fh_src"][a:b], gsynth["fh_dst"][a:b])
        assert (H is not None) == bool(gsynth["fh_found"][k]), k
        assert np.array_equal(mask, gsynth["fh_mask"][a:b]), k
        if H is not None:
            G = gsynth["fh_H"][k].reshape(3, 3)
            rel = np.max(np.abs(H - G) / np.maximum(np.abs(G), 1e-12))
            assert rel < 1e-5, (k, rel)
            exact += np.array_equal(H, G); total += 1
    assert exact >= 40, (exact, total)                       # small sets are bit-exact end to end


def test_find_homography_ransac_stage_and_params(ctx, api, oracle, gsynth):
    src, dst = gsynth["fhp_src"], gsynth["fhp_dst"]
    for (thr, it, conf), H, mask in zip(gsynth["fhp_params"], gsynth["fhp_H"], gsynth["fhp_mask"]):
        gH, gmask, rmask = ctx.find_homography(src, dst, float(thr), int(it), float(conf), want_ransac_mask=True)
        ref = oracle.find_homography(src, dst, thr=float(thr), max_iters=int(it), conf=float(conf))
        assert np.array_equal(rmask, ref["ransac_mask"])     # RANSAC-stage mask: RNG replay, bit-exact
        assert np.array_equal(gmask, mask)
        assert np.max(np.abs(gH.ravel() - H) / np.maximum(np.abs(H), 1e-12)) < 1e-5
    # NO_REFINE returns the RANSAC-stage model itself
    gH, gmask = ctx.find_homography(src, dst, flags=api.RANSAC_NO_REFINE)
    ref = oracle.ransac_stage(src, dst)
    assert np.array_equal(gmask, ref["mask"]) and np.array_equal(gH, ref["H"])


def test_find_homography_small_n_bit_exact_vs_oracle(ctx, oracle):
    rng = np.random.default_rng(202)
    srcs, dsts, offs = [], [], [0]
    for _ in range(200):
        n = int(rng.integers(4, 100))
        s, d, _ = synth.correspondences(rng, n, float(rng.uniform(0.2, 0.95)), dup=float(rng.choice([0, 0.3, 0.7])))
        srcs.append(s); dsts.append(d); offs.append(offs[-1] + n)
    out = ctx.find_homography_batch(np.concatenate(srcs), np.concatenate(dsts), offs, want_ransac_mask=True)
    n_exact = 0
    for k in range(200):
        ref = oracle.find_homography(srcs[k], dsts[k])
        a, b = offs[k], offs[k + 1]
        assert out["found"][k] == ref["found"], k
        assert np.array_equal(out["ransac_mask"][a:b], ref["ransac_mask"]), k
        assert np.array_equal(out["mask"][a:b], ref["mask"]), k
        if ref["found"]:
            n_exact += np.array_equal(out["H"][k], ref["H"])
            assert np.allclose(out["H"][k], ref["H"], rtol=1e-9, atol=1e-12), k
            if len(srcs[k]) > 4:
                assert out["iters"][k] == ref["info"]["iters_run"], k
    assert n_exact >= 195, n_exact


def test_find_homography_large_n(ctx, oracle):
    """n = 8192 at 30% inliers (BASELINE config 3): parallel refit/LM path; tolerance 1e-5 on H."""
    rng = np.random.default_rng(3003)
    src, dst, _ = synth.correspondences(rng, 8192, 0.3)
    H, mask, rmask = ctx.find_homography(src, dst, want_ransac_mask=True)
    ref = oracle.find_homography(src, dst)
    assert np.array_equal(rmask, ref["ransac_mask"])
    assert np.max(np.abs(H - ref["H"]) / np.maximum(np.abs(ref["H"]), 1e-12)) < 1e-5
    assert (mask != ref["mask"]).sum() <= 2                  # points within 1e-8 of the threshold may flip
    corners = np.array([[0, 0, 1], [640, 0, 1], [640, 480, 1], [0, 480, 1]], float)
    pa = corners @ H.T; pb = corners @ ref["H"].T
    assert np.max(np.abs(pa[:, :2] / pa[:, 2:] - pb[:, :2] / pb[:, 2:])) < 0.5      # north_star: 0.5 px


def test_find_homography_edge_cases(ctx, api):
    with pytest.raises(api.CvgError) as e:
        ctx.find_homography(np.zeros((3, 2), np.float32), np.zeros((3, 2), np.float32))
    assert e.value.code == 3
    n = 12
    xs = np.linspace(0, 100, n).astype(np.float32)
    H, mask = ctx.find_homography(np.c_[xs, 2 * xs], np.c_[xs + 5, 2 * xs + 1])      # all collinear
    assert H is None and not mask.any()
    H, mask = ctx.find_homography(np.full((n, 2), 7, np.float32), np.full((n, 2), 9, np.float32))
    assert H is None and not mask.any()


def test_find_homography_no_early_stop_scores_every_hypothesis(ctx, api, oracle):
    rng = np.random.default_rng(5005)
    src, dst, _ = synth.correspondences(rng, 512, 0.3)
    H, mask, rmask = ctx.find_homography(src, dst, max_iters=20000, flags=api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE,
                                         want_ransac_mask=True)
    tr = oracle.ransac_stage(src, dst, max_iters=2000, want_trace=True)
    assert mask.sum() >= tr["mask"].sum()                    # more hypotheses can only improve the best count
    # at 5 % inliers the adaptive niters of the reference stays above 30 000, so its loop IS the exhaustive one:
    # the parallel argmax selection must pick the same hypothesis as the serial scan
    for seed in (1, 2, 3):
        s2, d2, _ = synth.correspondences(np.random.default_rng(5100 + seed), 600, 0.05)
        ref = oracle.ransac_stage(s2, d2, max_iters=30000)
        assert ref["info"]["iters_run"] == 30000
        H2, m2 = ctx.find_homography(s2, d2, max_iters=30000, flags=api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE)
        assert np.array_equal(m2, ref["mask"]) and np.array_equal(H2, ref["H"])


def test_find_homography_batch_shapes_thread_kernel(ctx, api, oracle):
    """Shapes that exercise the thread-per-hypothesis kernel's block layout: tiny rounds (many sets per CTA), sets far
    larger than the shared-memory staging buffer (chunked scoring), and wildly mixed set sizes in one batch — RANSAC-stage
    masks bit-exact against the oracle, iteration counts equal."""
    rng = np.random.default_rng(7007)
    cases = [
        dict(sizes=[int(v) for v in rng.integers(5, 60, size=700)], max_iters=10),      # round_len 10: ~22 sets per CTA
        dict(sizes=[20000, 15000, 30001, 14112, 14113, 9, 4, 250], max_iters=600),      # > 14 112 points: staged in chunks
        dict(sizes=[4, 5, 6, 3000, 7, 64, 1, 0, 2, 800] * 3, max_iters=2000),           # mixed, incl. < 4 points
    ]
    for case in cases:
        srcs, dsts, offs = [], [], [0]
        for n in case["sizes"]:
            if n >= 4:
                s, d, _ = synth.correspondences(rng, n, float(rng.uniform(0.25, 0.9)))
            else:
                s = rng.uniform(0, 600, size=(n, 2)).astype(np.float32); d = s + np.float32(3)
            srcs.append(s); dsts.append(d); offs.append(offs[-1] + n)
        out = ctx.find_homography_batch(np.concatenate(srcs), np.concatenate(dsts), offs, max_iters=case["max_iters"],
                                        want_ransac_mask=True)
        for k, n in enumerate(case["sizes"]):
            a, b = offs[k], offs[k + 1]
            if n < 4:
                assert not out["found"][k]
                continue
            ref = oracle.find_homography(srcs[k], dsts[k], max_iters=case["max_iters"])
            assert out["found"][k] == ref["found"], (case["max_iters"], k, n)
            assert np.array_equal(out["ransac_mask"][a:b], ref["ransac_mask"]), (case["max_iters"], k, n)
            if n > 4:
                assert out["iters"][k] == ref["info"]["iters_run"], (case["max_iters"], k, n)
            if ref["found"] and n < 100:
                assert np.array_equal(out["mask"][a:b], ref["mask"]), (case["max_iters"], k, n)
                assert np.allclose(out["H"][k], ref["H"], rtol=1e-9, atol=1e-12), (case["max_iters"], k, n)


def test_find_homography_batch_more_sets_than_a_grid_dimension(ctx, oracle):
    """70 000 sets in one call (more than gridDim.y can hold): every kernel of the verify stage indexes sets on x.  The
    same 40 correspondence sets repeated; every copy must give the first copy's result, the first 40 the oracle's."""
    rng = np.random.default_rng(9090)
    base = [synth.correspondences(rng, int(n), 0.6)[:2] for n in rng.integers(6, 14, size=40)]
    reps = 1750
    srcs = [b[0] for b in base] * reps; dsts = [b[1] for b in base] * reps
    offs = np.concatenate([[0], np.cumsum([len(s) for s in srcs])])
    out = ctx.find_homography_batch(np.concatenate(srcs), np.concatenate(dsts), offs, max_iters=300)
    per = offs[40]
    m0 = out["mask"][:per]
    assert np.array_equal(out["mask"].reshape(reps, per), np.broadcast_to(m0, (reps, per)))
    assert np.array_equal(out["H"].reshape(reps, 40, 9), np.broadcast_to(out["H"][:40].reshape(40, 9), (reps, 40, 9)))
    assert np.array_equal(out["found"].reshape(reps, 40), np.broadcast_to(out["found"][:40], (reps, 40)))
    for k in range(40):
        ref = oracle.find_homography(base[k][0], base[k][1], max_iters=300)
        assert out["found"][k] == ref["found"], k
        if ref["found"]:
            assert np.array_equal(out["mask"][offs[k]:offs[k + 1]], ref["mask"]), k
            assert np.allclose(out["H"][k], ref["H"], rtol=1e-9, atol=1e-12), k


def test_selftest_reciprocal_exhaustive(ctx):
    """The scoring kernel's hand-written reciprocal (MUFU.RCP + one Newton step, four at a time behind one range test)
    against __frcp_rn and 1.f / x on every float with 2^-126 <= |x| < 2^126: 0 mismatches of 2 x 4.2e9 comparisons."""
    assert ctx.selftest(0) == 0


def test_chunked_sampler_huge_single_round(ctx, api, oracle):
    """max_iters >= 32768 without early stop: the draw stream is walked by many CTAs at once (per-chunk entry -> exit
    maps composed in order give every chunk its true entry; accepted only if exit(c-1) == entry(c)).  The result must
    be the serial loop's: at 4-5 % inliers the reference's adaptive niters never drops below max_iters, so its loop is
    exhaustive.  last_sampler_serial_sets says how many sets the chunked sampler gave up on: none here."""
    rng = np.random.default_rng(6100)
    srcs, dsts, offs, refs = [], [], [0], []
    for n, rho in ((600, 0.05), (300, 0.04), (4, 1.0), (2000, 0.03), (7, 0.6)):
        s, d, _ = synth.correspondences(rng, n, rho)
        srcs.append(s); dsts.append(d); offs.append(offs[-1] + n)
    iters = 70000
    out = ctx.find_homography_batch(np.concatenate(srcs), np.concatenate(dsts), offs, max_iters=iters,
                                    flags=api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE)
    assert ctx.last_sampler_serial_sets == 0
    for k, (s, d) in enumerate(zip(srcs, dsts)):
        a, b = offs[k], offs[k + 1]
        if len(s) == 4:
            assert out["found"][k] and out["mask"][a:b].all()
            continue
        ref = oracle.ransac_stage(s, d, max_iters=iters)
        if ref["info"]["iters_run"] != iters:
            continue                                             # the reference stopped early on this set: not comparable
        assert out["found"][k] == ref["found"], k
        assert np.array_equal(out["mask"][a:b], ref["mask"]), k
        assert np.array_equal(out["H"][k], ref["H"]), k
        refs.append(k)
    assert len(refs) >= 3
    # many correspondences: nearly every attempt consumes exactly four draws, chains of different phase never meet
    s8, d8, _ = synth.correspondences(rng, 8192, 0.02)
    ref = oracle.ransac_stage(s8, d8, max_iters=40000)
    assert ref["info"]["iters_run"] == 40000
    H, mask = ctx.find_homography(s8, d8, max_iters=40000, flags=api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE)
    assert ctx.last_sampler_serial_sets == 0
    assert np.array_equal(mask, ref["mask"]) and np.array_equal(H, ref["H"])
    H, mask = ctx.find_homography(s8, d8, max_iters=2000)
    assert ctx.last_sampler_serial_sets == -1
    # a high-rejection set (most attempts fail checkSubset): long failure runs, the draw table is regrown
    n = 200
    src, dst, _ = synth.correspondences(rng, n, 0.5)
    line = rng.random(n) < 0.85
    t = rng.uniform(0, 600, size=int(line.sum())).astype(np.float32)
    src[line] = np.c_[t, 0.5 * t + 20]
    ref = oracle.ransac_stage(src, dst, max_iters=40000, conf=0.9999999)
    assert ref["info"]["iters_run"] == 40000
    H, mask = ctx.find_homography(src, dst, max_iters=40000, flags=api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE)
    assert np.array_equal(mask, ref["mask"]) and np.array_equal(H, ref["H"])


def test_rng_table_grows_on_high_rejection_rate(api, oracle):
    """85 % of the points on one line: ~95 % of the 4-point attempts fail checkSubset, so an iteration consumes ~80
    draws of the cv::RNG stream instead of ~5.  The draw table (48 per iteration) runs out, is regrown, and the verify
    stage repeats — the result must still be the oracle's."""
    rng = np.random.default_rng(8008)
    n = 200
    src, dst, _ = synth.correspondences(rng, n, 0.5)
    line = rng.random(n) < 0.85
    t = rng.uniform(0, 600, size=int(line.sum())).astype(np.float32)
    src[line] = np.c_[t, 0.5 * t + 20]                                    # collinear in src only: never inliers
    ref = oracle.find_homography(src, dst, max_iters=30000, conf=0.9999999)
    assert ref["info"]["draws"] > 30000 * 48 + (1 << 16)                 # really beyond the initial table
    with api.Context(0) as c:
        H, mask, rmask = c.find_homography(src, dst, max_iters=30000, confidence=0.9999999, want_ransac_mask=True)
    assert (H is not None) == ref["found"]
    assert np.array_equal(rmask, ref["ransac_mask"]) and np.array_equal(mask, ref["mask"])


def test_hypothesis_kernel_variants_agree(api):
    """CVG_HYP_MODE selects the kernel (1 warp, 2 eight-lane groups, 4 thread per hypothesis): identical counts ->
    identical winners, masks and H, checked through a subprocess per mode."""
    import json, os, subprocess, sys
    code = (
        "import sys, json, numpy as np\n"
        "sys.path.insert(0, %r)\n"
        "from computervision_objectdetection_featurematching_b200 import api, synth\n"
        "rng = np.random.default_rng(9009); srcs=[]; dsts=[]; offs=[0]\n"
        "for _ in range(40):\n"
        "    n = int(rng.integers(4, 400)); s, d, _ = synth.correspondences(rng, n, float(rng.uniform(0.2, 0.9)), dup=float(rng.choice([0, 0.4])))\n"
        "    srcs.append(s); dsts.append(d); offs.append(offs[-1] + n)\n"
        "c = api.Context(0); o = c.find_homography_batch(np.concatenate(srcs), np.concatenate(dsts), offs, want_ransac_mask=True)\n"
        "import hashlib\n"
        "print(json.dumps({k: hashlib.sha256(np.ascontiguousarray(o[k]).tobytes()).hexdigest() for k in ('H','mask','ransac_mask','iters','found')}))\n"
    ) % os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    digests = []
    for mode in ("1", "2", "4"):
        env = dict(os.environ, CVG_HYP_MODE=mode)
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, env=env, timeout=600)
        assert r.returncode == 0, r.stderr[-2000:]
        digests.append(json.loads(r.stdout.strip().splitlines()[-1]))
    assert digests[0] == digests[1] == digests[2]


# ---------------------------------------------------------------- fused path on real features
def test_detect_pairs_real_dataset_vs_cv2_goldens(ctx, api, feats, gpairs):
    """Golden real pairs (89 views x 10 scene-scales): gate status, counts, inlier masks (through the
    inlier scene points) and H against cv2 4.13.0."""
    md = feats["model_desc"].astype(np.float32)
    models = ctx.upload_models(md, feats["model_kpt"], feats["view_offsets"], feats["view_model"])
    so = feats["scene_offsets"]; vo = feats["view_offsets"]
    moff = gpairs["mask_offsets"]
    V = len(vo) - 1
    scales = feats["scales"]
    n_acc = 0
    for s in range(len(so) - 1):
        t = feats["scene_desc"][so[s]:so[s + 1]].astype(np.float32)
        tk = feats["scene_kpt"][so[s]:so[s + 1]]
        scale = float(scales[s % 5])
        res, inl, ioff = ctx.detect_pairs(models, t, tk, scale=scale)
        assert ctx.last_match_path == api.PATH_TENSOR
        assert np.array_equal(res["status"], gpairs["status"][s].astype(np.int32)), s
        assert np.array_equal(res["n_good"], gpairs["n_good"][s]), s
        idx = gpairs["idx"][s].astype(np.int32); acc = gpairs["accept"][s]
        for v in range(V):
            st = int(gpairs["status"][s, v])
            if st in (0, 3, 4):
                assert res["n_inliers"][v] == gpairs["n_inliers"][s, v], (s, v)
                G = gpairs["H"][s, v]
                rel = np.max(np.abs(res["H"][v] - G) / np.maximum(np.abs(G), 1e-12))
                assert rel < 1e-5, (s, v, rel)
            if st == 0:
                n_acc += 1
                sel = np.nonzero(acc[vo[v]:vo[v + 1]])[0] + vo[v]
                gmask = gpairs["mask"][moff[s * V + v]:moff[s * V + v + 1]].astype(bool)
                pts = tk[idx[sel, 0]][gmask]
                if np.float32(scale) != np.float32(1.0):
                    pts = pts / np.float32(scale)
                assert np.array_equal(inl[ioff[v]:ioff[v + 1]], pts.astype(np.float32)), (s, v)
            else:
                assert ioff[v + 1] == ioff[v]
    assert n_acc == int((gpairs["status"] == 0).sum())
    models.free()


def test_detect_scenes_resident_equals_per_scene_calls(ctx, feats, gpairs):
    md = feats["model_desc"].astype(np.float32)
    models = ctx.upload_models(md, feats["model_kpt"], feats["view_offsets"], feats["view_model"])
    so = feats["scene_offsets"]
    scenes = ctx.upload_scenes(feats["scene_desc"].astype(np.float32), feats["scene_kpt"], so)
    scales = np.tile(feats["scales"], (len(so) - 1) // 5)
    res = ctx.detect_scenes(models, scenes, scales=scales)
    assert np.array_equal(res["status"], gpairs["status"].astype(np.int32))
    assert np.array_equal(res["n_inliers"][gpairs["status"] == 0], gpairs["n_inliers"][gpairs["status"] == 0])
    scenes.free(); models.free()


def test_async_upload_pipeline_equals_sync(ctx, feats, api):
    """cvg_scenes_upload_async (copy stream, device-side path decision) + cvg_detect_scenes == the synchronous
    upload, for integer (tensor path) and non-integer (exact path) scene batches, two batches in flight."""
    md = feats["model_desc"].astype(np.float32)
    models = ctx.upload_models(md, feats["model_kpt"], feats["view_offsets"], feats["view_model"])
    so = feats["scene_offsets"]
    n_sc = min(10, len(so) - 1)
    off = np.asarray(so[:n_sc + 1], np.int64)
    d_int = np.ascontiguousarray(feats["scene_desc"][:off[-1]].astype(np.float32))
    kp = np.ascontiguousarray(feats["scene_kpt"][:off[-1]].astype(np.float32))
    d_flt = d_int.copy(); d_flt[::7, 3] += 0.25                          # non-integer rows -> candidate path
    want = []
    for d in (d_int, d_flt):
        sc = ctx.upload_scenes(d, kp, off)
        want.append(ctx.detect_scenes(models, sc).copy()); sc.free()
    a = ctx.upload_scenes_async(d_int, kp, off)
    b = ctx.upload_scenes_async(d_flt, kp, off)                           # second upload in flight during detect(a)
    ra = ctx.detect_scenes(models, a).copy(); pa = ctx.last_match_path
    rb = ctx.detect_scenes(models, b).copy(); pb = ctx.last_match_path
    b.wait()
    a.free(); b.free()
    u = ctx.upload_scenes_u8_async(d_int.astype(np.uint8), kp, off)      # uint8 rows: same results as their fp32 form
    ru = ctx.detect_scenes(models, u).copy(); u.free()
    assert np.array_equal(ru["status"], want[0]["status"]) and np.array_equal(ru["H"], want[0]["H"])
    assert pa == api.PATH_TENSOR and pb == api.PATH_TENSOR_RERANK
    for got, w in zip((ra, rb), want):
        assert np.array_equal(got["status"], w["status"]) and np.array_equal(got["n_inliers"], w["n_inliers"])
        assert np.array_equal(got["H"], w["H"])
    models.free()


def test_contexts_on_concurrent_host_threads(api, feats, gpairs):
    """The library's concurrency model: a context is not re-entrant, callers that want concurrency create one context per
    host thread (include/cvgraft.h).  Three contexts on three threads, each running the fused path over the same scenes
    several times while the others run too, must all reproduce the cv2 gate decisions."""
    import threading
    md = feats["model_desc"].astype(np.float32)
    so = feats["scene_offsets"]
    scales = np.tile(feats["scales"], (len(so) - 1) // 5)
    sd = feats["scene_desc"].astype(np.float32)
    want = gpairs["status"].astype(np.int32)
    errors = []

    def work(i):
        try:
            with api.Context(0) as c:
                models = c.upload_models(md, feats["model_kpt"], feats["view_offsets"], feats["view_model"])
                for rep in range(3):
                    sc = c.upload_scenes_async(sd, feats["scene_kpt"], so) if (rep + i) % 2 else c.upload_scenes(sd, feats["scene_kpt"], so)
                    res = c.detect_scenes(models, sc, scales=scales)
                    sc.free()
                    if not np.array_equal(res["status"], want):
                        errors.append((i, rep, int((res["status"] != want).sum())))
                models.free()
        except Exception as e:                                  # noqa: BLE001
            errors.append((i, repr(e)))
    th = [threading.Thread(target=work, args=(i,)) for i in range(3)]
    [t.start() for t in th]; [t.join() for t in th]
    assert not errors, errors


def test_full_dataset_stored_scenes_vs_cv2(ctx, feats):
    """The reference's loop nest (5 scales x 89 views per test image, src/TestsDetector.cpp:38,58,99-100) on the two test
    images whose features are stored (features_small.npz), against cv2 4.13.0's results for the same pairs taken from its
    run over the whole dataset (tests/golden/full_dataset_cv2.npz, written by tools/full_dataset_replay.py --cv2)."""
    import os
    root = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
    Z = feats
    G = np.load(os.path.join(root, "tests", "golden", "full_dataset_cv2.npz"))
    so = Z["scene_offsets"]; K = len(Z["scales"])
    names = list(G["scene_names"])
    rows = np.concatenate([K * names.index(n) + np.arange(K) for n in Z["scene_names"]])     # golden rows of the stored scenes
    scales = np.tile(Z["scales"], (len(so) - 1) // K)
    models = ctx.upload_models(Z["model_desc"].astype(np.float32), Z["model_kpt"], Z["view_offsets"], Z["view_model"])
    scenes = ctx.upload_scenes(Z["scene_desc"].astype(np.float32), Z["scene_kpt"], so)
    res = ctx.detect_scenes(models, scenes, scales=scales)
    V = res.shape[1]
    assert res.shape == (10, 89) and G["status"].shape == (150, 89)
    assert np.array_equal(res["status"], G["status"][rows].astype(np.int32))                  # 890 gate decisions
    assert np.array_equal(res["n_good"], G["n_good"][rows])
    has_h = np.isin(G["status"][rows], (0, 3, 4))
    assert np.array_equal(res["n_inliers"][has_h], G["n_inliers"][rows][has_h])
    rel = np.abs(res["H"][has_h] - G["H"][rows][has_h]) / np.maximum(np.abs(G["H"][rows][has_h]), 1e-12)
    assert rel.max() < 1e-5
    # what the reference consumes (src/TestsDetector.cpp:87-94): the inlier scene points of the accepted pairs, divided by
    # the scale, pair after pair — bit for bit cv2's
    res2, xy, off = ctx.detect_scenes_inliers(models, scenes, scales=scales)
    assert res2.tobytes() == res.tobytes()
    gpairs = (rows[:, None] * V + np.arange(V)).ravel()
    goff = G["inlier_offsets"]
    want_xy = np.concatenate([G["inlier_xy"][goff[p]:goff[p + 1]] for p in gpairs])
    assert np.array_equal(np.diff(off), goff[gpairs + 1] - goff[gpairs])
    assert np.array_equal(xy, want_xy) and len(xy) > 0
    scenes.free()
    # the returned inlier MASK of every pair that reaches findHomography (:78), accepted or not: the pairs' correspondences are
    # rebuilt from the match stage and verified in one batch per scaled scene
    vo = Z["view_offsets"]; mk = Z["model_kpt"]
    gmask = np.unpackbits(G["mask"])[:G["mask_offsets"][-1]]; moff = G["mask_offsets"]
    n_masks = 0
    for s in range(0, len(so) - 1):
        r = rows[s]
        t = Z["scene_desc"][so[s]:so[s + 1]].astype(np.float32); tk = Z["scene_kpt"][so[s]:so[s + 1]]
        idx, dist, acc = ctx.match_knn2(models, t)
        src, dst, offs, views = [], [], [0], []
        for v in range(V):
            sel = np.nonzero(acc[vo[v]:vo[v + 1]])[0] + vo[v]
            assert len(sel) == G["n_good"][r, v]
            if len(sel) >= 4:
                src.append(mk[sel]); dst.append(tk[idx[sel, 0]]); offs.append(offs[-1] + len(sel)); views.append(v)
        if not views:
            continue
        out = ctx.find_homography_batch(np.concatenate(src), np.concatenate(dst), offs)
        for k, v in enumerate(views):
            a, b = moff[r * V + v], moff[r * V + v + 1]
            assert np.array_equal(out["mask"][offs[k]:offs[k + 1]], gmask[a:b]), (s, v)
            assert bool(out["found"][k]) == (G["status"][r, v] != 2)
            n_masks += 1
    assert n_masks == int((G["n_good"][rows] >= 4).sum()) > 0  # every pair with >= 4 matches
    models.free()
