"""Hypothesis-range sharded RANSAC (cvg_find_homography_sharded): one point set, the hypotheses of every round split
over the devices of a multi-device context, one all-gather of inlier counts per round.  The result must be the bytes of
cvg_find_homography_batch for that one set on a single-device context, for every parameter set and flag.  With one GPU
visible the devices are logical (the GPU listed 2-4 times, exchange by device-to-device copies); with more GPUs the
distinct-device lists exchange through NCCL, and once more through copies with CVG_NO_NCCL=1."""
import numpy as np
import pytest

from computervision_objectdetection_featurematching_b200 import synth

pytestmark = pytest.mark.gpu

KEYS = ("H", "mask", "found", "iters", "ransac_mask")


@pytest.fixture(scope="module")
def api():
    from computervision_objectdetection_featurematching_b200 import api as _api
    return _api


@pytest.fixture(scope="module")
def ref_ctx(api):
    with api.Context(0) as c:
        yield c


def _n_gpus():
    import torch
    return torch.cuda.device_count()


def _device_lists():
    """(devices, no_nccl) pairs: logical shards on one GPU always, distinct GPUs (NCCL, then copies) when visible."""
    lists = [([0], False), ([0, 0], False), ([0, 0, 0], False), ([0, 0, 0, 0], False)]
    n = _n_gpus()
    if n >= 2:
        lists += [([0, 1], False), ([0, 1], True)]
    if n >= 4:
        lists.append(([0, 1, 2, 3], False))
    return lists


@pytest.fixture(params=_device_lists(), ids=lambda p: "-".join(map(str, p[0])) + ("-nonccl" if p[1] else ""))
def multi(api, request, monkeypatch):
    devs, no_nccl = request.param
    if no_nccl:
        monkeypatch.setenv("CVG_NO_NCCL", "1")                  # read when the context is created
    with api.Context(devs) as c:
        if no_nccl or devs.count(devs[0]) > 1:
            assert c.exchange_kind == "memcpy"
        yield c


def _reference(ctx, src, dst, **kw):
    out = ctx.find_homography_batch(src, dst, [0, len(src)], want_ransac_mask=True, **kw)
    return {"H": out["H"][0], "mask": out["mask"], "found": bool(out["found"][0]), "iters": int(out["iters"][0]),
            "ransac_mask": out["ransac_mask"]}


def _same(got, ref, what=""):
    for k in KEYS:
        a, b = np.asarray(got[k]), np.asarray(ref[k])
        assert a.dtype == b.dtype and a.shape == b.shape and a.tobytes() == b.tobytes(), (what, k)


def _sharded(ctx, src, dst, **kw):
    return ctx.find_homography_sharded(src, dst, want_ransac_mask=True, **kw)


# ---------------------------------------------------------------- 1. adaptive stop, one round
_ONE_ROUND = [(n, rho, 100 + i) for i, (n, rho) in enumerate(((5, 0.9), (32, 0.6), (127, 0.3), (600, 0.5), (8192, 0.3),
                                                               (600, 0.9), (127, 0.7)))]


@pytest.fixture(scope="module")
def one_round_cases(oracle):
    cases = []
    for n, rho, seed in _ONE_ROUND:
        s, d, _ = synth.correspondences(np.random.default_rng(seed), n, rho)
        cases.append((s, d, oracle.find_homography(s, d)))
    return cases


def test_adaptive_one_round(multi, ref_ctx, one_round_cases):
    for s, d, orc in one_round_cases:
        got = _sharded(multi, s, d)
        _same(got, _reference(ref_ctx, s, d), len(s))
        assert multi.last_exchange()[0] == 1
        assert got["found"] == orc["found"] and np.array_equal(got["ransac_mask"], orc["ransac_mask"]), len(s)
        if len(s) > 4:
            assert got["iters"] == orc["info"]["iters_run"], len(s)
        if orc["found"] and len(s) < 100:
            assert np.array_equal(got["mask"], orc["mask"])
            assert np.allclose(got["H"], orc["H"], rtol=1e-9, atol=1e-12)


# ---------------------------------------------------------------- 2. adaptive stop, several rounds
@pytest.fixture(scope="module")
def multi_round_cases(oracle):
    """n = 600, confidence 0.9999999, max_iters 200 000: at 5 % inliers niters stays at the cap (every round runs);
    at 12 % it drops to ~73 500 inside the second round of two devices, and the later rounds exit early everywhere."""
    cases = []
    for seed, rho in ((7001, 0.05), (7002, 0.12)):
        s, d, _ = synth.correspondences(np.random.default_rng(seed), 600, rho)
        cases.append((s, d, oracle.ransac_stage(s, d, conf=0.9999999, max_iters=200000)))
    assert cases[0][2]["info"]["iters_run"] == 200000
    assert 66304 < cases[1][2]["info"]["iters_run"] < 132608
    return cases


def _check_multi_round(ctx, ref_ctx, cases):
    kw = dict(confidence=0.9999999, max_iters=200000)
    for s, d, orc in cases:
        got = _sharded(ctx, s, d, **kw)
        _same(got, _reference(ref_ctx, s, d, **kw))
        G = ctx.n_devices
        assert ctx.last_exchange()[0] >= (3 if G <= 3 else 2)
        assert got["iters"] == orc["info"]["iters_run"]
        assert np.array_equal(got["ransac_mask"], orc["mask"])


def test_adaptive_several_rounds(multi, ref_ctx, multi_round_cases):
    _check_multi_round(multi, ref_ctx, multi_round_cases)


# ---------------------------------------------------------------- 3. no early stop, chunked sampler
@pytest.fixture(scope="module")
def huge_round(oracle):
    s, d, _ = synth.correspondences(np.random.default_rng(7010), 8192, 0.02)
    orc = oracle.ransac_stage(s, d, max_iters=40000)
    assert orc["info"]["iters_run"] == 40000                      # the reference's loop is the exhaustive one
    return s, d, orc


def test_no_early_stop_chunked_sampler(api, multi, ref_ctx, huge_round):
    s, d, orc = huge_round
    flags = api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE
    got = _sharded(multi, s, d, max_iters=40000, flags=flags)
    assert multi.last_sampler_serial_sets == 0                    # the chunked sampler served the first device
    assert multi.last_exchange()[0] == 1
    _same(got, _reference(ref_ctx, s, d, max_iters=40000, flags=flags))
    assert np.array_equal(got["mask"], orc["mask"]) and np.array_equal(got["H"], orc["H"])
    got = _sharded(multi, s, d, max_iters=40000, flags=api.RANSAC_NO_EARLY_STOP)          # with refit / LM
    _same(got, _reference(ref_ctx, s, d, max_iters=40000, flags=api.RANSAC_NO_EARLY_STOP))


# ---------------------------------------------------------------- 4. first maximum wins across a shard boundary
def test_first_maximum_wins_across_shards(api, ref_ctx, oracle):
    """A set whose largest count occurs at several iterations, the first of them outside slice 0 for 2, 3 and 4 devices
    (one round of 2000 iterations: slices of 1000, 667, 500): every device count must pick the oracle's first one."""
    pick = None
    for seed in range(60):
        s, d, _ = synth.correspondences(np.random.default_rng(seed), 30, 0.2)
        tr = oracle.ransac_stage(s, d, conf=0.9999999, max_iters=2000, want_trace=True)
        c = tr["counts"][:tr["info"]["iters_run"]]
        pos = np.nonzero(c == c.max())[0] if len(c) else []
        if len(pos) >= 2 and pos[0] >= 1000 and c.max() >= 4:
            pick = (s, d, tr)
            break
    assert pick is not None, "no seed with a repeated maximum beyond the first slice"
    s, d, tr = pick
    assert tr["info"]["best_iter"] == np.nonzero(tr["counts"] == tr["counts"].max())[0][0]
    for devs in ([0, 0], [0, 0, 0], [0, 0, 0, 0]):
        with api.Context(devs) as c:
            got = _sharded(c, s, d, confidence=0.9999999)
            _same(got, _reference(ref_ctx, s, d, confidence=0.9999999))
            assert np.array_equal(got["ransac_mask"], tr["mask"]) and got["iters"] == tr["info"]["iters_run"]


# ---------------------------------------------------------------- 5. niters answered by the host on every device
def test_niters_all_on_host(api, ref_ctx, multi_round_cases):
    """CVG_NITERS_ALL_ON_HOST: every RANSACUpdateNumIters evaluation is answered by the host and the verify stage repeats
    with the table; a device left without the table would ask forever."""
    for devs, _ in _device_lists():
        with api.Context(devs, api.NITERS_ALL_ON_HOST) as c:
            _check_multi_round(c, ref_ctx, multi_round_cases)


# ---------------------------------------------------------------- 6. the draw table grows during the call
def test_draw_table_grows(api, ref_ctx, oracle):
    """85 % of the points on one line: most 4-point attempts fail checkSubset, the table of 48 draws per iteration runs
    out and every device regrows it to the same length.  Run once more on a context whose first device already holds a
    longer table than the others (a find_homography call with a larger max_iters runs on the first device only)."""
    rng = np.random.default_rng(8008)
    n = 200
    src, dst, _ = synth.correspondences(rng, n, 0.5)
    line = rng.random(n) < 0.85
    t = rng.uniform(0, 600, size=int(line.sum())).astype(np.float32)
    src[line] = np.c_[t, 0.5 * t + 20]
    kw = dict(max_iters=30000, confidence=0.9999999)
    orc = oracle.find_homography(src, dst, max_iters=30000, conf=0.9999999)
    assert orc["info"]["draws"] > 30000 * 48 + (1 << 16)
    ref = _reference(ref_ctx, src, dst, **kw)
    for devs, _ in _device_lists():
        with api.Context(devs) as c:
            got = _sharded(c, src, dst, **kw)
            _same(got, ref, devs)
            assert got["found"] == orc["found"]
            assert np.array_equal(got["ransac_mask"], orc["ransac_mask"]) and np.array_equal(got["mask"], orc["mask"])
    with api.Context([0, 0, 0]) as c:
        c.find_homography(src, dst, max_iters=120000, confidence=0.9999999)
        _same(_sharded(c, src, dst, **kw), ref, "longer table on the first device")


# ---------------------------------------------------------------- 7. edges
def test_edges(api, multi, ref_ctx):
    rng = np.random.default_rng(4242)
    s, d, _ = synth.correspondences(rng, 50, 0.6)
    for it in (1, 2, 3):                                          # fewer iterations than devices: empty slices
        _same(_sharded(multi, s, d, max_iters=it), _reference(ref_ctx, s, d, max_iters=it), it)
    s4, d4, _ = synth.correspondences(rng, 4, 1.0)
    got = _sharded(multi, s4, d4)
    _same(got, _reference(ref_ctx, s4, d4))
    assert got["found"] and got["mask"].all()
    xs = np.linspace(0, 100, 12).astype(np.float32)
    for a, b in ((np.c_[xs, 2 * xs], np.c_[xs + 5, 2 * xs + 1]),                                  # all collinear
                 (np.full((12, 2), 7, np.float32), np.full((12, 2), 9, np.float32))):             # all identical
        got = _sharded(multi, a, b)
        _same(got, _reference(ref_ctx, a, b))
        assert not got["found"] and not got["mask"].any()
    with pytest.raises(api.CvgError) as e:
        multi.find_homography_sharded(np.zeros((3, 2), np.float32), np.zeros((3, 2), np.float32))
    assert e.value.code == 3


def test_needs_a_multi_device_context(api, ref_ctx):
    s, d, _ = synth.correspondences(np.random.default_rng(1), 40, 0.5)
    with pytest.raises(api.CvgError) as e:
        ref_ctx.find_homography_sharded(s, d)
    assert e.value.code == 1
    assert ref_ctx.last_exchange() == (0, 0.0)
    with api.Context([0, 0]) as c:
        assert c.last_exchange() == (0, 0.0)


def test_timing_fields(api, ref_ctx):
    """With timing on, the first device reports its verify stage, solve and score kernels and the exchange time."""
    s, d, _ = synth.correspondences(np.random.default_rng(5), 2000, 0.05)
    kw = dict(max_iters=100000, confidence=0.9999999)
    with api.Context([0, 0]) as c:
        c.set_timing(True)
        got = _sharded(c, s, d, **kw)
        k, ms = c.last_exchange()
        tm = c.last_timing()
    _same(got, _reference(ref_ctx, s, d, **kw))
    assert k >= 2 and ms > 0
    assert tm["ransac_ms"] > tm["hyp_ms"] > 0 and tm["score_ms"] > 0 and tm["hyp_launches"] == k


# ---------------------------------------------------------------- 8. sharded calls do not disturb the other entry points
def test_interleaved_with_other_entry_points(api, ref_ctx):
    rng = np.random.default_rng(31)
    sets = [synth.correspondences(rng, n, rho)[:2] for n, rho in ((300, 0.4), (8192, 0.3), (60, 0.7), (2500, 0.1))]
    src_b = np.concatenate([s for s, _ in sets]); dst_b = np.concatenate([d for _, d in sets])
    off_b = np.cumsum([0] + [len(s) for s, _ in sets])
    q, qk, t, tk, _, _ = synth.image_pair(rng, 700, 1500, p_match=0.5, inlier_ratio=0.5)

    def detect(c):
        m = c.upload_models(q, qk, [0, 300, 700], [0, 0])
        sc = c.upload_scenes(t, tk, [0, 700, 1500])
        out = c.detect_scenes_inliers(m, sc, scales=[1.0, 1.15])
        sc.free(); m.free()
        return out

    ref_det = detect(ref_ctx)
    ref_b = ref_ctx.find_homography_batch(src_b, dst_b, off_b, want_ransac_mask=True)
    for devs, _ in _device_lists():
        with api.Context(devs) as c:
            for k, (s, d) in enumerate(sets):
                it = (2000, 500, 30000, 50000)[k]
                _same(_sharded(c, s, d, max_iters=it), _reference(ref_ctx, s, d, max_iters=it), (devs, k))
                H, mask = c.find_homography(s, d)
                rH, rmask = ref_ctx.find_homography(s, d)
                assert np.array_equal(mask, rmask) and (H is None) == (rH is None) and (H is None or np.array_equal(H, rH))
                b = c.find_homography_batch(src_b, dst_b, off_b, want_ransac_mask=True)
                for key in ("H", "mask", "found", "iters", "ransac_mask"):
                    assert np.array_equal(b[key], ref_b[key]), (devs, key)
                res, inl, off = detect(c)
                assert res.tobytes() == ref_det[0].tobytes() and np.array_equal(inl, ref_det[1]) and np.array_equal(off, ref_det[2])
