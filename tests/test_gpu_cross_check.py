"""BFMatcher(NORM_L2, crossCheck=True).match on the GPU (cvg_match_cross_check / _raw) against cv2's goldens
(golden_crosscheck.npz) and the CPU oracle's mutual rule: exact indices and distance bytes on both match paths."""
import os
import sys

import numpy as np
import pytest

from computervision_objectdetection_featurematching_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
import crosscheck_cases  # noqa: E402

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


@pytest.fixture(scope="module")
def golden():
    return crosscheck_cases.load_golden()


def _same(got, want_idx, want_dist):
    idx, dist = got
    assert np.array_equal(idx, want_idx)
    assert np.array_equal(dist.view(np.uint32), np.asarray(want_dist, np.float32).view(np.uint32))


@pytest.mark.parametrize("tag", ["sat", "tie", "float", "small", "big"])
def test_goldens_raw(ctx, ctx_exact, api, golden, tag):
    sets, gi, gd, off = golden[tag]
    for k, (q, t) in enumerate(sets):
        want = gi[off[k]:off[k + 1]], gd[off[k]:off[k + 1]]
        _same(ctx.match_cross_check(q, t), *want)
        integer = bool(np.all(q == np.round(q)) and np.all(t == np.round(t)) and q.min() >= 0 and t.min() >= 0
                       and q.max() <= 255 and t.max() <= 255)
        assert ctx.last_match_path == (api.PATH_TENSOR if integer else api.PATH_EXACT), (tag, k)
        if tag != "big":
            _same(ctx_exact.match_cross_check(q, t), *want)
            assert ctx_exact.last_match_path == api.PATH_EXACT


def test_real_pairs_view_all_and_raw(ctx, ctx_exact, api, golden, feats):
    sets, gi, gd, off = golden["real"]
    vo = feats["view_offsets"]; so = feats["scene_offsets"]; V = len(vo) - 1
    m = ctx.upload_models(feats["model_desc"].astype(np.float32), feats["model_kpt"], vo)
    me = ctx_exact.upload_models(feats["model_desc"].astype(np.float32), feats["model_kpt"], vo)
    try:
        for s in range(len(so) - 1):
            t = feats["scene_desc"][so[s]:so[s + 1]].astype(np.float32)
            k0, k1 = s * V, (s + 1) * V
            want = gi[off[k0]:off[k1]], gd[off[k0]:off[k1]]
            _same(ctx.match_cross_check(m, t, view=-1), *want)          # every view its own query matrix
            assert ctx.last_match_path == api.PATH_TENSOR
            assert ctx.last_match_guard_rows == 0                       # SIFT rows stay below d = 2048
            if s == 0:
                _same(ctx_exact.match_cross_check(me, t, view=-1), *want)
                assert ctx_exact.last_match_path == api.PATH_EXACT
            for v in range(V):
                k = k0 + v
                want_v = gi[off[k]:off[k + 1]], gd[off[k]:off[k + 1]]
                _same(ctx.match_cross_check(m, t, view=v), *want_v)
                if v % 11 == s:
                    _same(ctx.match_cross_check(sets[k][0], t), *want_v)
    finally:
        m.free(); me.free()


def test_guard_redoes_saturated_rows(ctx, api, golden, oracle):
    sets, gi, gd, off = golden["sat"]
    q, t = sets[0]
    _same(ctx.match_cross_check(q, t), gi, gd)
    assert ctx.last_match_path == api.PATH_TENSOR
    assert ctx.last_match_guard_rows >= len(q)                          # every row (and column) is at d >= 2048
    rng = np.random.default_rng(9201)
    for nq, nt in [(333, 1000), (40, 3000), (700, 129)]:
        q, t = synth.saturated_pair(rng, nq, nt)
        _same(ctx.match_cross_check(q, t), *crosscheck_cases.mutual(oracle, q, t))
        assert ctx.last_match_guard_rows > 0


def test_random_sizes_against_oracle(ctx, ctx_exact, api, oracle):
    rng = np.random.default_rng(9202)
    for _ in range(12):
        nq, nt = int(rng.integers(1, 1500)), int(rng.integers(1, 2500))
        q, t, _ = synth.planted_pair(rng, nq, nt)
        want = crosscheck_cases.mutual(oracle, q, t)
        _same(ctx.match_cross_check(q, t), *want)
        assert ctx.last_match_path == api.PATH_TENSOR
        _same(ctx_exact.match_cross_check(q, t), *want)                 # the same bytes on the SIMT path
    q, t = synth.float_desc(rng, 517), synth.float_desc(rng, 901)
    _same(ctx.match_cross_check(q, t), *crosscheck_cases.mutual(oracle, q, t))
    assert ctx.last_match_path == api.PATH_EXACT


def test_zero_row_views_and_tiny_train(ctx, api, oracle):
    rng = np.random.default_rng(9203)
    rows = [0, 130, 0, 1, 255, 0, 129]
    vo = np.cumsum([0] + rows).astype(np.int32)
    q = synth.sift_like(rng, int(vo[-1]))
    m = ctx.upload_models(q, np.zeros((len(q), 2), np.float32), vo)
    try:
        for nt in (0, 1, 2, 300):
            t = synth.sift_like(rng, nt)
            idx, dist = ctx.match_cross_check(m, t, view=-1)
            for v in range(len(rows)):
                a, b = vo[v], vo[v + 1]
                want = crosscheck_cases.mutual(oracle, q[a:b], t)
                _same((idx[a:b], dist[a:b]), *want)
                _same(ctx.match_cross_check(m, t, view=v), *want)
            if nt == 0:
                assert np.all(idx == -1) and np.all(dist == 0)
            if nt == 1:
                assert (idx == 0).sum() == sum(1 for r in rows if r > 0)   # one match per non-empty view
        i, d = ctx.match_cross_check(np.zeros((0, 128), np.float32), synth.sift_like(rng, 5))
        assert i.shape == (0,) and d.shape == (0,)
    finally:
        m.free()


def test_rows_outside_every_view(ctx, oracle):
    rng = np.random.default_rng(9206)
    t = synth.sift_like(rng, 200)
    for vo in ([2, 50, 50], [3, 3]):
        q = synth.sift_like(rng, vo[-1])
        m = ctx.upload_models(q, None, vo)
        try:
            idx, dist = ctx.match_cross_check(m, t, view=-1)
            assert np.all(idx[:vo[0]] == -1) and np.all(dist[:vo[0]] == 0)
            _same((idx[vo[0]:vo[1]], dist[vo[0]:vo[1]]), *crosscheck_cases.mutual(oracle, q[vo[0]:vo[1]], t))
        finally:
            m.free()


def test_invalid_arguments(ctx, api):
    m = ctx.upload_models(np.zeros((4, 128), np.float32), None, [0, 4])
    try:
        t = np.zeros((3, 128), np.float32); idx = np.zeros(4, np.int32); dist = np.zeros(4, np.float32)
        for view in (1, -2):                                            # the view checks of cvg_match_knn2
            assert ctx.lib.cvg_match_cross_check(ctx.handle, m.handle, view, api._ptr(t), 3, api._ptr(idx), api._ptr(dist)) == 1
        assert ctx.lib.cvg_match_cross_check(ctx.handle, m.handle, 0, None, 3, api._ptr(idx), api._ptr(dist)) == 1
        assert ctx.lib.cvg_match_cross_check(ctx.handle, m.handle, 0, api._ptr(t), 3, None, api._ptr(dist)) == 1
        assert ctx.lib.cvg_match_cross_check_raw(ctx.handle, None, 5, api._ptr(t), 3, api._ptr(idx), api._ptr(dist)) == 1
    finally:
        m.free()


def test_interleaved_with_knn2(api, oracle):
    rng = np.random.default_rng(9204)
    q, t, _ = synth.planted_pair(rng, 1000, 1300)
    q2, t2, _ = synth.planted_pair(rng, 600, 2000)
    with api.Context(0) as fresh:
        k_ref = fresh.match_knn2(q, t)
        k2_ref = fresh.match_knn2(q2, t2)
    want = crosscheck_cases.mutual(oracle, q, t)
    with api.Context(0) as c:
        for _ in range(2):
            _same(c.match_cross_check(q, t), *want)
            for got, ref in zip(c.match_knn2(q, t), k_ref):
                assert np.array_equal(got, ref)
            for got, ref in zip(c.match_knn2(q2, t2), k2_ref):
                assert np.array_equal(got, ref)


def test_timing_reports_match_ms(ctx):
    rng = np.random.default_rng(9205)
    q, t, _ = synth.planted_pair(rng, 2048, 4096)
    ctx.lib.cvg_set_timing(ctx.handle, 1)
    try:
        ctx.match_cross_check(q, t)
        import ctypes as C
        m, r, tt = C.c_float(), C.c_float(), C.c_float()
        ctx.lib.cvg_last_timing(ctx.handle, C.byref(m), C.byref(r), C.byref(tt))
        assert m.value > 0 and r.value == 0
    finally:
        ctx.lib.cvg_set_timing(ctx.handle, 0)


def test_logical_multi_device_context(api, golden, feats):
    sets, gi, gd, off = golden["real"]
    vo = feats["view_offsets"]; so = feats["scene_offsets"]; V = len(vo) - 1
    with api.Context([0, 0]) as c:
        m = c.upload_models(feats["model_desc"].astype(np.float32), feats["model_kpt"], vo)
        t = feats["scene_desc"][so[3]:so[4]].astype(np.float32)
        _same(c.match_cross_check(m, t, view=-1), gi[off[3 * V]:off[4 * V]], gd[off[3 * V]:off[4 * V]])
        assert c.last_match_path == api.PATH_TENSOR
        q, t2 = sets[5]
        _same(c.match_cross_check(q, t2), gi[off[5]:off[6]], gd[off[5]:off[6]])
        m.free()
