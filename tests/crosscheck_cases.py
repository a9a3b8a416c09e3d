"""The query/train sets of the cross-check goldens (tests/golden/golden_crosscheck.npz, written by
tests/golden/make_golden_crosscheck.py): BFMatcher(NORM_L2, crossCheck=True).match.  Seeded sets are regenerated here,
the real pairs come from features_small.npz and the saturated rows from golden_sat.npz, so the golden file holds cv2's
outputs only.  TEST INFRASTRUCTURE."""
import os

import numpy as np

from computervision_objectdetection_featurematching_b200 import synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def real_pairs():
    """(view, scene) in scene-major order: the 890 (view, scaled scene) pairs of features_small.npz, query = the view's rows."""
    Z = np.load(os.path.join(GOLDEN_DIR, "features_small.npz"))
    q = Z["model_desc"].astype(np.float32); t = Z["scene_desc"].astype(np.float32)
    vo = Z["view_offsets"]; so = Z["scene_offsets"]
    for s in range(len(so) - 1):
        for v in range(len(vo) - 1):
            yield q[vo[v]:vo[v + 1]], t[so[s]:so[s + 1]]


def sat_pair():
    """golden_sat.npz's u8 rows: every distance is above 2048."""
    Z = np.load(os.path.join(GOLDEN_DIR, "golden_sat.npz"))
    return Z["q"].astype(np.float32), Z["t"].astype(np.float32)


def tie_sets():
    """Integer rows 0..2 in few columns: most distances tie, both tie rules decide."""
    rng = np.random.default_rng(9101)
    for _ in range(40):
        nq, nt = int(rng.integers(1, 300)), int(rng.integers(1, 300))
        cols = int(rng.integers(1, 6))
        q = np.zeros((nq, 128), np.float32); t = np.zeros((nt, 128), np.float32)
        q[:, :cols] = rng.integers(0, 3, (nq, cols)); t[:, :cols] = rng.integers(0, 3, (nt, cols))
        yield q, t


def float_sets():
    """N(0, 1) * 37 rows: the fp32 summation order of cv::batchDistance matters."""
    rng = np.random.default_rng(9102)
    for _ in range(12):
        nq, nt = int(rng.integers(1, 700)), int(rng.integers(1, 700))
        yield ((rng.standard_normal((nq, 128)) * 37).astype(np.float32),
               (rng.standard_normal((nt, 128)) * 37).astype(np.float32))


def small_sets():
    """n_train = 1 (several queries at the same minimum distance), n_query = 1, and the no-second-choice case: query 0's
    nearest train row prefers query 1, and query 0 gets no match although train row 1's nearest query is query 0."""
    rng = np.random.default_rng(9103)
    t1 = synth.sift_like(rng, 1)
    q1 = np.concatenate([synth.sift_like(rng, 5), t1 + 2, t1 + 1, t1 + 1]).clip(0, 255).astype(np.float32)
    yield q1, t1
    yield synth.sift_like(rng, 1), synth.sift_like(rng, 77)
    t = np.zeros((2, 128), np.float32); t[1, 0] = 10
    q = np.zeros((2, 128), np.float32); q[0, 0] = 1
    yield q, t


def big_pair():
    """An 8192 x 8192 SIFT-like pair with planted matches."""
    q, t, _ = synth.planted_pair(np.random.default_rng(9104), 8192, 8192)
    return q, t


def groups():
    """tag -> list of (query, train)"""
    return {"real": list(real_pairs()), "sat": [sat_pair()], "tie": list(tie_sets()), "float": list(float_sets()),
            "small": list(small_sets()), "big": [big_pair()]}


def mutual(oracle, q, t, nthreads=8):
    """The cross-check rule over the CPU oracle's knnMatch in both directions."""
    nq = len(q)
    idx = np.full(nq, -1, np.int32); dist = np.zeros(nq, np.float32)
    if nq == 0 or len(t) == 0:
        return idx, dist
    fi, fd = oracle.knn2(q, t, nthreads=nthreads)
    bi, _ = oracle.knn2(t, q, nthreads=nthreads)
    j = fi[:, 0]
    ok = (j >= 0) & (bi[np.maximum(j, 0), 0] == np.arange(nq))
    idx[ok] = j[ok]; dist[ok] = fd[ok, 0]
    return idx, dist


def load_golden():
    """tag -> (list of (query, train), idx, dist, offsets) with idx / dist concatenated over the group's sets"""
    Z = np.load(os.path.join(GOLDEN_DIR, "golden_crosscheck.npz"))
    out = {}
    for tag, sets in groups().items():
        off = np.cumsum([0] + [len(q) for q, _ in sets]).astype(np.int64)
        assert np.array_equal(off, Z[f"{tag}_offsets"]), tag
        out[tag] = (sets, Z[f"{tag}_idx"], Z[f"{tag}_dist"], off)
    return out
