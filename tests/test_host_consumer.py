"""C++ host consumer stages (host/detect_objects.cpp: cluster -> box -> merge -> area filter, the reference's
src/TestsDetector.cpp:112-248 restated without OpenCV) against an independent numpy/scipy restatement, and the
cv::boundingRect model against cv2 goldens."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))


@pytest.fixture(scope="module")
def host():
    from computervision_objectdetection_featurematching_b200 import build
    build.build()
    subprocess.check_call(["make", "-s", "-C", os.path.join(ROOT, "host"), "libcvghost_consumer.so"])
    return C.CDLL(os.path.join(ROOT, "host", "libcvghost_consumer.so"))


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def py_consume(pts):
    """-> list of (x, y, w, h) or None when a margin sits on an integer boundary (summation-order sensitive)."""
    n = len(pts)
    if n == 0:
        return []
    d = np.sqrt(((pts[:, None, :].astype(np.float64) - pts[None, :, :].astype(np.float64)) ** 2).sum(-1)).astype(np.float32)
    adj = coo_matrix(d <= np.float32(20.0))
    ncomp, lab = connected_components(adj, directed=False)
    boxes = []
    for c in range(ncomp):
        m = pts[lab == c]
        if len(m) < 18:
            continue
        x0 = int(np.floor(m[:, 0].min())); y0 = int(np.floor(m[:, 1].min()))
        x1 = int(np.floor(m[:, 0].max())); y1 = int(np.floor(m[:, 1].max()))
        dd = np.sqrt(((m[:, None, :].astype(np.float64) - m[None, :, :].astype(np.float64)) ** 2).sum(-1))
        iu = np.triu_indices(len(m), 1)
        sd = float(np.sqrt(((dd[iu].astype(np.float32) - dd[iu].astype(np.float32).mean()) ** 2).mean()))
        if abs(sd - round(sd)) < 1e-3 or abs(2 * sd - round(2 * sd)) < 1e-3:
            return None
        boxes.append((x0 - int(sd), y0 - int(sd), x1 - x0 + 1 + int(2 * sd), y1 - y0 + 1 + int(2 * sd)))
    # merge: chains of boxes whose centres are within 250
    if not boxes:
        return []
    cen = np.array([[b[0] + b[2] / 2.0, b[1] + b[3] / 2.0] for b in boxes], np.float32)
    dc = np.sqrt(((cen[:, None, :].astype(np.float64) - cen[None, :, :].astype(np.float64)) ** 2).sum(-1))
    ng, gl = connected_components(coo_matrix(dc <= 250.0), directed=False)
    out = []
    for g in range(ng):
        bs = [boxes[i] for i in range(len(boxes)) if gl[i] == g]
        x0 = min(b[0] for b in bs); y0 = min(b[1] for b in bs)
        x1 = max(b[0] + b[2] for b in bs); y1 = max(b[1] + b[3] for b in bs)
        if (x1 - x0) * (y1 - y0) >= 2500:
            out.append((x0, y0, x1 - x0, y1 - y0))
    return sorted(out)


def test_bounding_rect_matches_cv2(host):
    """Against cv2.boundingRect of the same point sets (tests/golden/golden_rect.npz, make_golden.py rect_cases)."""
    want = np.load(os.path.join(ROOT, "tests", "golden", "golden_rect.npz"))["rect"]
    rng = np.random.default_rng(0)
    for k in range(500):
        p = rng.uniform(-50, 700, size=(int(rng.integers(1, 40)), 2)).astype(np.float32)
        if rng.random() < 0.3:
            p = np.round(p)
        out = np.zeros(4, np.int32)
        host.cvh_bounding_rect(_p(p), len(p), _p(out))
        assert tuple(out) == tuple(want[k]), k


def test_cluster_box_merge_filter(host):
    rng = np.random.default_rng(1)
    checked = 0
    for case in range(300):
        k = int(rng.integers(1, 5))
        parts = []
        for _ in range(k):
            c = rng.uniform([50, 50], [590, 430])
            parts.append(c + rng.normal(0, rng.uniform(3, 25), size=(int(rng.integers(5, 80)), 2)))
        parts.append(rng.uniform([0, 0], [640, 480], size=(int(rng.integers(0, 30)), 2)))     # stray points
        pts = np.concatenate(parts).astype(np.float32)
        pts = pts[rng.permutation(len(pts))]
        want = py_consume(pts)
        if want is None:
            continue
        boxes = np.zeros((16, 4), np.int32)
        n = host.cvh_consume_points(_p(pts), len(pts), _p(boxes), 16)
        got = sorted(tuple(int(v) for v in boxes[i]) for i in range(n))
        assert got == want, case
        checked += 1
    assert checked > 250


def test_results_file_layout(host, tmp_path):
    """saveDetections: 'name xmin ymin xmax ymax' (reference src/utils.cpp:12-20) — exercised through cvg_replay on
    the GPU box (tests/test_gpu_replay.py); here only that the consumer library exposes the stages."""
    assert hasattr(host, "cvh_consume_points") and hasattr(host, "cvh_bounding_rect")
