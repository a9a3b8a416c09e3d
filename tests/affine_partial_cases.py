"""The point sets of the estimateAffinePartial2D goldens (tests/golden/golden_affine_partial.npz, written by
tests/golden/make_golden_affine_partial.py).  They are regenerated from fixed seeds, so the golden file holds cv2's outputs
only.  TEST INFRASTRUCTURE."""
import os

import numpy as np

import affine_cases
from affine_cases import PARAMS, pack, real_sets  # noqa: F401  (the same parameter variants and real pairs)
from computervision_objectdetection_featurematching_b200 import synth

GOLDEN = os.path.join(affine_cases.GOLDEN_DIR, "golden_affine_partial.npz")


def similarity_correspondences(rng, n, inlier_ratio, noise=0.7, dup=0.0):
    """synth.correspondences with the inliers following a random similarity (rotation, uniform scale, translation)"""
    src, _, _ = synth.correspondences(rng, n, 1.0, dup=0.0)
    th = rng.uniform(-np.pi, np.pi); s = np.exp(rng.normal(0, .3))
    A = np.array([[s * np.cos(th), -s * np.sin(th), rng.normal(320, 60)],
                  [s * np.sin(th), s * np.cos(th), rng.normal(240, 60)]])
    dst = np.c_[src, np.ones(n)] @ A.T + rng.normal(0, noise, size=(n, 2))
    out = rng.random(n) > inlier_ratio
    dst[out] = rng.uniform([0, 0], [640, 480], size=(int(out.sum()), 2))
    dst = dst.astype(np.float32)
    if dup > 0:
        k = int(n * dup)
        ii = rng.integers(0, n, size=k); jj = rng.integers(0, n, size=k)
        src[ii] = src[jj]; dst[ii] = dst[jj]
    return src, dst


def synthetic_sets():
    """Similarity-plus-noise sets over n = 2..8192 and 5-90 % inliers, duplicate-heavy sets, n = 1 and 2 (a coincident
    pair among them), the collinear set and all-identical points."""
    rng = np.random.default_rng(5001)
    for n in (2, 3, 4, 5, 6, 8, 12, 20, 33, 47, 60, 90, 127, 200, 387, 1000, 2000, 8192):
        for rho in (0.05, 0.3, 0.9):
            yield similarity_correspondences(rng, n, rho)
    for _ in range(24):
        yield similarity_correspondences(rng, int(rng.integers(5, 120)), float(rng.uniform(0.2, 0.9)),
                                         dup=float(rng.uniform(0.2, 0.8)))
    tri = np.array([[0, 0], [10, 0], [0, 10]], np.float32)
    yield tri[:1], tri[:1] + 3                              # n = 1: cv2 returns None
    yield tri[:2], (tri[:2] * 1.5 + 3).astype(np.float32)   # n = 2: the closed form, which cv2 does not refine
    yield tri[[0, 0]], tri[[1, 2]]                          # n = 2 with coincident source points: M all NaN, found
    xs = np.linspace(0, 100, 12).astype(np.float32)         # every point on one line: found (estimateAffine2D: None)
    yield np.c_[xs, 2 * xs].astype(np.float32), np.c_[xs + 5, 2 * xs + 1].astype(np.float32)
    yield np.full((4, 2), 7, np.float32), np.full((4, 2), 9, np.float32)    # every model NaN: None
    yield np.full((12, 2), 7, np.float32), np.full((12, 2), 9, np.float32)


def same_bytes(a, b):
    """bit-equal, except that a NaN matches any NaN (its payload is not compared)"""
    a = np.asarray(a, np.float64).ravel(); b = np.asarray(b, np.float64).ravel()
    na, nb = np.isnan(a), np.isnan(b)
    return bool(np.array_equal(na, nb) and a[~na].tobytes() == b[~nb].tobytes())


def params_set():
    return similarity_correspondences(np.random.default_rng(5002), 150, 0.4)


def load_golden():
    """golden_affine_partial.npz with the point sets it was made from: tags syn / real (src, dst, offsets, M, M0, mask,
    found) and par (src, dst, params, M, M0, mask)."""
    Z = np.load(GOLDEN)
    g = {}
    for tag, sets in (("syn", synthetic_sets()), ("real", real_sets())):
        src, dst, off = pack(sets)
        assert np.array_equal(off, Z[f"{tag}_offsets"]), tag
        g[f"{tag}_src"], g[f"{tag}_dst"], g[f"{tag}_offsets"] = src, dst, off
        g[f"{tag}_mask"] = np.unpackbits(Z[f"{tag}_mask"], count=int(off[-1]))
        for k in ("M", "M0", "found"):
            g[f"{tag}_{k}"] = Z[f"{tag}_{k}"]
    g["par_src"], g["par_dst"] = params_set()
    g["par_params"] = np.array(PARAMS)
    g["par_mask"] = np.unpackbits(Z["par_mask"], axis=1, count=len(g["par_src"]))
    g["par_M"], g["par_M0"] = Z["par_M"], Z["par_M0"]
    return g
