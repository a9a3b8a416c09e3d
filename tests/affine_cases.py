"""The point sets of the estimateAffine2D goldens (tests/golden/golden_affine.npz, written by
tests/golden/make_golden_affine.py).  They are regenerated from fixed seeds, so the golden file holds cv2's outputs only.
TEST INFRASTRUCTURE."""
import os

import numpy as np

from computervision_objectdetection_featurematching_b200 import synth

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# (ransacReprojThreshold, maxIters, confidence, refineIters)
PARAMS = [(3.0, 2000, 0.99, 10), (3.0, 2000, 0.99, 0), (3.0, 2000, 0.99, 1), (3.0, 2000, 0.99, 5),
          (3.0, 2000, 0.99, 12), (1.0, 2000, 0.99, 10), (8.0, 2000, 0.99, 10), (3.0, 50, 0.99, 10),
          (3.0, 2000, 0.9, 10), (3.0, 2000, 0.999, 10), (3.0, 1, 0.99, 10), (2.0, 500, 0.995, 3)]
REJECTION_SIZES = (500, 2000, 4000, 6000, 9000, 15000)


def affine_correspondences(rng, n, inlier_ratio, noise=0.7, dup=0.0):
    """synth.correspondences with the inliers following a random affine map instead of a homography"""
    src, dst, _ = synth.correspondences(rng, n, 1.0, dup=0.0)
    A = np.array([[1 + rng.normal(0, .2), rng.normal(0, .2), rng.normal(0, 30)],
                  [rng.normal(0, .2), 1 + rng.normal(0, .2), rng.normal(0, 30)]])
    dst = np.c_[src, np.ones(n)] @ A.T + rng.normal(0, noise, size=(n, 2))
    out = rng.random(n) > inlier_ratio
    dst[out] = rng.uniform([0, 0], [640, 480], size=(int(out.sum()), 2))
    dst = dst.astype(np.float32)
    if dup > 0:
        k = int(n * dup)
        ii = rng.integers(0, n, size=k); jj = rng.integers(0, n, size=k)
        src[ii] = src[jj]; dst[ii] = dst[jj]
    return src, dst


def rejection_heavy(rng, n):
    """Every point but one on a line (exactly collinear in fp32): checkSubset rejects ~n/3 attempts per sample."""
    A = np.array([[0.9, 0.1, 12.0], [-0.05, 1.1, -7.0]])
    x = rng.integers(0, 20000, n).astype(np.float32)
    src = np.c_[x, 2 * x + 3].astype(np.float32)
    src[int(rng.integers(0, n))] = (300.0, 50.0)
    dst = (np.c_[src, np.ones(n)] @ A.T + rng.normal(0, 0.5, (n, 2))).astype(np.float32)
    return src, dst


def synthetic_sets():
    """Synthetic sets over n = 3..8192 and 5-90 % inliers, duplicate-heavy sets, n = 1, 2, 3, degenerate sets and the
    rejection-heavy sets, one of which exhausts getSubset's 10000 attempts."""
    rng = np.random.default_rng(4001)
    for n in (3, 4, 5, 6, 8, 12, 20, 33, 47, 60, 90, 127, 200, 387, 1000, 2000, 8192):
        for rho in (0.05, 0.3, 0.9):
            yield affine_correspondences(rng, n, rho)
    for _ in range(24):
        yield affine_correspondences(rng, int(rng.integers(5, 120)), float(rng.uniform(0.2, 0.9)),
                                     dup=float(rng.uniform(0.2, 0.8)))
    tri = np.array([[0, 0], [10, 0], [0, 10]], np.float32)
    yield tri[:1], tri[:1] + 3                              # n = 1, 2: cv2 returns None
    yield tri[:2], tri[:2] + 3
    yield tri, (tri * 1.5 + 2).astype(np.float32)           # n = 3: the closed form, which cv2 does not refine
    yield tri, np.array([[1, 2], [13, -1], [4, 9]], np.float32)
    xs = np.linspace(0, 100, 12).astype(np.float32)         # every point on one line: no subset passes
    yield np.c_[xs, 2 * xs].astype(np.float32), np.c_[xs + 5, 2 * xs + 1].astype(np.float32)
    yield np.full((12, 2), 7, np.float32), np.full((12, 2), 9, np.float32)
    yield tri[np.arange(12) % 3], tri[np.arange(12) % 3] + 3
    for n in REJECTION_SIZES:
        yield rejection_heavy(rng, n)


def params_set():
    return affine_correspondences(np.random.default_rng(4002), 150, 0.4)


def real_sets():
    """The ratio-test correspondences of the 890 (view, scene-scale) pairs of features_small.npz / golden_pairs.npz."""
    Z = np.load(os.path.join(GOLDEN_DIR, "features_small.npz"))
    G = np.load(os.path.join(GOLDEN_DIR, "golden_pairs.npz"))
    mk = Z["model_kpt"]; vo = Z["view_offsets"]; so = Z["scene_offsets"]
    for s in range(len(so) - 1):
        tk = Z["scene_kpt"][so[s]:so[s + 1]]
        idx = G["idx"][s].astype(np.int32); acc = G["accept"][s]
        for v in range(len(vo) - 1):
            sel = np.nonzero(acc[vo[v]:vo[v + 1]])[0] + vo[v]
            yield mk[sel].astype(np.float32), tk[idx[sel, 0]].astype(np.float32)


def pack(sets):
    """list of (src, dst) -> concatenated src, dst and offsets [P+1]"""
    sets = list(sets)
    off = np.cumsum([0] + [len(s) for s, _ in sets]).astype(np.int64)
    return (np.concatenate([s for s, _ in sets]).astype(np.float32), np.concatenate([d for _, d in sets]).astype(np.float32),
            off)


def load_golden():
    """golden_affine.npz with the point sets it was made from: tags syn / real (src, dst, offsets, M, M0, mask, found) and
    par (src, dst, params, M, M0, mask)."""
    Z = np.load(os.path.join(GOLDEN_DIR, "golden_affine.npz"))
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
