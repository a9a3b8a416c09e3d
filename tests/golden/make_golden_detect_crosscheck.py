"""Write tests/golden/golden_detect_crosscheck.npz: cv2 4.13.0's record of the fused detect path with cross-check matching on
the 890 real (view, scaled scene) pairs of features_small.npz, scene-major (the order of crosscheck_cases.real_pairs).  Per
pair: the correspondences of BFMatcher(NORM_L2, crossCheck=True).match in query-row order (model keypoint of queryIdx,
scene keypoint of trainIdx), then for each geometric check

    homography  cv2.findHomography(src, dst, cv2.RANSAC, 5.0)                       (maxIters 2000, confidence 0.995)
    affine      cv2.estimateAffine2D(src, dst, RANSAC, 3.0, 2000, 0.99, refineIters 10)
    partial     cv2.estimateAffinePartial2D(src, dst, RANSAC, 3.0, 2000, 0.99, refineIters 10)

whether a model came back, the model (H 3x3, or M 2x3), cv2.determinant of it (M promoted to 3x3) and the returned mask
(bit-packed over the concatenated correspondences).  The script first checks that cv2's matches are golden_crosscheck.npz's
real_idx, so the two goldens describe the same correspondences.

    python tests/golden/make_golden_detect_crosscheck.py          (needs cv2)
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))

import crosscheck_cases  # noqa: E402

METHODS = ("homography", "affine", "partial")


def correspondences():
    """-> query index per pair (cv2's order), src [k,2], dst [k,2], offsets [P+1]"""
    Z = np.load(os.path.join(HERE, "features_small.npz"))
    mk = Z["model_kpt"].astype(np.float32); sk = Z["scene_kpt"].astype(np.float32)
    vo = Z["view_offsets"]; so = Z["scene_offsets"]
    V = len(vo) - 1
    qidx, src, dst, offs = [], [], [], [0]
    for p, (q, t) in enumerate(crosscheck_cases.real_pairs()):
        s, v = divmod(p, V)
        ms = cv2.BFMatcher(cv2.NORM_L2, crossCheck=True).match(q, t)
        qi = np.array([m.queryIdx for m in ms], np.int64); ti = np.array([m.trainIdx for m in ms], np.int64)
        assert np.all(np.diff(qi) > 0), p                            # query-row order, as the fused path compacts
        qidx.append(qi)
        src.append(mk[vo[v]:vo[v + 1]][qi].reshape(-1, 2)); dst.append(sk[so[s]:so[s + 1]][ti].reshape(-1, 2))
        offs.append(offs[-1] + len(qi))
    return qidx, src, dst, np.asarray(offs, np.int64)


def run(name, s, d):
    if name == "homography":
        if len(s) < 4:                                               # the reference's :74 gate: never called
            return None, np.zeros(len(s), np.uint8)
        H, mask = cv2.findHomography(s, d, cv2.RANSAC, 5.0)
    else:
        fn = cv2.estimateAffine2D if name == "affine" else cv2.estimateAffinePartial2D
        H, mask = fn(s, d, method=cv2.RANSAC, ransacReprojThreshold=3.0, maxIters=2000, confidence=0.99, refineIters=10)
    mask = np.zeros(len(s), np.uint8) if mask is None else mask.ravel().astype(np.uint8)
    return H, mask


def main():
    G = np.load(os.path.join(HERE, "golden_crosscheck.npz"))
    qidx, src, dst, offs = correspondences()
    # the same matches as golden_crosscheck.npz's real group
    ro = G["real_offsets"]; ri = G["real_idx"]
    for p, qi in enumerate(qidx):
        assert np.array_equal(np.nonzero(ri[ro[p]:ro[p + 1]] >= 0)[0], qi), p
    out = {"offsets": offs, "cv2_version": np.array(cv2.__version__)}
    lo, hi = float(np.float32(0.1)), float(np.float32(10.0))
    for name in METHODS:
        P = len(src); w = 9 if name == "homography" else 6
        found = np.zeros(P, bool); model = np.zeros((P, w)); det = np.zeros(P); masks = []
        status = np.zeros(P, np.int32)
        for k in range(P):
            H, mask = run(name, src[k], dst[k])
            masks.append(mask)
            n = len(src[k])
            if H is not None and H.size:
                found[k] = True; model[k] = H.ravel()
                H3 = H if name == "homography" else np.vstack([H, [0.0, 0.0, 1.0]])
                det[k] = cv2.determinant(H3)
            cnt = int(mask.sum()) if found[k] else 0
            status[k] = 1 if n < 4 else (2 if not found[k] else (3 if cnt < 4 else (4 if not lo <= abs(det[k]) <= hi else 0)))
        out[f"{name}_found"] = found; out[f"{name}_model"] = model; out[f"{name}_det"] = det
        out[f"{name}_mask"] = np.packbits(np.concatenate(masks).astype(bool))
        print(name, "status histogram", np.bincount(status, minlength=5).tolist())
    path = os.path.join(HERE, "golden_detect_crosscheck.npz")
    np.savez_compressed(path, **out)
    print(path, "pairs", len(src), "median correspondences", int(np.median(np.diff(offs))))


if __name__ == "__main__":
    main()
