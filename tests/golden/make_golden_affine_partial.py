"""Write tests/golden/golden_affine_partial.npz: cv2.estimateAffinePartial2D(method=RANSAC) outputs (cv2 4.13.0) on the
point sets of tests/affine_partial_cases.py, which regenerates them from fixed seeds and from features_small.npz /
golden_pairs.npz.  Stored per set: found, M (refineIters as given), M0 (refineIters = 0: the RANSAC winner), and the
inlier masks as packed bits.

    python tests/golden/make_golden_affine_partial.py          (needs cv2)
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))

import affine_partial_cases as cases  # noqa: E402


def cv_partial(src, dst, thr=3.0, max_iters=2000, conf=0.99, refine=10):
    """-> found, M[6] (zeros when cv2 returns None), mask [n]"""
    if len(src) == 0:                                       # cv2 fails an assertion: nothing to record
        return False, np.zeros(6), np.zeros(0, np.uint8)
    M, inl = cv2.estimateAffinePartial2D(src, dst, method=cv2.RANSAC, ransacReprojThreshold=thr, maxIters=max_iters,
                                         confidence=conf, refineIters=refine)
    if M is None:
        return False, np.zeros(6), np.zeros(len(src), np.uint8)
    return True, M.ravel().copy(), inl.ravel().astype(np.uint8)


def main():
    out = {}
    for tag, sets in (("syn", cases.synthetic_sets()), ("real", cases.real_sets())):
        sets = list(sets)
        res = [cv_partial(s, d) for s, d in sets]
        out[f"{tag}_offsets"] = cases.pack(sets)[2]
        out[f"{tag}_found"] = np.array([r[0] for r in res])
        out[f"{tag}_M"] = np.stack([r[1] for r in res])
        out[f"{tag}_M0"] = np.stack([cv_partial(s, d, refine=0)[1] for s, d in sets])
        out[f"{tag}_mask"] = np.packbits(np.concatenate([r[2] for r in res]))
    src, dst = cases.params_set()
    Ms, M0s, masks = [], [], []
    for thr, it, conf, ref in cases.PARAMS:
        kw = dict(thr=thr, max_iters=int(it), conf=conf)
        f, M, m = cv_partial(src, dst, refine=int(ref), **kw)
        assert f
        Ms.append(M); masks.append(m); M0s.append(cv_partial(src, dst, refine=0, **kw)[1])
    out["par_M"] = np.stack(Ms); out["par_M0"] = np.stack(M0s); out["par_mask"] = np.packbits(np.stack(masks), axis=1)
    out["cv2_version"] = np.array(cv2.__version__)
    np.savez_compressed(cases.GOLDEN, **out)
    print(cases.GOLDEN)


if __name__ == "__main__":
    main()
