"""Write tests/golden/golden_crosscheck.npz: cv2.BFMatcher(NORM_L2, crossCheck=True).match outputs (cv2 4.13.0) on the sets
of tests/crosscheck_cases.py, which regenerates them from fixed seeds, features_small.npz and golden_sat.npz.  Stored per
group: offsets of the sets' query rows, and per query row the matched train index (-1 = none) and its distance (0 = none).

    python tests/golden/make_golden_crosscheck.py          (needs cv2)
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "..")))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))

import crosscheck_cases  # noqa: E402


def cv_cross_check(q, t):
    idx = np.full(len(q), -1, np.int32); dist = np.zeros(len(q), np.float32)
    for m in cv2.BFMatcher(cv2.NORM_L2, crossCheck=True).match(q, t):
        idx[m.queryIdx] = m.trainIdx; dist[m.queryIdx] = m.distance
    return idx, dist


def main():
    out = {}
    for tag, sets in crosscheck_cases.groups().items():
        res = [cv_cross_check(q, t) for q, t in sets]
        out[f"{tag}_offsets"] = np.cumsum([0] + [len(q) for q, _ in sets]).astype(np.int64)
        out[f"{tag}_idx"] = np.concatenate([r[0] for r in res])
        out[f"{tag}_dist"] = np.concatenate([r[1] for r in res])
    out["cv2_version"] = np.array(cv2.__version__)
    path = os.path.join(HERE, "golden_crosscheck.npz")
    np.savez_compressed(path, **out)
    print(path)


if __name__ == "__main__":
    main()
