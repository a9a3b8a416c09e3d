"""Generate the golden fixtures in this directory by running the reference's own arithmetic —
cv2 4.13.0 (opencv-python-headless 4.13.0.92) — in the build container.  The reference's hot path
(src/TestsDetector.cpp:59-84) is replayed call for call:

    BFMatcher(NORM_L2).knnMatch(view_desc, scene_desc, 2)   :59-60
    ratio test d0 < 0.9f*d1, gather points                   :62-72
    findHomography(obj, scene, RANSAC, 5.0, mask)            :77-78
    gates                                                    :74,79,81,84

Run:  python tests/golden/make_golden.py          (needs /root/reference/data and cv2)
Outputs (committed): features_small.npz, golden_pairs.npz, golden_synth.npz, golden_sat.npz
      python tests/golden/make_golden.py sat      (only golden_sat.npz; needs cv2 alone)
      python tests/golden/make_golden.py rect     (only golden_rect.npz; needs cv2 alone)
"""
import os
import sys

import cv2
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.abspath(os.path.join(HERE, "..", ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from computervision_objectdetection_featurematching_b200 import synth  # noqa: E402

RATIO = np.float32(0.9)


def cv_knn(q, t):
    nq = q.shape[0]
    idx = np.full((nq, 2), -1, np.int32)
    dist = np.zeros((nq, 2), np.float32)
    if nq == 0 or t.shape[0] == 0:
        return idx, dist
    m = cv2.BFMatcher(cv2.NORM_L2).knnMatch(q, t, 2)
    for i, row in enumerate(m):
        for k, dm in enumerate(row):
            idx[i, k] = dm.trainIdx
            dist[i, k] = dm.distance
    return idx, dist


def cv_accept(idx, dist):
    return ((idx[:, 1] >= 0) & (dist[:, 0] < RATIO * dist[:, 1])).astype(np.uint8)


def det3(H):
    m = H.ravel()
    return m[0] * (m[4] * m[8] - m[5] * m[7]) - m[1] * (m[3] * m[8] - m[5] * m[6]) + m[2] * (m[3] * m[7] - m[4] * m[6])


def cv_verify(src, dst, thr=5.0, max_iters=2000, conf=0.995):
    """-> status, H[9], mask.  status codes as in include/cvgraft.h."""
    n = len(src)
    if n < 4:
        return 1, np.zeros(9), np.zeros(n, np.uint8)
    H, mask = cv2.findHomography(src, dst, cv2.RANSAC, thr, maxIters=max_iters, confidence=conf)
    if H is None:
        return 2, np.zeros(9), np.zeros(n, np.uint8)
    mask = mask.ravel().astype(np.uint8)
    if int(np.count_nonzero(mask)) < 4:
        return 3, H.ravel(), mask
    d = abs(det3(H))
    if d < np.float32(0.1) or d > np.float32(10.0):
        return 4, H.ravel(), mask
    return 0, H.ravel(), mask


def make_features_small(full):
    """All 89 model views + 2 test images x 5 scales, cut from the full cache."""
    Z = np.load(full)
    so = Z["scene_offsets"]
    pick = [0, 25]   # one sugar-box scene, one power-drill scene
    sd, sk, off, names, folder = [], [], [0], [], []
    for s in pick:
        for k in range(5):
            a, b = so[5 * s + k], so[5 * s + k + 1]
            sd.append(Z["scene_desc"][a:b]); sk.append(Z["scene_kpt"][a:b]); off.append(off[-1] + b - a)
        names.append(str(Z["scene_names"][s])); folder.append(int(Z["scene_folder"][s]))
    out = os.path.join(HERE, "features_small.npz")
    np.savez_compressed(out, model_desc=Z["model_desc"], model_kpt=Z["model_kpt"],
                        view_offsets=Z["view_offsets"], view_model=Z["view_model"],
                        model_names=Z["model_names"], view_names=Z["view_names"],
                        scene_desc=np.concatenate(sd), scene_kpt=np.concatenate(sk),
                        scene_offsets=np.array(off, np.int32), scene_names=np.array(names),
                        scene_folder=np.array(folder, np.int32), scales=Z["scales"])
    return out


def make_golden_pairs(feat):
    Z = np.load(feat)
    md = Z["model_desc"].astype(np.float32); mk = Z["model_kpt"]; vo = Z["view_offsets"]
    so = Z["scene_offsets"]
    V = len(vo) - 1; S = len(so) - 1
    idx_all, dist_all, acc_all = [], [], []
    status = np.zeros((S, V), np.int8); ngood = np.zeros((S, V), np.int32); ninl = np.zeros((S, V), np.int32)
    Hs = np.zeros((S, V, 9)); masks = []; moff = [0]
    for s in range(S):
        t = Z["scene_desc"][so[s]:so[s + 1]].astype(np.float32); tk = Z["scene_kpt"][so[s]:so[s + 1]]
        # all views at once == per-view calls (rows are independent, SURVEY App. A.5)
        idx, dist = cv_knn(md, t)
        acc = cv_accept(idx, dist)
        idx_all.append(idx.astype(np.int16)); dist_all.append(dist); acc_all.append(acc)
        for v in range(V):
            a, b = vo[v], vo[v + 1]
            sel = np.nonzero(acc[a:b])[0] + a
            src = mk[sel]; dst = tk[idx[sel, 0]]
            st, H, mask = cv_verify(src, dst)
            status[s, v] = st; ngood[s, v] = len(sel); ninl[s, v] = int(mask.sum()); Hs[s, v] = H
            masks.append(mask); moff.append(moff[-1] + len(mask))
        print("scene-scale", s, "accepted pairs", int((status[s] == 0).sum()), flush=True)
    out = os.path.join(HERE, "golden_pairs.npz")
    np.savez_compressed(out, idx=np.stack(idx_all), dist=np.stack(dist_all), accept=np.stack(acc_all),
                        status=status, n_good=ngood, n_inliers=ninl, H=Hs,
                        mask=np.concatenate(masks), mask_offsets=np.array(moff, np.int64),
                        cv2_version=np.array(cv2.__version__))
    return out


def make_golden_sat():
    """Saturated u8-range rows: all distances above 2048 (distinct integer d^2 collide after sqrtf), planted pairs whose
    d^2 differ by 1 with the larger one at the lower index.  cv2 orders by the rounded distance, ties to the lower index."""
    rng = np.random.default_rng(7001)
    q, t = synth.saturated_pair(rng, 300, 2000)
    idx, dist = cv_knn(q, t)
    d2 = ((q[:, None, :].astype(np.float64) - t[None, idx[:, 0], :][0].astype(np.float64)) ** 2).sum(-1) if False else None
    path = os.path.join(HERE, "golden_sat.npz")
    np.savez_compressed(path, q=q.astype(np.uint8), t=t.astype(np.uint8), idx=idx, dist=dist, accept=cv_accept(idx, dist))
    # how many rows does the rounded-distance order decide differently from the d^2 order?
    D2 = (q.astype(np.float64) ** 2).sum(1)[:, None] + (t.astype(np.float64) ** 2).sum(1)[None, :] - 2.0 * q.astype(np.float64) @ t.astype(np.float64).T
    order = np.lexsort((np.broadcast_to(np.arange(t.shape[0]), D2.shape), D2), axis=1)[:, :2]
    print("golden_sat: rows where cv2 differs from the d^2 order:", int((order != idx).any(axis=1).sum()), "of", len(q),
          "min distance", float(dist.min()))
    return path


def make_golden_synth():
    out = {}
    # --- kNN: float descriptors (summation-order sensitive), ties, tiny train sets
    rng = np.random.default_rng(3001)
    q = synth.float_desc(rng, 257, 128); t = synth.float_desc(rng, 1003, 128)
    out["knn_float_q"], out["knn_float_t"] = q, t
    out["knn_float_idx"], out["knn_float_dist"] = cv_knn(q, t)
    q, t, _ = synth.planted_pair(np.random.default_rng(3002), 300, 700)
    t[5] = t[400]; t[17] = t[18]                      # exact duplicate train rows -> distance ties
    q[3] = t[17]; q[4] = t[400]                       # zero distances with ties
    out["knn_int_q"], out["knn_int_t"] = q, t
    out["knn_int_idx"], out["knn_int_dist"] = cv_knn(q, t)
    out["knn_nt1_idx"], out["knn_nt1_dist"] = cv_knn(q[:9], t[:1])
    out["knn_nt2_idx"], out["knn_nt2_dist"] = cv_knn(q[:9], t[:2])
    # --- findHomography: synthetic sets, with / without duplicates, small n, n == 4, degenerate
    cases = []
    rng = np.random.default_rng(3003)
    specs = [(int(rng.integers(5, 300)), float(rng.uniform(0.15, 0.9)), 0.0) for _ in range(40)]
    specs += [(int(rng.integers(5, 90)), float(rng.uniform(0.2, 0.9)), float(rng.uniform(0.2, 0.8))) for _ in range(40)]
    specs += [(4, 1.0, 0.0), (4, 1.0, 0.0), (5, 1.0, 0.0), (6, 0.5, 0.0), (2000, 0.3, 0.0), (8192, 0.3, 0.0)]
    for n, rho, dup in specs:
        src, dst, _ = synth.correspondences(rng, n, rho, dup=dup)
        cases.append((src, dst))
    # degenerate: all points collinear; all identical; only 3 distinct points
    n = 12
    xs = np.linspace(0, 100, n).astype(np.float32)
    cases.append((np.c_[xs, 2 * xs].astype(np.float32), np.c_[xs + 5, 2 * xs + 1].astype(np.float32)))
    cases.append((np.full((n, 2), 7, np.float32), np.full((n, 2), 9, np.float32)))
    tri = np.array([[0, 0], [10, 0], [0, 10]], np.float32)
    cases.append((tri[np.arange(n) % 3], tri[np.arange(n) % 3] + 3))
    srcs, dsts, offs, Hs, masks, founds = [], [], [0], [], [], []
    for src, dst in cases:
        H, mask = cv2.findHomography(src, dst, cv2.RANSAC, 5.0)
        srcs.append(src); dsts.append(dst); offs.append(offs[-1] + len(src))
        founds.append(H is not None)
        Hs.append(np.zeros(9) if H is None else H.ravel())
        masks.append(np.zeros(len(src), np.uint8) if mask is None else mask.ravel().astype(np.uint8))
    out["fh_src"] = np.concatenate(srcs); out["fh_dst"] = np.concatenate(dsts)
    out["fh_offsets"] = np.array(offs, np.int64); out["fh_H"] = np.stack(Hs)
    out["fh_mask"] = np.concatenate(masks); out["fh_found"] = np.array(founds)
    # --- other maxIters / confidence / threshold settings
    rng = np.random.default_rng(3004)
    src, dst, _ = synth.correspondences(rng, 150, 0.4)
    out["fhp_src"], out["fhp_dst"] = src, dst
    params = [(3.0, 2000, 0.995), (5.0, 50, 0.995), (5.0, 2000, 0.9), (1.0, 500, 0.99), (10.0, 1, 0.995)]
    out["fhp_params"] = np.array(params)
    hh, mm = [], []
    for thr, it, conf in params:
        H, mask = cv2.findHomography(src, dst, cv2.RANSAC, thr, maxIters=int(it), confidence=conf)
        hh.append(np.zeros(9) if H is None else H.ravel()); mm.append(mask.ravel().astype(np.uint8))
    out["fhp_H"] = np.stack(hh); out["fhp_mask"] = np.stack(mm)
    # --- building blocks: eigen / solve / invert (DECOMP_EIG), DLT (n==4 bypasses RANSAC and LM)
    rng = np.random.default_rng(3005)
    mats, evals, evecs, rhs, sol, inv = [], [], [], [], [], []
    for k in range(24):
        n = 9 if k % 2 else 8
        B = rng.normal(size=(n, n)); A = B @ B.T
        if k % 3 == 0:
            A[:, -1] = A[:, 0]; A[-1, :] = A[0, :]
        _, w, v = cv2.eigen(A)
        b = rng.normal(size=(n, 1))
        _, x = cv2.solve(A, b, flags=cv2.DECOMP_EIG)
        _, Ai = cv2.invert(A, flags=cv2.DECOMP_EIG)
        pad = lambda M: np.pad(M, ((0, 9 - M.shape[0]), (0, 9 - M.shape[1])))
        mats.append(pad(A)); evals.append(np.pad(w.ravel(), (0, 9 - n))); evecs.append(pad(v))
        rhs.append(np.pad(b.ravel(), (0, 9 - n))); sol.append(np.pad(x.ravel(), (0, 9 - n))); inv.append(pad(Ai))
    out["eig_A"] = np.stack(mats); out["eig_w"] = np.stack(evals); out["eig_v"] = np.stack(evecs)
    out["eig_b"] = np.stack(rhs); out["eig_x"] = np.stack(sol); out["eig_inv"] = np.stack(inv)
    out["eig_n"] = np.array([9 if k % 2 else 8 for k in range(24)])
    d_src, d_dst, d_H = [], [], []
    for _ in range(50):
        s4 = rng.uniform(0, 640, size=(4, 2)).astype(np.float32)
        d4 = (s4 + rng.normal(0, 20, size=(4, 2))).astype(np.float32)
        H, _ = cv2.findHomography(s4, d4, 0)
        if H is not None:
            d_src.append(s4); d_dst.append(d4); d_H.append(H.ravel())
    out["dlt_src"] = np.stack(d_src); out["dlt_dst"] = np.stack(d_dst); out["dlt_H"] = np.stack(d_H)
    # --- LM solver observed iterate by iterate through estimateAffine2D(refineIters=k)
    a_src, a_dst, a_H = [], [], []
    for _ in range(6):
        n = 24
        s = rng.uniform(0, 600, size=(n, 2)).astype(np.float32)
        At = np.array([[1 + rng.normal(0, .2), rng.normal(0, .2), rng.normal(0, 30)],
                       [rng.normal(0, .2), 1 + rng.normal(0, .2), rng.normal(0, 30)]])
        d = (np.c_[s, np.ones(n)] @ At.T + rng.normal(0, 2.0, size=(n, 2))).astype(np.float32)
        its = []
        for k in range(0, 13):
            Hk, inl = cv2.estimateAffine2D(s, d, method=cv2.RANSAC, ransacReprojThreshold=1000.0, refineIters=k)
            assert inl.all()
            its.append(Hk.ravel())
        a_src.append(s); a_dst.append(d); a_H.append(np.stack(its))
    out["lm_aff_src"] = np.stack(a_src); out["lm_aff_dst"] = np.stack(a_dst); out["lm_aff_H"] = np.stack(a_H)
    # --- DLT + LM isolated (method 0) on well-conditioned sets
    l_src, l_dst, l_H = [], [], []
    for _ in range(20):
        s, d, _ = synth.correspondences(rng, 20, 1.0)
        H, _ = cv2.findHomography(s, d, 0)
        l_src.append(s); l_dst.append(d); l_H.append(H.ravel())
    out["lm_h_src"] = np.stack(l_src); out["lm_h_dst"] = np.stack(l_dst); out["lm_h_H"] = np.stack(l_H)
    out["cv2_version"] = np.array(cv2.__version__)
    path = os.path.join(HERE, "golden_synth.npz")
    np.savez_compressed(path, **out)
    return path


def rect_cases():
    """Point sets of the cv::boundingRect cases (tests/test_host_consumer.py): 500 sets, some of them on integer coordinates."""
    rng = np.random.default_rng(0)
    for _ in range(500):
        p = rng.uniform(-50, 700, size=(int(rng.integers(1, 40)), 2)).astype(np.float32)
        if rng.random() < 0.3:
            p = np.round(p)
        yield p


def make_golden_rect():
    path = os.path.join(HERE, "golden_rect.npz")
    np.savez_compressed(path, rect=np.array([cv2.boundingRect(p) for p in rect_cases()], np.int32),
                        cv2_version=np.array(cv2.__version__))
    return path


if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "rect":
    print(make_golden_rect())
    sys.exit(0)

if __name__ == "__main__" and len(sys.argv) > 1 and sys.argv[1] == "sat":
    print(make_golden_sat())
    sys.exit(0)

if __name__ == "__main__":
    full = os.path.join(ROOT, "data_cache", "features_full.npz")
    if not os.path.exists(full):
        import build_feature_cache
        os.makedirs(os.path.dirname(full), exist_ok=True)
        build_feature_cache.build("/root/reference/data", full)
    print(make_features_small(full))
    print(make_golden_synth())
    print(make_golden_pairs(os.path.join(HERE, "features_small.npz")))
