"""ctypes binding of tests/affine_partial_oracle.c, the CPU restatement of cv2.estimateAffinePartial2D(method=RANSAC)
that the partial-affine tests compare the GPU with.  TEST INFRASTRUCTURE.  It is compiled on first use into a temporary
directory (the tree may be read-only) and resolves the pinned pieces it builds on — cv::RNG, RANSACUpdateNumIters,
solve / invert(DECOMP_EIG) — from the CPU oracle's libcvoracle.so."""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

from affine_oracle import RansacInfo, _p

HERE = os.path.dirname(os.path.abspath(__file__))

_lib = None


def lib():
    global _lib
    if _lib is None:
        from oracle import cvoracle
        C.CDLL(cvoracle.build(), mode=C.RTLD_GLOBAL)       # the symbols affine_partial_oracle.c calls
        out = os.path.join(tempfile.mkdtemp(prefix="affine_partial_oracle_"), "libaffine_partial_oracle.so")
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c11", "-ffp-contract=off", "-fno-fast-math", "-shared",
                               "-o", out, os.path.join(HERE, "affine_partial_oracle.c"), "-lm"])
        _lib = C.CDLL(out)
    return _lib


def estimate_affine_partial2d(src, dst, thr=3.0, max_iters=2000, conf=0.99, refine_iters=10):
    """cv2.estimateAffinePartial2D(src, dst, method=RANSAC, ransacReprojThreshold=thr, maxIters=, confidence=,
    refineIters=) -> dict(found, M [2,3] (zeros when cv2 returns None), mask [n] (the RANSAC-stage mask), M_ransac [2,3],
    info), as affine_oracle.estimate_affine2d."""
    src = np.ascontiguousarray(src, np.float32).reshape(-1, 2); dst = np.ascontiguousarray(dst, np.float32).reshape(-1, 2)
    n = src.shape[0]
    M = np.zeros(6); M0 = np.zeros(6); mask = np.zeros(max(n, 1), np.uint8); info = RansacInfo()
    rc = lib().affp_estimate(_p(src, C.c_float), _p(dst, C.c_float), n, C.c_double(thr), C.c_double(conf), int(max_iters),
                             int(refine_iters), _p(M, C.c_double), _p(mask, C.c_uint8), _p(M0, C.c_double), C.byref(info))
    if rc < 0:
        raise ValueError("estimateAffinePartial2D needs at least one correspondence")
    return {"found": bool(rc), "M": M.reshape(2, 3), "mask": mask[:n], "M_ransac": M0.reshape(2, 3),
            "info": {k: getattr(info, k) for k, _ in info._fields_}}
