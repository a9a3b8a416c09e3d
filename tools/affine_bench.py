"""estimateAffine2D and estimateAffinePartial2D on the GPU: ms per batched call and hypotheses/s for
  A. 64 sets x n = 8192 at 2000 iterations without early stop, next to cvg_find_homography_batch on the same points;
  B. 445 sets of <= 127 real ratio-test correspondences (tests/affine_cases.py: the first test image of
     features_small.npz at its five scales),
     with OpenCV's defaults (adaptive stop);
then the device time of the affine kernels in one profiled call of each (torch.profiler, a run of its own).  The partial
method's keys carry "partial" in their names.
Prints one JSON line, with the GPU name and power limit, and writes it to --out if given.

    python tools/affine_bench.py [--reps 20] --out results/affine_bench.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import affine_cases  # noqa: E402
from computervision_objectdetection_featurematching_b200 import api, synth  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def timed(fn, reps):
    import torch
    fn()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(reps):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t) / reps * 1e3


def kernel_times(fn):
    import torch
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if "ransac" in ev.key:
            out[ev.key[:80]] = {"count": ev.count, "device_ms": round(ev.device_time_total / 1e3, 4)}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    torch.cuda.init()
    rng = np.random.default_rng(2026)
    sets = [synth.correspondences(rng, 8192, 0.3)[:2] for _ in range(64)]
    src = np.concatenate([s for s, _ in sets]); dst = np.concatenate([d for _, d in sets])
    off = np.arange(65, dtype=np.int64) * 8192
    rsrc, rdst, roff = affine_cases.pack(list(affine_cases.real_sets())[:445])
    res = {"gpu": gpu_info(), "reps": a.reps}
    with api.Context(0) as ctx:
        nes = api.RANSAC_NO_EARLY_STOP
        fa = lambda: ctx.estimate_affine2d_batch(src, dst, off, max_iters=2000, flags=nes)  # noqa: E731
        fh = lambda: ctx.find_homography_batch(src, dst, off, max_iters=2000, flags=nes)    # noqa: E731
        fr = lambda: ctx.estimate_affine2d_batch(rsrc, rdst, roff)                          # noqa: E731
        fpa = lambda: ctx.estimate_affine_partial2d_batch(src, dst, off, max_iters=2000, flags=nes)  # noqa: E731
        fpr = lambda: ctx.estimate_affine_partial2d_batch(rsrc, rdst, roff)                      # noqa: E731
        ms_a, ms_h, ms_r = timed(fa, a.reps), timed(fh, a.reps), timed(fr, a.reps)
        ms_pa, ms_pr = timed(fpa, a.reps), timed(fpr, a.reps)
        it_r = int(fr()["iters"].sum())
        it_pr = int(fpr()["iters"].sum())
        res["A_64x8192_2000it"] = {"affine_ms": round(ms_a, 3), "homography_ms": round(ms_h, 3),
                                   "affine_hyp_per_s": round(64 * 2000 / ms_a * 1e3),
                                   "homography_hyp_per_s": round(64 * 2000 / ms_h * 1e3)}
        res["B_445_real_sets"] = {"affine_ms": round(ms_r, 3), "max_n": int(np.diff(roff).max()),
                                  "iterations": it_r, "hyp_per_s": round(it_r / ms_r * 1e3)}
        res["A_64x8192_2000it_partial"] = {"partial_ms": round(ms_pa, 3), "partial_hyp_per_s": round(64 * 2000 / ms_pa * 1e3)}
        res["B_445_real_sets_partial"] = {"partial_ms": round(ms_pr, 3), "iterations": it_pr,
                                          "hyp_per_s": round(it_pr / ms_pr * 1e3)}
        res["kernels_A_affine"] = kernel_times(fa)
        res["kernels_A_homography"] = kernel_times(fh)
        res["kernels_B_affine"] = kernel_times(fr)
        res["kernels_A_partial"] = kernel_times(fpa)
        res["kernels_B_partial"] = kernel_times(fpr)
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
