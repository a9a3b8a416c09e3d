"""The fused detect path with its two correspondence sources, knnMatch(k = 2) + ratio test and BFMatcher(NORM_L2,
crossCheck = true).match (detect_params(cross_check=True)), for each geometric check (findHomography, estimateAffine2D,
estimateAffinePartial2D).

  value workload: bench.py's (one model view of 8192 SIFT-like rows against 64 resident scenes of 8192 rows per call,
      50 % planted matches, 30 % of them following a homography), three calls in flight on one context
      (cvg_detect_scenes_submit / cvg_job_wait): pairs/s;
  real: the 890 (view, scaled scene) pairs of tests/golden/features_small.npz, one detect_scenes_inliers call: pairs/s;
  match_ms: cvg_last_timing's match kernel time of one synchronous call on the context's own engine (median over --reps),
      for both workloads; plus, per mode, the status histogram [accept, lt4 matches, H empty, lt4 inliers, det reject]
      and the mean good-match count.

The six (source, method) combinations take turns inside every repetition, so that drift of the shared machine hits all
alike; the median over repetitions is reported.  Homography runs with the reference's parameters (5.0, 2000, 0.995), the
affine methods with OpenCV's affine defaults (3.0, 2000, 0.99, refineIters 10).  Prints one JSON line with the GPU name
and power limit read in the same call, and writes it to --out if given.

    python tools/detect_cross_check_bench.py [--steps 20] [--reps 5] --out results/detect_cross_check_bench.json
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

import bench  # noqa: E402  (its workload generator)
from computervision_objectdetection_featurematching_b200 import api  # noqa: E402

METHODS = ("homography", "affine", "partial")
SOURCES = ("ratio", "cross_check")


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def params_of(method, source):
    xc = source == "cross_check"
    if method == "homography":
        return api.detect_params(cross_check=xc)
    m = api.VERIFY_AFFINE if method == "affine" else api.VERIFY_AFFINE_PARTIAL
    return api.detect_params(ransac=api.ransac_params(3.0, 2000, 0.99), method=m, refine_iters=10, cross_check=xc)


def summary(res):
    r = res.ravel()
    return {"status_hist": np.bincount(r["status"], minlength=5).tolist(), "mean_good": round(float(r["n_good"].mean()), 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="calls per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5, help="timed windows per combination and workload (combinations alternate)")
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("detect_cross_check_bench.py needs a CUDA device: libcvgraft has no CPU fallback")
    out = {"gpu": gpu_info(), "steps": a.steps, "reps": a.reps, "pairs_per_call": a.pairs,
           "workload": "bench.py value: 1 model view x 8192 vs %d scenes x 8192 (SIFT-like), 3 calls in flight" % a.pairs,
           "params": {"homography": [5.0, 2000, 0.995], "affine": [3.0, 2000, 0.99, 10], "partial": [3.0, 2000, 0.99, 10]}}
    q, qk, batches = bench.make_workload(3000, a.pairs, a.batches)
    Z = np.load(os.path.join(ROOT, "tests", "golden", "features_small.npz"))
    so = Z["scene_offsets"]
    scales = np.tile(Z["scales"], (len(so) - 1) // len(Z["scales"])).astype(np.float32)
    combos = [(m, s) for m in METHODS for s in SOURCES]
    with api.Context(0) as ctx:
        models = ctx.upload_models(q, qk, [0, bench.NQ], [0])
        resident = [ctx.upload_scenes(d, k, o) for d, k, o in batches]
        rmodels = ctx.upload_models(Z["model_desc"].astype(np.float32), Z["model_kpt"], Z["view_offsets"], Z["view_model"])
        rscenes = ctx.upload_scenes(Z["scene_desc"].astype(np.float32), Z["scene_kpt"], so)
        P = {c: params_of(*c) for c in combos}

        def pipelined(p, steps):
            jobs = []
            for k in range(steps):
                jobs.append(ctx.submit_scenes(models, resident[k % len(resident)], params=p, want_inliers=False))
                if len(jobs) > 2:
                    jobs.pop(0).wait()
            for j in jobs:
                j.wait()

        def real(p, steps):
            for _ in range(steps):
                ctx.detect_scenes_inliers(rmodels, rscenes, scales=scales, params=p)

        def timed(fn, p, steps):
            fn(p, a.warmup)
            torch.cuda.synchronize()
            t = time.perf_counter()
            fn(p, steps)                                    # every call / wait returns with its results on the host
            return (time.perf_counter() - t) * 1e3

        key = lambda c: f"{c[0]}_{c[1]}"                    # noqa: E731
        for mode, (fn, per_call) in {"pipelined_3_in_flight": (pipelined, a.pairs), "real_890": (real, 890)}.items():
            ctx.set_lanes(0)
            rates = {c: [] for c in combos}
            for _ in range(a.reps):
                for c in combos:
                    rates[c].append(per_call * a.steps / (timed(fn, P[c], a.steps) * 1e-3))
            out[mode] = {key(c): {"pairs_per_s": round(statistics.median(rates[c])), "runs": [round(x) for x in rates[c]]}
                         for c in combos}
        # match kernel time of one synchronous call on the context's own engine
        ctx.set_lanes(1)
        ctx.set_timing(True)
        for mode, (m, sc, kw) in {"pipelined_3_in_flight": (models, resident[0], {}),
                                  "real_890": (rmodels, rscenes, {"scales": scales})}.items():
            ms = {c: [] for c in combos}; path = {}
            for _ in range(a.reps + 1):
                for c in combos:
                    ctx.detect_scenes(m, sc, params=P[c], **kw)
                    ms[c].append(ctx.last_timing()["match_ms"]); path[c] = ctx.last_match_path
            for c in combos:
                out[mode][key(c)].update({"match_ms": round(statistics.median(ms[c][1:]), 4), "match_path": path[c]},
                                         **summary(ctx.detect_scenes(m, sc, params=P[c], **kw)))
        ctx.set_timing(False)
        ctx.set_lanes(0)
        for s in resident:
            s.free()
        rscenes.free(); rmodels.free(); models.free()
    line = json.dumps(out)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
