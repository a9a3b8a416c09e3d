"""The fused detect path with each geometric check (cvg_detect_params.method): findHomography, estimateAffine2D and
estimateAffinePartial2D on the same inputs.

  value workload: bench.py's (one model view of 8192 SIFT-like rows against 64 resident scenes of 8192 rows per call,
      50 % planted matches, 30 % of them following a homography), timed
        pipelined: three calls in flight on one context (cvg_detect_scenes_submit / cvg_job_wait, three lanes);
        serial:    one lane, synchronous calls back to back;
      pairs/s, launches per call, mean inliers of the pairs with a model and accepted pairs per call, per method;
  real: the 890 (view, scaled scene) pairs of tests/golden/features_small.npz, one detect_scenes_inliers call: pairs/s
      and the status histogram [accept, lt4 matches, H empty, lt4 inliers, det reject].

The methods take turns inside every repetition, so that drift of the shared machine hits all three alike; the median
over repetitions is reported.  Homography runs with the reference's parameters (5.0, 2000, 0.995), the affine methods with
OpenCV's affine defaults (3.0, 2000, 0.99, refineIters 10).  Prints one JSON line with the GPU name and power limit read
in the same call, and writes it to --out if given.

    python tools/detect_verify_bench.py [--steps 20] [--reps 5] --out results/detect_verify_bench.json
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


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def params_of(name):
    if name == "homography":
        return api.detect_params()
    m = api.VERIFY_AFFINE if name == "affine" else api.VERIFY_AFFINE_PARTIAL
    return api.detect_params(ransac=api.ransac_params(3.0, 2000, 0.99), method=m, refine_iters=10)


def summary(res):
    r = res.ravel()
    has = r["H"][:, 8] != 0
    return {"mean_inliers": round(float(r["n_inliers"][has].mean()), 2) if has.any() else 0.0,
            "accepted": int((r["status"] == api.ACCEPT).sum()), "pairs": int(r.size),
            "status_hist": np.bincount(r["status"], minlength=5).tolist()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20, help="calls per timed window")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=5, help="timed windows per method and mode (methods alternate)")
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--batches", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("detect_verify_bench.py needs a CUDA device: libcvgraft has no CPU fallback")
    out = {"gpu": gpu_info(), "steps": a.steps, "reps": a.reps, "pairs_per_call": a.pairs,
           "workload": "bench.py value: 1 model view x 8192 vs %d scenes x 8192 (SIFT-like), ratio 0.9" % a.pairs,
           "params": {"homography": [5.0, 2000, 0.995], "affine": [3.0, 2000, 0.99, 10], "partial": [3.0, 2000, 0.99, 10]}}
    q, qk, batches = bench.make_workload(3000, a.pairs, a.batches)
    Z = np.load(os.path.join(ROOT, "tests", "golden", "features_small.npz"))
    so = Z["scene_offsets"]
    scales = np.tile(Z["scales"], (len(so) - 1) // len(Z["scales"])).astype(np.float32)
    with api.Context(0) as ctx:
        models = ctx.upload_models(q, qk, [0, bench.NQ], [0])
        resident = [ctx.upload_scenes(d, k, o) for d, k, o in batches]
        rmodels = ctx.upload_models(Z["model_desc"].astype(np.float32), Z["model_kpt"], Z["view_offsets"], Z["view_model"])
        rscenes = ctx.upload_scenes(Z["scene_desc"].astype(np.float32), Z["scene_kpt"], so)
        P = {m: params_of(m) for m in METHODS}

        def pipelined(p, steps):
            jobs = []
            for k in range(steps):
                jobs.append(ctx.submit_scenes(models, resident[k % len(resident)], params=p, want_inliers=False))
                if len(jobs) > 2:
                    jobs.pop(0).wait()
            for j in jobs:
                j.wait()

        def serial(p, steps):
            for k in range(steps):
                ctx.detect_scenes(models, resident[k % len(resident)], params=p)

        def real(p, steps):
            for _ in range(steps):
                ctx.detect_scenes_inliers(rmodels, rscenes, scales=scales, params=p)

        def timed(fn, p, steps):
            fn(p, a.warmup)
            torch.cuda.synchronize()
            l0 = ctx.launch_count
            t = time.perf_counter()
            fn(p, steps)                                    # every call / wait returns with its results on the host
            ms = (time.perf_counter() - t) * 1e3
            return ms, (ctx.launch_count - l0) / steps

        modes = {"pipelined_3_in_flight": (pipelined, 3, a.pairs), "serial": (serial, 1, a.pairs), "real_890": (real, 0, 890)}
        for mode, (fn, lanes, per_call) in modes.items():
            ctx.set_lanes(lanes)
            rates = {m: [] for m in METHODS}; launches = {}
            for _ in range(a.reps):
                for m in METHODS:
                    ms, launches[m] = timed(fn, P[m], a.steps)
                    rates[m].append(per_call * a.steps / (ms * 1e-3))
            out[mode] = {m: {"pairs_per_s": round(statistics.median(rates[m])), "runs": [round(x) for x in rates[m]],
                             "launches_per_call": launches[m]} for m in METHODS}
        ctx.set_lanes(0)
        for m in METHODS:
            out["pipelined_3_in_flight"][m].update(summary(ctx.detect_scenes(models, resident[0], params=P[m])))
            out["real_890"][m].update(summary(ctx.detect_scenes(rmodels, rscenes, scales=scales, params=P[m])))
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
