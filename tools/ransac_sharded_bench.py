"""Hypothesis-range sharded RANSAC (cvg_find_homography_sharded) over N devices of one multi-device context.

Workloads (one point set of 8192 correspondences each):
  A  BASELINE config 5: 2^20 hypotheses on synth.correspondences(default_rng(5002), 8192, 0.3), CVG_RANSAC_NO_EARLY_STOP |
     CVG_RANSAC_NO_REFINE (bench.py's c5_ransac set).  One round.
  B  OpenCV semantics: max_iters = 2^20, confidence 0.9999999, default flags, 2 % inliers: the adaptive niters stays at the
     cap, so the serial loop really runs 2^20 iterations, in several rounds, followed by refit and LM.
Per N: 2 warm-up calls, then 10 calls timed with a host clock around the synchronous call (it ends in a device
synchronise); median and spread.  One extra call with timing on gives the first device's phase split: ransac_ms (whole
verify stage), hyp_ms (solve kernels), score_ms (score kernels), exchange_ms, and the rest (sampler + select + finish + the
wait for the slowest device outside the exchange).  host_outside_gpu0_ms = median call time - ransac_ms: uploads, draw
table checks, enqueue and result copies, i.e. what the first device's verify-stage events do not cover.

  python tools/ransac_sharded_bench.py --out DIR [--ns 1,2,4,8] [--logical]

--logical lists GPU 0 N times (logical devices: the shards share one GPU, the exchange is a device-to-device copy); those
lines measure the overheads of sharding (replicated sampler, exchange, enqueue), not a speed-up.  Writes
DIR/r04_ransac_sharded_n{N}[_logical].json, one JSON object per file, and prints each."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..")
sys.path.insert(0, ROOT)
from computervision_objectdetection_featurematching_b200 import api, synth  # noqa: E402

N_HYP = 1 << 20
WARMUP, REPS = 2, 10


def gpu_info():
    r = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    return [dict(zip(("index", "name", "power_limit", "clocks_max_sm"), [x.strip() for x in l.split(",")]))
            for l in r.stdout.strip().splitlines()]


def workloads():
    a_src, a_dst, _ = synth.correspondences(np.random.default_rng(5002), 8192, 0.3)
    b_src, b_dst, _ = synth.correspondences(np.random.default_rng(5003), 8192, 0.02)
    return {
        "A": dict(src=a_src, dst=a_dst, kw=dict(max_iters=N_HYP, flags=api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE)),
        "B": dict(src=b_src, dst=b_dst, kw=dict(max_iters=N_HYP, confidence=0.9999999)),
    }


def timed(fn):
    for _ in range(WARMUP):
        out = fn()
    ts = []
    for _ in range(REPS):
        t0 = time.perf_counter()
        out = fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return out, ts


def stats(ts):
    return {"median_ms": float(np.median(ts)), "min_ms": float(np.min(ts)), "max_ms": float(np.max(ts)),
            "spread_pct": float((np.max(ts) - np.min(ts)) / np.median(ts) * 100), "all_ms": [round(t, 3) for t in ts]}


def same_bytes(a, b):
    return all(np.asarray(a[k]).tobytes() == np.asarray(b[k]).tobytes() for k in ("H", "mask", "found", "iters", "ransac_mask"))


def run(n_dev, logical, W, base, info):
    devs = [0] * n_dev if logical else list(range(n_dev))
    line = {"devices": devs, "logical_devices": logical, "gpu": info, "workloads": {}}
    with api.Context(devs) as ctx:
        line["exchange_kind"] = ctx.exchange_kind
        for name, w in W.items():
            call = lambda: ctx.find_homography_sharded(w["src"], w["dst"], want_ransac_mask=True, **w["kw"])  # noqa: E731
            out, ts = timed(call)
            st = stats(ts)
            k, _ = ctx.last_exchange()
            ctx.set_timing(True)
            out_t = call()
            tm = ctx.last_timing()
            k_t, x_ms = ctx.last_exchange()
            ctx.set_timing(False)
            r = {"n": len(w["src"]), "params": {kk: int(v) if isinstance(v, int) else v for kk, v in w["kw"].items()},
                 "iters": out["iters"], "best_count": int(out["ransac_mask"].sum()), **st,
                 "hyps_per_s": out["iters"] / (st["median_ms"] * 1e-3),
                 "exchanges": k, "exchange_ms": x_ms,
                 "first_device": {"ransac_ms": tm["ransac_ms"], "hyp_ms": tm["hyp_ms"], "score_ms": tm["score_ms"],
                                  "exchange_ms": x_ms,
                                  "rest_ms": tm["ransac_ms"] - tm["hyp_ms"] - tm["score_ms"] - x_ms,
                                  "rounds_timed": tm["hyp_launches"]},
                 "host_outside_gpu0_ms": st["median_ms"] - tm["ransac_ms"],
                 "timed_call_same_bytes": same_bytes(out, out_t)}
            if base is not None and name in base:
                r["same_bytes_as_n1"] = same_bytes(out, base[name])
            else:
                base[name] = out
            if name == "A":
                from oracle import cvoracle as o
                err = o.compute_error(w["src"], w["dst"], out["H"])
                ref = o.ransac_stage(w["src"], w["dst"], max_iters=2000)
                r["parity_oracle"] = bool(np.array_equal((err <= np.float32(25.0)).astype(np.uint8), out["mask"])
                                          and out["mask"].sum() >= ref["mask"].sum())
                r["oracle_best_count_2000_iters"] = int(ref["mask"].sum())
            line["workloads"][name] = r
    if n_dev == 1 and not logical:
        # the same work through cvg_find_homography on a single-device context of the same GPU
        with api.Context(0) as c0:
            line["single_device_find_homography"] = {}
            for name, w in W.items():
                _, ts = timed(lambda: c0.find_homography(w["src"], w["dst"], **w["kw"]))
                line["single_device_find_homography"][name] = stats(ts)
    return line


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--ns", default="1,2,4,8")
    ap.add_argument("--logical", action="store_true")
    a = ap.parse_args()
    import torch
    visible = torch.cuda.device_count()
    if visible < 1:
        raise SystemExit("no CUDA device visible")
    info = gpu_info()
    os.makedirs(a.out, exist_ok=True)
    W = workloads()
    base = {}
    for n in [int(x) for x in a.ns.split(",")]:
        if not a.logical and n > visible:
            print(f"N={n}: only {visible} GPU(s) visible, skipped", flush=True)
            continue
        line = run(n, a.logical and n > 1, W, base, info)
        name = f"r04_ransac_sharded_n{n}{'_logical' if a.logical and n > 1 else ''}.json"
        with open(os.path.join(a.out, name), "w") as f:
            json.dump(line, f)
        print(json.dumps(line), flush=True)


if __name__ == "__main__":
    main()
