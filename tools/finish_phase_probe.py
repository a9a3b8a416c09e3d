#!/usr/bin/env python
"""Where the refit/LM kernel (`ransac_finish_kernel`) spends its time on bench.py's workload (64 pairs of 8192 x 8192,
2000-iteration RANSAC, the first batch of `make_workload(3000, ...)`), one lane, kernels alone on the GPU.

  --phases   builds a -DFIN_PROF variant of libcvgraft.so in a temporary directory and prints, per phase of the kernel,
             the SM cycles thread 0 of a set's CTA saw between phase ends (compaction, DLT sums, DLT LtL, each eigen-solve
             with its rotation count and cycles per rotation, each lm_eval, the final mask), summed over the sets
  --kernels  torch.profiler over `--steps` serial calls of the build being imported: mean device time per launch of every
             kernel of the verify stage
  --root DIR imports the package from another tree (A/B against an older build)

Writes one JSON object to stdout (and to --out if given).  Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

HERE = os.path.dirname(os.path.abspath(__file__))
PHASES = ["total", "compact", "dlt_sums", "dlt_ltl", "refit_eig", "eval_J", "lm_solve", "eval_xd", "lm_update",
          "lm_proceed", "mask"]


def build_probe(root, tmp):
    env = dict(os.environ, CVG_NVCC_EXTRA="-DFIN_PROF", CVGRAFT_SO=os.path.join(tmp, "libcvgraft_finprof.so"),
               CVGRAFT_OBJ_DIR=os.path.join(tmp, "obj"))
    subprocess.run([sys.executable, os.path.join(root, "computervision_objectdetection_featurematching_b200", "build.py")],
                   check=True, env=env, stdout=subprocess.DEVNULL)
    return env["CVGRAFT_SO"]


def setup(root, pairs):
    sys.path.insert(0, root)
    import bench
    from computervision_objectdetection_featurematching_b200 import api
    q, qk, batches = bench.make_workload(3000, pairs, 1)
    ctx = api.Context(0)
    models = ctx.upload_models(q, qk, [0, bench.NQ], [0])
    scenes = ctx.upload_scenes(*batches[0])
    ctx.set_lanes(1)
    params = api.detect_params()
    return ctx, lambda: ctx.detect_scenes(models, scenes, params=params)


def sm_clock_mhz():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return out
    except Exception as e:           # the probe's numbers stand without it
        return f"unavailable: {e}"


def run_phases(root, pairs, steps):
    import ctypes as C
    import numpy as np
    with tempfile.TemporaryDirectory() as tmp:
        os.environ["CVGRAFT_SO"] = build_probe(root, tmp)
        ctx, call = setup(root, pairs)
        lib = C.CDLL(os.environ["CVGRAFT_SO"])
        lib.cvg_finish_profile.restype = C.c_int
        lib.cvg_finish_profile.argtypes = [C.c_void_p, C.c_void_p, C.c_int]
        call()
        n_ev = 96
        log = np.zeros((pairs, n_ev, 2), np.int64); cnt = np.zeros(pairs, np.int32)
        lib.cvg_finish_profile(log.ctypes.data, cnt.ctypes.data, pairs)
        per_phase = {p: {"cycles": 0, "count": 0, "rotations": 0} for p in PHASES[1:]}
        sets = []
        for _ in range(steps):
            call()
            assert lib.cvg_finish_profile(log.ctypes.data, cnt.ctypes.data, pairs) == n_ev
            for s in range(pairs):
                if cnt[s] == 0:
                    continue
                ev = []
                for e in range(1, cnt[s]):
                    ph, rot, cyc = int(log[s, e, 0] & 255), int(log[s, e, 0] >> 8), int(log[s, e, 1])
                    d = per_phase[PHASES[ph]]
                    d["cycles"] += cyc; d["count"] += 1; d["rotations"] += rot
                    ev.append([PHASES[ph], cyc, rot])
                sets.append({"n_inl": int(log[s, 0, 0] >> 8), "ns": int(log[s, 0, 1]),
                             "cycles": sum(c for _, c, _ in ev), "events": ev})
        ctx.close()
    n = len(sets)
    tot = sum(s["cycles"] for s in sets)
    table = {}
    for p, d in per_phase.items():
        if d["count"]:
            table[p] = {"cycles_per_set": d["cycles"] / n, "share": d["cycles"] / tot, "per_set": d["count"] / n,
                        "cycles_per_call": d["cycles"] / d["count"]}
            if d["rotations"]:
                table[p]["rotations_per_call"] = d["rotations"] / d["count"]
                table[p]["cycles_per_rotation"] = d["cycles"] / d["rotations"]
    return {"sets": n, "cycles_per_set": tot / n, "us_per_set_globaltimer": sum(s["ns"] for s in sets) / n / 1e3,
            "n_inl_range": [min(s["n_inl"] for s in sets), max(s["n_inl"] for s in sets)],
            "phases": table, "set0_events": sets[0]["events"]}


def run_kernels(root, pairs, steps):
    import torch
    from torch.profiler import ProfilerActivity, profile
    ctx, call = setup(root, pairs)
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            call()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        if e.device_type.name == "CUDA" and ("ransac" in e.key or "match" in e.key):
            name = e.key.split("(")[0].replace("void cvg::", "").replace("cvg::", "")
            t = getattr(e, "device_time_total", None) or e.cuda_time_total
            out[name] = {"launches_per_step": e.count / steps, "us_per_launch": t / e.count}
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--phases", action="store_true")
    ap.add_argument("--kernels", action="store_true")
    ap.add_argument("--root", default=os.path.dirname(HERE))
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--out")
    a = ap.parse_args()
    root = os.path.abspath(a.root)
    res = {"root": root, "pairs": a.pairs, "steps": a.steps, "gpu": sm_clock_mhz()}
    if a.phases:
        res["phases"] = run_phases(root, a.pairs, a.steps)
    if a.kernels:
        res["kernels"] = run_kernels(root, a.pairs, a.steps)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
