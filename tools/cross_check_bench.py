"""BFMatcher(NORM_L2, crossCheck=True).match against knnMatch(k=2) on the same inputs: the match kernel's device time per
call (CUDA events around the match kernels, cvg_last_timing's match_ms; median over --reps calls after a warm-up call) for
  A. a SIFT-like 8192 x 8192 pair (synth.planted_pair), tensor-core path;
  B. all 89 views of features_small.npz (one cross-check call with view = -1, each view its own query matrix; one knn2
     call on all views) against each of its 10 scaled scenes, tensor-core path, summed over the scenes;
  C. float descriptors 8192 x 8192 (synth.float_desc): cross-check on the exact SIMT kernel (path 2), knn2 on the
     candidate path (3).
Prints one JSON line, with the GPU name and power limit read in the same run, and writes it to --out if given.

    python tools/cross_check_bench.py [--reps 10] --out results/cross_check_bench.json
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
sys.path.insert(0, ROOT)

from computervision_objectdetection_featurematching_b200 import api, synth  # noqa: E402


def gpu_info():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"unavailable: {e}"


def match_ms(ctx, fn, reps):
    """median match_ms of reps calls after one warm-up call, and the path that served them"""
    fn()
    out = []
    for _ in range(reps):
        fn()
        m = C.c_float()
        ctx.lib.cvg_last_timing(ctx.handle, C.byref(m), None, None)
        out.append(m.value)
    return float(np.median(out)), ctx.last_match_path


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    res = {"gpu": gpu_info(), "reps": a.reps}
    rng = np.random.default_rng(8801)
    with api.Context(0) as ctx:
        ctx.lib.cvg_set_timing(ctx.handle, 1)
        q, t, _ = synth.planted_pair(rng, 8192, 8192)
        xc, px = match_ms(ctx, lambda: ctx.match_cross_check(q, t), a.reps)
        kn, pk = match_ms(ctx, lambda: ctx.match_knn2(q, t), a.reps)
        res["A_sift_8192x8192"] = {"cross_check_ms": round(xc, 4), "knn2_ms": round(kn, 4), "paths": [px, pk]}

        Z = np.load(os.path.join(ROOT, "tests", "golden", "features_small.npz"))
        vo = Z["view_offsets"]; so = Z["scene_offsets"]
        m = ctx.upload_models(Z["model_desc"].astype(np.float32), Z["model_kpt"], vo)
        xs = ks = 0.0
        paths = set()
        for s in range(len(so) - 1):
            ts = Z["scene_desc"][so[s]:so[s + 1]].astype(np.float32)
            x, p1 = match_ms(ctx, lambda: ctx.match_cross_check(m, ts, view=-1), a.reps)
            k, p2 = match_ms(ctx, lambda: ctx.match_knn2(m, ts), a.reps)
            xs += x; ks += k; paths |= {p1, p2}
        m.free()
        res["B_89_views_x_10_scenes"] = {"cross_check_ms": round(xs, 4), "knn2_ms": round(ks, 4), "query_rows": int(vo[-1]),
                                         "scene_rows": int(so[-1]), "paths": sorted(paths)}

        qf, tf = synth.float_desc(rng, 8192), synth.float_desc(rng, 8192)
        xc, px = match_ms(ctx, lambda: ctx.match_cross_check(qf, tf), max(1, a.reps // 5))
        kn, pk = match_ms(ctx, lambda: ctx.match_knn2(qf, tf), a.reps)
        res["C_float_8192x8192"] = {"cross_check_ms": round(xc, 4), "knn2_ms": round(kn, 4), "paths": [px, pk]}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
