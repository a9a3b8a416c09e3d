#!/usr/bin/env python
"""bench.py — image-pairs/s of the matching-and-verification hot path (BF-L2 kNN k=2 + ratio test +
RANSAC homography), BASELINE.json metric, on synthetic descriptors of the named shape.

Workload at every N ("c3"): per GPU and per step, ONE resident model view of 8192 SIFT-like 128-D
descriptors is matched against B scene descriptor sets of 8192 rows each and each of the B pairs is
verified with a 2000-iteration RANSAC homography — BASELINE config 3 (8k x 8k + 2000-iter RANSAC), batched
the way the reference batches it (one model view vs. many test images, src/TestsDetector.cpp:58).

ONE context per GPU, driven by ONE host thread, in every number below.

  value : pairs/s with the scene sets already resident in HBM, whole job over N GPUs; the thread keeps `--depth` calls in
          flight (cvg_detect_scenes_submit / cvg_job_wait), so that one call's latency-bound refit/LM kernel runs under the
          next calls' match and hypothesis kernels.  value_single_context = synchronous calls back to back (each split over
          the context's lanes); value_serial = one lane, every kernel alone on the GPU (timed region of the rooflines)
  e2e   : pairs/s through the public host-buffer API: every step uploads its B scene sets from pinned host memory
          (cvg_scenes_upload_async), runs the fused call and reads back the per-pair results AND the inlier scene points
  roofline : the tcgen05 match kernel, the largest kernel of the step that has a roofline (2*Nq*Nt*128 flop per pair
             against the measured burst cuBLAS bf16 rate); roofline_score: the inlier-counting kernel against the fp32 issue
             rate (its SURVEY-8d HBM figure is kept as algorithmic_gbs); solve_stage: the 4-point DLT kernel (fp64 Jacobi,
             latency-bound) — all from CUDA events around the kernels inside the serial timed steps
  cpu_baseline : cv2 4.13.0 (the reference's own arithmetic) on this host's cores, bounded sample
  c4, c5_match, c5_ransac (N >= 2 only, outside the timed regions above): BASELINE config 4 (4096 pairs of 4096 x 4096, pair
             p -> GPU p mod N), config 5's match (262 144 queries x 131 072 train rows per GPU, train-tile sharded, ONE NCCL
             all-gather + top-2 merge) and config 5's 2^20-hypothesis RANSAC, each with an inline check against the CPU oracle

`--impl reference` times the reference's CPU implementation (cv2 BFMatcher.knnMatch + findHomography, all
host threads; the C oracle port if cv2 is unavailable) on the same workload, metric and unit.

Launch: python bench.py --gpus N --steps K --warmup W      (N > 1: under torchrun, one rank per GPU)
"""
import argparse
import atexit
import json
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

# a context runs 1 + lanes compute streams and two copy streams: more hardware queues than the default 8, so that none of them
# alias (set before CUDA is initialised; libcvgraft does the same in cvg_create for hosts that do not)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from computervision_objectdetection_featurematching_b200 import synth  # noqa: E402

# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner to stdout when the
# box sets NCCL_DEBUG), so file descriptor 1 is pointed at stderr for everything but the result line.
_RESULT_OUT = sys.stdout                 # main() swaps the descriptors; importing this module (tools/) does not

METRIC = "image-pairs/s (BF-L2 kNN + RANSAC H)"
UNIT = "pairs/s"
NQ = NT = 8192
DIM = 128


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return {"bf16_burst": p.get("bf16_tflops", 1590.0), "bf16_sustained": p.get("bf16_tflops_sustained", 1400.0),
                "hbm": p.get("hbm_gbs", 6650.0), "source": "measured"}
    return {"bf16_burst": 1590.0, "bf16_sustained": 1400.0, "hbm": 6650.0, "source": "fallback"}


def make_workload(seed, n_scenes, n_batches, desc="sift"):
    """One model view + n_batches batches of n_scenes scene sets (planted matches, 30% geometric inliers).
    desc = "sift": integer-valued fp32 rows as cv2 SIFT emits them; "float": non-integer rows (SURVEY 8d 'float'
    generator), which take the candidate + fp32 re-rank match path."""
    rng = np.random.default_rng(seed)
    gen = synth.sift_like if desc == "sift" else synth.float_desc
    q = gen(rng, NQ)
    qk = rng.uniform([0, 0], [640, 480], size=(NQ, 2)).astype(np.float32)
    batches = []
    for _ in range(n_batches):
        descs, kpts = [], []
        for _ in range(n_scenes):
            t = gen(rng, NT)
            tk = rng.uniform([0, 0], [640, 480], size=(NT, 2)).astype(np.float32)
            k = NQ // 2                                           # 50% planted matches
            rq = rng.permutation(NQ)[:k]; rt = rng.permutation(NT)[:k]
            if desc == "sift":
                t[rt] = np.clip(q[rq] + np.round(rng.normal(0, 12.0, size=(k, DIM))).astype(np.float32), 0, 255)
            else:
                t[rt] = q[rq] + rng.normal(0, 6.0, size=(k, DIM)).astype(np.float32)
            H = synth.random_homography(rng)
            geo = rng.random(k) < 0.3                             # 30% of the planted matches follow H
            p = np.c_[qk[rq[geo]], np.ones(int(geo.sum()))] @ H.T
            tk[rt[geo]] = (p[:, :2] / p[:, 2:3] + rng.normal(0, 0.7, size=(int(geo.sum()), 2))).astype(np.float32)
            descs.append(t); kpts.append(tk)
        batches.append((np.concatenate(descs), np.concatenate(kpts), np.arange(n_scenes + 1, dtype=np.int64) * NT))
    return q, qk, batches


class ClockSampler:
    """nvidia-smi clocks / throttle reasons (B200_PROFILING.md recipe).  Started at process start so that the tool is
    already looping when the short timed regions run; samples are kept by timestamp for the windows marked."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu):
        self.gpu = gpu; self.proc = None; self.path = None; self.windows = []

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv"); os.close(fd)
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "10"],
                                         stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
            atexit.register(lambda p=self.proc: p.poll() is None and p.kill())     # a run that fails leaves no sampler behind
        except Exception:
            self.proc = None

    def mark(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        import datetime
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.proc:
            return out
        time.sleep(0.05)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, sm_all = [], [], set(), []
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 10:
                    continue
                try:
                    ts = datetime.datetime.strptime(f[0], "%Y/%m/%d %H:%M:%S.%f").timestamp()
                    v = float(f[2]); m = float(f[3])
                except ValueError:
                    continue
                sm_all.append(v); mx.append(m)
                if any(a - 0.02 <= ts <= b + 0.02 for a, b in self.windows):
                    sm.append(v)
                    for name, r in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                        if r.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if not sm and sm_all:                                   # windows shorter than the sampling period: busy samples of the run
            sm = [v for v in sm_all if v >= 0.5 * max(sm_all)]
        if sm:
            out = {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}
        return out


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, res, inlier_xy, inlier_offsets):
    """--dump-outputs: what a caller received from the last timed step, as <name>.npy in float64 (float32 for the points).
    The per-pair fields come from the headline loop (resident scenes, calls in flight); the inlier scene points and their
    per-pair offsets from the e2e loop, whose last step ran the same scene batch.  Above DUMP_LIMIT bytes in all, the points
    are replaced by a fixed sample of their rows (seed 0), whose indices are written as inlier_xy_rows."""
    arrays = {name: np.ascontiguousarray(res[name], np.float64) for name in res.dtype.names}
    arrays["inlier_offsets"] = inlier_offsets.astype(np.float64)
    arrays["inlier_xy"] = np.ascontiguousarray(inlier_xy, np.float32)
    budget = DUMP_LIMIT - 4096 - sum(a.nbytes for k, a in arrays.items() if k != "inlier_xy")     # 4096: the .npy headers
    n = len(inlier_xy)
    if arrays["inlier_xy"].nbytes > budget:
        keep = budget // (8 + 8)                                 # a sampled row costs its point and its float64 index
        rows = np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
        arrays["inlier_xy"] = arrays["inlier_xy"][rows]
        arrays["inlier_xy_rows"] = rows.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def bind_to_gpu_numa_node(props):
    """Run this rank's host threads (and first-touch its pinned buffers) on the NUMA node the GPU hangs off, when the
    box exposes one: with 8 ranks streaming 50 GB/s each the host memory is the end-to-end limit."""
    try:
        bus = f"{props.pci_domain_id:04x}:{props.pci_bus_id:02x}:{props.pci_device_id:02x}.0"
        with open(f"/sys/bus/pci/devices/{bus}/numa_node") as f:
            node = int(f.read().strip())
        if node < 0:
            return None
        with open(f"/sys/devices/system/node/node{node}/cpulist") as f:
            cpus = set()
            for part in f.read().strip().split(","):
                a, _, b = part.partition("-")
                cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return node
    except Exception:
        pass
    return None


def cpu_pairs(q, qk, batch, n_pairs, threads, first=0):
    """The reference's CPU path on pairs [first, first + n_pairs) of a batch; returns (seconds, kind).
    All host threads are used: knnMatch is parallel inside OpenCV (parallel_for_ over query rows), findHomography
    is serial inside, so the verify calls of the sample run side by side in a thread pool (cv2 releases the GIL)."""
    desc, kpt, off = batch
    try:
        import cv2
        from concurrent.futures import ThreadPoolExecutor
        cv2.setNumThreads(threads)
        bf = cv2.BFMatcher(cv2.NORM_L2)
        t0 = time.perf_counter()
        sets = []
        for s in range(first, first + n_pairs):
            t = desc[off[s]:off[s + 1]]; tk = kpt[off[s]:off[s + 1]]
            m = bf.knnMatch(q, t, 2)                                               # src/TestsDetector.cpp:60
            good = [(a.queryIdx, a.trainIdx) for a, b in m if a.distance < np.float32(0.9) * b.distance]   # :67
            if len(good) >= 4:                                                      # :74
                gi = np.asarray(good)
                sets.append((qk[gi[:, 0]], tk[gi[:, 1]]))
        with ThreadPoolExecutor(max_workers=max(1, min(threads, len(sets) or 1))) as ex:
            list(ex.map(lambda sd: cv2.findHomography(sd[0], sd[1], cv2.RANSAC, 5.0), sets))          # :78
        return time.perf_counter() - t0, "reference"
    except ImportError:
        from oracle import cvoracle as o
        t0 = time.perf_counter()
        for s in range(first, first + n_pairs):
            t = desc[off[s]:off[s + 1]]; tk = kpt[off[s]:off[s + 1]]
            idx, dist = o.knn2(q, t, nthreads=threads)
            acc = o.ratio(idx, dist).astype(bool)
            if acc.sum() >= 4:
                o.find_homography(qk[acc], tk[idx[acc, 0]])
        return time.perf_counter() - t0, "port"


WORKLOAD = ("c3: 1 resident model view x 8192 desc vs scenes of 8192 desc (128-D, SIFT-like), ratio 0.9, "
            "RANSAC 2000 iters thr 5.0 conf 0.995")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    pairs_per_step = max(2, min(threads, 32))            # enough pairs per step to keep every thread busy in the verify stage
    q, qk, batches = make_workload(3000, pairs_per_step, 1, args.desc)
    for _ in range(args.warmup):
        cpu_pairs(q, qk, batches[0], 2, threads)
    total = 0.0; kind = "reference"
    for _ in range(args.steps):
        dt, kind = cpu_pairs(q, qk, batches[0], pairs_per_step, threads)
        total += dt
    value = pairs_per_step * args.steps / total
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": WORKLOAD, "pairs_per_step": pairs_per_step},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind,
                             "sample": f"{pairs_per_step} pairs per step, knnMatch on {threads} threads, findHomography calls of the step on a {threads}-thread pool"},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), file=_RESULT_OUT, flush=True)


# ---- BASELINE config 5 (match): train-tile sharded kNN with ONE exchange step over NCCL, inline parity ------------------
def run_c5_match(ctx, dev, rank, world, dist, all_max, barrier):
    """262 144 queries x (131 072 x world) train rows: every rank holds one train tile (the tile size of SURVEY 8d; the full
    1 048 576-row set at 8 GPUs) and the replicated queries; local top-2 (cvg_dev_match_top2), all-gather of 16 B per query and
    rank over NCCL, merge (cvg_dev_merge_top2).  Rank 0 regenerates every tile and checks 512 sampled queries against the
    CPU oracle over the WHOLE train set (reference src/TestsDetector.cpp:59-72)."""
    import torch
    from computervision_objectdetection_featurematching_b200 import sharding
    NQ, TILE = 262144, 131072
    NT = TILE * world
    q = synth.sift_like(np.random.default_rng(5000), NQ)           # replicated queries (same seed everywhere)

    def make_tile(r):
        rng = np.random.default_rng(5001 + r)
        t = synth.sift_like(rng, TILE)
        k = NQ // 16                                               # planted noisy copies of some queries in every tile
        rq = rng.permutation(NQ)[:k]; rt = rng.permutation(TILE)[:k]
        t[rt] = np.clip(q[rq] + np.round(rng.normal(0, 12.0, size=(k, 128))).astype(np.float32), 0, 255)
        return t

    t_mine = make_tile(rank)
    qd = torch.from_numpy(q).to(dev); td = torch.from_numpy(t_mine).to(dev)
    base = rank * TILE
    stream = torch.cuda.current_stream(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    d_loc = torch.empty((NQ, 2), dtype=torch.float32, device=dev); i_loc = torch.empty((NQ, 2), dtype=torch.int32, device=dev)
    d_all = torch.empty((world, NQ, 2), dtype=torch.float32, device=dev); i_all = torch.empty((world, NQ, 2), dtype=torch.int32, device=dev)
    idx = torch.empty((NQ, 2), dtype=torch.int32, device=dev); dd = torch.empty((NQ, 2), dtype=torch.float32, device=dev)
    acc = torch.empty((NQ,), dtype=torch.uint8, device=dev)

    def once():
        ev[0].record(stream)
        ctx.dev_match_top2(qd.data_ptr(), NQ, td.data_ptr(), TILE, base, d_loc.data_ptr(), i_loc.data_ptr(), stream=stream.cuda_stream)
        ev[1].record(stream)
        if world > 1:
            dist.all_gather_into_tensor(d_all, d_loc)               # the one exchange step of the path
            dist.all_gather_into_tensor(i_all, i_loc)
        else:
            d_all[0].copy_(d_loc); i_all[0].copy_(i_loc)
        ev[2].record(stream)
        ctx.dev_merge_top2(d_all.data_ptr(), i_all.data_ptr(), world, NQ, 0.9, idx.data_ptr(), dd.data_ptr(), acc.data_ptr(),
                           stream=stream.cuda_stream)
        ev[3].record(stream)
        ev[3].synchronize()
        return ev[0].elapsed_time(ev[3]), ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3])

    for _ in range(3):
        once()
    barrier()
    reps = [once() for _ in range(5)]
    ms = all_max(min(r[0] for r in reps))
    best = min(reps, key=lambda r: r[0])
    out = {"nq": NQ, "nt": NT, "tile_rows_per_gpu": TILE, "ms": ms, "match_pflops": 2.0 * NQ * NT * 128 / (ms * 1e-3) / 1e15,
           "local_match_ms": all_max(best[1]), "all_gather_us": 1e3 * all_max(best[2]), "merge_us": 1e3 * all_max(best[3]),
           "all_gather_share": best[2] / best[0],
           "bytes_gathered_per_gpu": int(16 * NQ * world), "accepted": int(acc.sum().item()),
           "note": "weak form of BASELINE config 5: 131 072 train rows per GPU (the full 262 144 x 1 048 576 at 8 GPUs); timed region = "
                   "operand prep + local top-2 + NCCL all-gather + merge, best of 5 after 3 warm-ups, max over ranks"}
    if rank == 0:
        from oracle import cvoracle as o
        t0 = time.time()
        t_all = np.concatenate([t_mine] + [make_tile(r) for r in range(1, world)])
        rows = np.random.default_rng(5999).permutation(NQ)[:512]
        oi, od = o.knn2(q[rows], t_all, nthreads=os.cpu_count())
        gi = idx.cpu().numpy()[rows]; gd = dd.cpu().numpy()[rows]; ga = acc.cpu().numpy()[rows]
        out["checked_queries"] = 512
        out["parity"] = bool(np.array_equal(gi, oi) and np.array_equal(gd, od) and np.array_equal(ga, o.ratio(oi, od)))
        out["oracle_s"] = time.time() - t0
    del qd, td, d_all, i_all
    torch.cuda.empty_cache()
    return out


# ---- BASELINE config 5 (verify): 2^20 RANSAC hypotheses on 8192 correspondences at 30 % inliers, every GPU a replica -------
def run_c5_ransac(ctx, api, dev, rank, world, all_max, barrier):
    """All 2^20 hypotheses are sampled (cv::RNG replay), solved and scored (CVG_RANSAC_NO_EARLY_STOP: a throughput mode outside
    OpenCV's maxIters semantics, SURVEY 8d), the first best one wins, no refit.  Checked on rank 0: the winner's mask is what the
    CPU oracle's computeError gives for the returned H, bit for bit, and it holds at least as many inliers as the oracle's own
    2000-iteration RANSAC stage finds on the same set."""
    import torch
    n_hyp = 1 << 20
    src, dst, _ = synth.correspondences(np.random.default_rng(5002), 8192, 0.3)
    flags = api.RANSAC_NO_EARLY_STOP | api.RANSAC_NO_REFINE
    ctx.set_lanes(1)
    H, mask = ctx.find_homography(src, dst, max_iters=n_hyp, flags=flags)               # warm-up: RNG table, scratch
    barrier()
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    H, mask = ctx.find_homography(src, dst, max_iters=n_hyp, flags=flags)
    e1.record(stream); e1.synchronize()
    ms = all_max(e0.elapsed_time(e1))
    serial_sets = ctx.last_sampler_serial_sets
    ctx.set_lanes(3)
    out = {"hypotheses_per_gpu": n_hyp, "n": 8192, "ms_incl_h2d_d2h": ms, "hyps_per_s_per_gpu": n_hyp / (ms * 1e-3),
           "hyps_per_s": world * n_hyp / (ms * 1e-3), "algorithmic_gbs_per_gpu": 16.0 * 8192 * n_hyp / (ms * 1e-3) / 1e9,
           "hbm_bound_hyps_per_s_per_gpu": load_peaks()["hbm"] * 1e9 / (16.0 * 8192), "best_count": int(mask.sum()),
           "sets_handed_to_the_serial_sampler": serial_sets,
           "note": "every GPU runs the same set (replicas: a single RANSAC set does not shard without an exchange of counts); "
                   "sampler + solve + score + select of 2^20 hypotheses, host copies of the 64 KB set and of H / mask included"}
    if rank == 0:
        from oracle import cvoracle as o
        err = o.compute_error(src, dst, H)
        ref = o.ransac_stage(src, dst, max_iters=2000)
        out["parity"] = bool(np.array_equal((err <= np.float32(25.0)).astype(np.uint8), mask) and mask.sum() >= ref["mask"].sum())
        out["oracle_best_count_2000_iters"] = int(ref["mask"].sum())
    return out


# ---- BASELINE config 4: 4096 pairs of 4096 x 4096, pair p -> GPU p mod N, no data-path collective ------------------------
def run_c4(ctx, api, dev, rank, world, all_max, barrier):
    import torch
    N4, B, POOL = 4096, 64, 2
    n_pairs = 4096
    rngq = np.random.default_rng(4000)
    q = synth.sift_like(rngq, N4); qk = rngq.uniform([0, 0], [640, 480], size=(N4, 2)).astype(np.float32)
    models = ctx.upload_models(q, qk, [0, N4], [0])

    def make_pair(p):
        """Scene p: planted copies of half the view's descriptors, 30 % of them on a homography."""
        rng = np.random.default_rng(4001 + p)
        t = synth.sift_like(rng, N4); tk = rng.uniform([0, 0], [640, 480], size=(N4, 2)).astype(np.float32)
        k = N4 // 2
        rq = rng.permutation(N4)[:k]; rt = rng.permutation(N4)[:k]
        t[rt] = np.clip(q[rq] + np.round(rng.normal(0, 12.0, size=(k, 128))).astype(np.float32), 0, 255)
        H = synth.random_homography(rng)
        geo = rng.random(k) < 0.3
        pp = np.c_[qk[rq[geo]], np.ones(int(geo.sum()))] @ H.T
        tk[rt[geo]] = (pp[:, :2] / pp[:, 2:3] + rng.normal(0, 0.7, size=(int(geo.sum()), 2))).astype(np.float32)
        return t, tk

    mine = list(range(rank, n_pairs, world))                      # pair p -> GPU p mod N (SURVEY 8d)
    pool = []
    for b in range(POOL):                                         # POOL x B distinct scenes per rank, cycled over its pairs
        ps = mine[b * B:(b + 1) * B]
        ts, ks = zip(*[make_pair(p) for p in ps])
        pool.append(ctx.upload_scenes(np.concatenate(ts), np.concatenate(ks), np.arange(B + 1, dtype=np.int64) * N4))
    steps = len(mine) // B
    first = ctx.detect_scenes_inliers(models, pool[0])[0].copy()
    barrier()
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    jobs = []; accepted = 0
    for s in range(steps):                                         # one host thread, three calls in flight
        jobs.append(ctx.submit_scenes(models, pool[s % POOL]))
        if len(jobs) == 3:
            accepted += int((jobs.pop(0).wait()[0]["status"] == 0).sum())
    for j in jobs:
        accepted += int((j.wait()[0]["status"] == 0).sum())
    e1.record(stream); e1.synchronize()
    ms = all_max(e0.elapsed_time(e1))
    out = {"pairs": steps * B * world, "nq": N4, "nt": N4, "ms": ms, "pairs_per_s": steps * B * world / (ms * 1e-3),
           "match_tflops_equiv": 2.0 * N4 * N4 * 128 * steps * B * world / (ms * 1e-3) / 1e12, "accepted_rank0": accepted,
           "note": f"pair p -> GPU p mod N; every rank cycles {POOL * B} distinct resident scenes over its {steps * B} pairs; "
                   "kNN + ratio + 2000-iteration RANSAC + refit per pair, inlier points returned; no data-path collective"}
    if rank == 0:
        from oracle import cvoracle as o
        ok = True
        for j in range(2):
            t, tk = make_pair(mine[j])
            oi, od = o.knn2(q, t, nthreads=os.cpu_count()); oa = o.ratio(oi, od).astype(bool)
            ref = o.find_homography(qk[oa], tk[oi[oa, 0]])
            r = first[j, 0]
            ok = ok and int(r["n_good"]) == int(oa.sum()) and (int(r["status"]) != api.H_EMPTY) == ref["found"] \
                and int(r["ransac_iters"]) == ref["info"]["iters_run"] \
                and (not ref["found"] or abs(int(r["n_inliers"]) - int(ref["mask"].sum())) <= 2)
        out["parity"] = bool(ok)
        out["parity_note"] = "first 2 pairs of rank 0 against the CPU oracle: matches kept, H found, RANSAC iterations, inlier count (<= 2 flips above 128 inliers)"
    for sc in pool:
        sc.free()
    models.free()
    return out


def run_cvgraft(args):
    import torch
    import torch.distributed as dist
    from computervision_objectdetection_featurematching_b200 import api

    world = int(os.environ.get("WORLD_SIZE", "1")); rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: libcvgraft has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    all_cpus = os.sched_getaffinity(0)
    numa = bind_to_gpu_numa_node(torch.cuda.get_device_properties(local))
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    B, R, DEPTH = args.pairs, args.batches, max(1, args.depth)
    clocks = ClockSampler(local); clocks.start()
    q, qk, batches = make_workload(3000 + rank, B, R, args.desc)
    ctx = api.Context(local)                             # ONE context, driven by this one host thread
    LANES = min(8, max(3, DEPTH))                        # one lane per call in flight (3 by default; more pay off on one GPU
                                                         # with cores to spare: 6 -> +7 %, 8 -> +12 %, but cost 20 % at 8 GPUs x 4 vCPUs)
    models = ctx.upload_models(q, qk, [0, NQ], [0])
    params = api.detect_params()
    stream = torch.cuda.ExternalStream(ctx.stream, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def all_max(ms):
        if world > 1:
            t = torch.tensor([ms], device="cuda", dtype=torch.float64)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms

    def timed(loop, steps):
        """K steps bracketed by barrier + synchronize; device time between two CUDA events on the context's stream: the
        first is recorded on the idle GPU before the first call, the second after the last call's results are on the host
        (every call / job wait returns only when its GPU work is complete, whichever internal stream ran it)."""
        barrier()
        e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        loop(steps)
        e1.record(stream)
        e1.synchronize()
        ms = e0.elapsed_time(e1)
        barrier()
        return all_max(ms)

    resident = [ctx.upload_scenes(d, k, o) for d, k, o in batches]

    # ---- phase 1: strictly serial (one lane), kernels alone — the timed region the rooflines are computed from ----------
    ctx.set_lanes(1); ctx.set_timing(True)
    match_ms, ransac_ms, hyp_ms, hyp_launches, scored, score_ms = [], [], [], [], [], []

    def loop_serial(steps, record=True):
        for k in range(steps):
            ctx.detect_scenes(models, resident[k % R], params=params)
            if record:
                t = ctx.last_timing()
                match_ms.append(t["match_ms"]); ransac_ms.append(t["ransac_ms"]); hyp_ms.append(t["hyp_ms"])
                hyp_launches.append(t["hyp_launches"]); scored.append(t["scored_points"]); score_ms.append(t["score_ms"])

    loop_serial(args.warmup, record=False)
    ms_serial = timed(loop_serial, args.steps)
    ctx.set_timing(False)

    # ---- phase 2: synchronous calls, each split over the context's lanes (what a caller of the blocking API gets) -------
    ctx.set_lanes(LANES)

    def loop_sync(steps):
        for k in range(steps):
            ctx.detect_scenes(models, resident[k % R], params=params)

    loop_sync(args.warmup)
    ms_sync = timed(loop_sync, args.steps)

    # ---- phase 3 (headline `value`): the same thread keeps DEPTH calls in flight (cvg_detect_scenes_submit / cvg_job_wait)
    accepted = 0
    last = {}                                          # what the last step of a loop handed back to its caller

    def loop_pipe(steps):
        nonlocal accepted
        jobs = []
        for k in range(steps):
            jobs.append(ctx.submit_scenes(models, resident[k % R], params=params, want_inliers=False))
            if len(jobs) > DEPTH - 1:
                accepted += int((jobs.pop(0).wait()[0]["status"] == 0).sum())
        for j in jobs:
            last["pipe"] = j.wait()[0]
            accepted += int((last["pipe"]["status"] == 0).sum())

    tw0 = time.time()                                  # clock samples: from the warm-up on (the timed region is short)
    loop_pipe(max(args.warmup, DEPTH))
    accepted = 0
    l0 = ctx.launch_count
    ms_total = timed(loop_pipe, args.steps)
    launches = ctx.launch_count - l0
    clocks.mark(tw0, time.time())
    value = world * B * args.steps / (ms_total * 1e-3)
    for sc in resident:
        sc.free()

    # ---- e2e: host buffers in; per-pair results, inlier masks' points and offsets out, every step -----------------------
    pinned = []
    for d, k, o in batches:
        pd = torch.from_numpy(d).pin_memory(); pk = torch.from_numpy(k).pin_memory()
        pinned.append((pd.numpy(), pk.numpy(), o, pd, pk))
    h2d = int(batches[0][0].nbytes + batches[0][1].nbytes + batches[0][2].nbytes)
    d2h_seen = []

    def loop_e2e_with(upload):
        """Streaming caller (the reference walks a list of test images, src/Output.cpp:27-47): every step's inputs cross PCIe
        inside the timed region (upload of step k+1.. enqueued while step k computes), and every step's per-pair results
        AND inlier points (what src/TestsDetector.cpp:87-94 hands to the consumer) come back to the host."""
        def loop(steps):
            inflight = []
            for k in range(steps):
                sc = upload(k % R)
                inflight.append((sc, ctx.submit_scenes(models, sc, params=params, want_inliers=True)))
                if len(inflight) > DEPTH - 1:
                    sc0, j0 = inflight.pop(0)
                    res, xy, off = j0.wait(); sc0.free()
                    d2h_seen.append(res.nbytes + xy.nbytes + off.nbytes)
            for sc0, j0 in inflight:
                res, xy, off = j0.wait(); sc0.free()
                d2h_seen.append(res.nbytes + xy.nbytes + off.nbytes)
                last["e2e"] = (res, xy, off)
        return loop

    loop_e2e = loop_e2e_with(lambda j: ctx.upload_scenes_async(pinned[j][0], pinned[j][1], pinned[j][2]))
    tw0 = time.time()
    loop_e2e(max(args.warmup, 2 * DEPTH))
    d2h_seen.clear()
    ms_e2e = timed(loop_e2e, args.steps)
    d2h = int(statistics.mean(d2h_seen))
    e2e_value = world * B * args.steps / (ms_e2e * 1e-3)
    clocks.mark(tw0, time.time())
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["pipe"], *last["e2e"][1:])
    clk = clocks.stop()

    # ---- same loop with uint8 descriptor rows in host memory (cv::SIFT can emit CV_8U; SURVEY 8f-3): extra key only
    e2e_u8 = None
    if args.desc == "sift" and not args.no_extras:
        pinned8 = []
        for d, k, o in batches:
            p8 = torch.from_numpy(d.astype(np.uint8)).pin_memory()
            pinned8.append((p8.numpy(), p8))
        loop_u8 = loop_e2e_with(lambda j: ctx.upload_scenes_u8_async(pinned8[j][0], pinned[j][1], pinned[j][2]))
        loop_u8(max(args.warmup, 2 * DEPTH))
        ms_u8 = timed(loop_u8, args.steps)
        e2e_u8 = {"value": world * B * args.steps / (ms_u8 * 1e-3), "unit": UNIT, "ms_per_step": ms_u8 / args.steps,
                  "h2d_bytes_per_step": int(batches[0][0].size + batches[0][1].nbytes + batches[0][2].nbytes),
                  "note": "uint8 descriptor rows in pinned host memory (cvg_scenes_upload_u8_async); not the headline"}

    # ---- single 8k x 8k pair: the match kernel's launch alone (SURVEY 8d target: <= 20.8 us) -----------------------------
    single_pair_us = None
    if not args.no_extras:
        d, k, o = batches[0]
        one = ctx.upload_scenes(d[:NT], k[:NT], o[:2])
        ctx.set_lanes(1); ctx.set_timing(True)
        ts = []
        for _ in range(6):
            ctx.detect_scenes(models, one, params=params)
            ts.append(ctx.last_timing()["match_ms"])
        ctx.set_timing(False); ctx.set_lanes(LANES)
        one.free()
        single_pair_us = 1e3 * min(ts[1:])

    # ---- N >= 2: BASELINE configs 4 and 5 on the same ranks, outside the c3 timed regions --------------------------------
    c4 = c5 = c5r = None
    if world > 1 and args.desc == "sift" and not args.no_multi:
        c5 = run_c5_match(ctx, dev, rank, world, dist, all_max, barrier)
        c5r = run_c5_ransac(ctx, api, dev, rank, world, all_max, barrier)
        c4 = run_c4(ctx, api, dev, rank, world, all_max, barrier)

    # ---- extra key: the reference's own dataset (BASELINE configs 1-2: 30 test images x 5 scales x 89 model views), when
    # the feature cache travelled with the tree (data_cache/, built by __graft_entry__.build() from the reference's
    # data with cv2 SIFT).  Per test image: one streaming upload of its 5 scaled scenes + one fused call, software-pipelined
    # on this one thread as the reference's processAllTestImages loop allows (src/Output.cpp:27-47 carries no state).
    real = None
    cache = os.path.join(ROOT, "data_cache", "features_full.npz")
    if rank == 0 and args.desc == "sift" and not args.no_extras and os.path.exists(cache):
        try:
            Z = np.load(cache)
            md = Z["model_desc"].astype(np.float32); so = Z["scene_offsets"]; n_img = (len(so) - 1) // 5
            sd = torch.from_numpy(Z["scene_desc"].astype(np.float32)).pin_memory(); sk = torch.from_numpy(Z["scene_kpt"].astype(np.float32)).pin_memory()
            sdn, skn = sd.numpy(), sk.numpy()
            rctx = api.Context(local)                      # own context: its buffer pools hold this workload's sizes
            rctx.set_lanes(LANES)
            rstream = torch.cuda.ExternalStream(rctx.stream, device=dev)
            rmodels = rctx.upload_models(md, Z["model_kpt"], Z["view_offsets"], Z["view_model"])
            sc5 = Z["scales"].astype(np.float32)

            def up(i):
                a, b = so[5 * i], so[5 * i + 5]
                return rctx.upload_scenes_async(sdn[a:b], skn[a:b], so[5 * i:5 * i + 6] - a)

            def whole(pipelined):
                hist = np.zeros(5, np.int64)
                torch.cuda.synchronize()
                r0 = torch.cuda.Event(enable_timing=True); r1 = torch.cuda.Event(enable_timing=True); r0.record(rstream)
                if pipelined:
                    fl = []
                    for i in range(n_img):
                        sc = up(i)
                        fl.append((sc, rctx.submit_scenes(rmodels, sc, scales=sc5, params=params)))
                        if len(fl) > DEPTH - 1:
                            sc0, j0 = fl.pop(0); res = j0.wait()[0]; sc0.free()
                            hist += np.bincount(res["status"].ravel(), minlength=5)[:5]
                    for sc0, j0 in fl:
                        res = j0.wait()[0]; sc0.free()
                        hist += np.bincount(res["status"].ravel(), minlength=5)[:5]
                else:
                    nxt = up(0)
                    for i in range(n_img):
                        cur = nxt; nxt = up(i + 1) if i + 1 < n_img else None
                        res = rctx.detect_scenes_inliers(rmodels, cur, scales=sc5, params=params)[0]
                        cur.free()
                        hist += np.bincount(res["status"].ravel(), minlength=5)[:5]
                r1.record(rstream); r1.synchronize()
                return hist, r0.elapsed_time(r1)
            whole(True); whole(False)                      # warm-up passes: allocations, lazy kernel loading
            hist, ms_real = whole(True)
            hist_s, ms_real_sync = whole(False)
            n_views = rmodels.n_views
            real = {"pairs": int(n_img * 5 * n_views), "images": int(n_img), "seconds": ms_real * 1e-3,
                    "pairs_per_s": n_img * 5 * n_views / (ms_real * 1e-3), "contexts": 1, "host_threads": 1,
                    "seconds_sync_calls": ms_real_sync * 1e-3,
                    "gate_histogram[accept,<4 matches,H empty,<4 inliers,det]": [int(v) for v in hist],
                    "gate_histogram_sync_equal": bool(np.array_equal(hist, hist_s)),
                    "note": f"host buffers in, per-pair results + inlier points out, one call per test image, {DEPTH} images in "
                            "flight from one thread (seconds) / strictly synchronous calls (seconds_sync_calls)"}
            rmodels.free(); rctx.close()
        except Exception as e:                             # the cache is optional
            real = {"unavailable": str(e)[:200]}

    if rank == 0:
        peaks = load_peaks()
        traffic = hyp_traffic = None                    # dram bytes per launch, from the committed ncu --set full captures
        tpath = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tpath):
            with open(tpath) as f:
                tj = json.load(f)
            traffic = tj.get("match_tc_kernel", {}).get("dram_bytes_per_pair", 0) * B or None
            hj = tj.get("ransac_score_kernel", {})
            if hj.get("measured_at_sets_per_launch") == B:
                hyp_traffic = hj.get("dram_bytes_per_launch")
        flops = 2.0 * NQ * NT * DIM * B
        kms = statistics.mean(match_ms)
        achieved = flops / (kms * 1e-3) / 1e12
        sm_hz = (clk.get("sm_mhz") or 1965.0) * 1e6
        score_s = max(sum(score_ms) * 1e-3, 1e-12)
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_total / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "bf16 operands (exact for u8 descriptors) / f32 accumulate; f64+f32 verify", "data": "synthetic",
                "config": {"workload": WORKLOAD, "pairs_per_step_per_gpu": B,
                           "descriptors": "fp32, integer-valued 0..255 (SIFT-like)" if args.desc == "sift" else
                                          "fp32, non-integer (candidate + fp32 re-rank match path)",
                           "match_path": ctx.last_match_path,
                           "scene_batches_rotated": R, "parallelism": f"pair-sharded x{world}, no data-path collective",
                           "contexts_per_gpu": 1, "host_threads_per_gpu": 1, "calls_in_flight": DEPTH, "lanes": LANES, "host_numa_node": numa,
                           "l2": f"{R} rotating batches, {R * B * NT * DIM * 2 / 2**20:.0f} MiB of bf16 operands > 126 MB L2"},
                "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": ms_e2e / args.steps,
                        "returns": "per-pair status/counts/H/det + inlier scene points + offsets (cvg_detect_scenes_submit with inlier buffers)"},
                "e2e_u8": e2e_u8,
                "real_dataset": real,
                "gpu_launches": int(launches),
                "clocks": clk,
                # The largest kernel of the step that has a roofline: the tcgen05 match kernel (tensor bound).  The refit/LM
                # kernel (ransac_finish_kernel) has a longer single launch when the kernels run alone, but it is 64 CTAs of
                # serial fp64 eigen-solves — latency, no roofline; with calls in flight it hides under the other calls' kernels.
                "roofline": {"kernel": "match_tc_kernel (tcgen05)", "bound": "tensor", "achieved": achieved,
                             "peak": peaks["bf16_burst"], "unit": "TFLOP/s", "frac": achieved / peaks["bf16_burst"],
                             "peak_sustained": peaks["bf16_sustained"], "frac_of_sustained": achieved / peaks["bf16_sustained"],
                             "peak_source": peaks["source"] + " (burst cuBLAS bf16: the timed region is tens of ms at full clocks)",
                             "kernel_ms_per_launch": kms, "launches_per_step": 1, "algorithmic_flops_per_launch": flops,
                             "share_of_step": sum(match_ms) / ms_serial, "traffic": traffic,
                             "single_pair_us": single_pair_us,
                             "timed_region": "serial pass (one lane, synchronous calls): with several calls in flight kernels of "
                                             "different batches overlap and a launch duration is no longer a utilisation figure"},
                # SURVEY 8d quotes scoring against HBM (16 B per (hypothesis, correspondence)); the set is shared-memory resident,
                # so that figure is reported as algorithmic_gbs and the utilisation is the fp32 issue fraction.
                "roofline_score": {"kernel": "ransac_score_kernel (inlier counting of a round's models, one hypothesis per thread, "
                                             "correspondences staged in shared memory; one launch per RANSAC round)",
                                   "bound": "fp32_issue",
                                   "achieved": 28.0 * sum(scored) / score_s / 1e12, "peak": 148 * 128 * sm_hz / 1e12,
                                   "unit": "T non-FMA fp32 instr/s (28 per (hypothesis, correspondence))",
                                   "frac": 28.0 * sum(scored) / score_s / (148 * 128 * sm_hz),
                                   "algorithmic_gbs": 16.0 * sum(scored) / score_s / 1e9, "hbm_peak_gbs": peaks["hbm"],
                                   "kernel_ms_per_launch": sum(score_ms) / max(sum(hyp_launches), 1),
                                   "launches_per_step": sum(hyp_launches) / args.steps,
                                   "algorithmic_bytes_per_launch": 16.0 * sum(scored) / max(sum(hyp_launches), 1),
                                   "share_of_step": sum(score_ms) / ms_serial, "traffic": hyp_traffic,
                                   "note": "a CTA reads its slice of the correspondences from HBM/L2 once and scores 256 hypotheses "
                                           "against it from shared memory: algorithmic_gbs exceeds the HBM peak by construction"},
                "solve_stage": {"kernel": "ransac_hyp_t_kernel (4-point DLT: bit-exact fp64 9x9 Jacobi, one hypothesis per thread; "
                                          "one launch per RANSAC round, rounds past the adaptive stop exit early)",
                                "ms_per_step": statistics.mean(hyp_ms), "launches_per_step": sum(hyp_launches) / args.steps,
                                "share_of_step": sum(hyp_ms) / ms_serial,
                                "note": "latency-bound (~140 dependent rotations per matrix); no bandwidth or tensor roofline applies"},
                # one context, one host thread in all three: serial (one lane; the rooflines' timed region), synchronous calls
                # split over the context's lanes, and the headline (calls_in_flight submitted ahead)
                "value_single_context": {"value": world * B * args.steps / (ms_sync * 1e-3), "unit": UNIT,
                                         "ms_per_step": ms_sync / args.steps,
                                         "note": "one context, one host thread, SYNCHRONOUS calls back to back, each split into sub-batches "
                                                 "over the context's lanes"},
                "value_serial": {"value": world * B * args.steps / (ms_serial * 1e-3), "unit": UNIT, "ms_per_step": ms_serial / args.steps,
                                 "note": "one lane: every kernel alone on the GPU (timed region of the rooflines)"},
                "stage_ms_per_step": {"match_kernel": kms, "verify": statistics.mean(ransac_ms), "verify_solve_kernels": statistics.mean(hyp_ms),
                                      "verify_score_kernels": statistics.mean(score_ms),
                                      "verify_rest(sampler, select, refit/LM finish, gates)": statistics.mean(ransac_ms) - statistics.mean(hyp_ms) - statistics.mean(score_ms)},
                "accepted_pairs": accepted}
        if c4 is not None:
            line["c4"] = c4
        if c5 is not None:
            line["c5_match"] = c5
        if c5r is not None:
            line["c5_ransac"] = c5r
        if world == 1 and not args.no_cpu:
            os.sched_setaffinity(0, all_cpus)           # the CPU baseline gets every core of the box
            threads = os.cpu_count() or 1
            n = 0; t_cpu = 0.0; kind = "reference"
            chunk = max(2, min(threads, 32, B))
            while t_cpu < args.cpu_seconds and n + chunk <= B:
                dt, kind = cpu_pairs(q, qk, batches[0], chunk, threads, first=n)
                t_cpu += dt; n += chunk
            line["cpu_baseline"] = {"value": n / t_cpu, "unit": UNIT, "cores": threads, "kind": kind,
                                    "sample": f"{n} pairs of the same workload (cv2 knnMatch on {threads} threads, "
                                              f"findHomography calls on a {threads}-thread pool)"}
        print(json.dumps(line), file=_RESULT_OUT, flush=True)
    models.free(); ctx.close()
    if world > 1:
        barrier()
        dist.destroy_process_group()


def main():
    global _RESULT_OUT
    sys.stdout.flush()
    _RESULT_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="cvgraft", choices=["cvgraft", "reference"])
    ap.add_argument("--pairs", type=int, default=64, help="scene sets (= pairs) per step per GPU")
    ap.add_argument("--batches", type=int, default=4, help="distinct scene batches rotated over the steps")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--depth", type=int, default=3,
                    help="calls the one host thread keeps in flight on the one context (cvg_detect_scenes_submit / cvg_job_wait)")
    ap.add_argument("--no-multi", action="store_true", help="N >= 2: skip the c4 / c5_match keys")
    ap.add_argument("--no-extras", action="store_true", help="skip the extra keys (e2e_u8, real_dataset): launch-list runs")
    ap.add_argument("--desc", default="sift", choices=["sift", "float"],
                    help="descriptor generator: integer-valued SIFT-like rows (default) or non-integer float rows")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step returned (per-pair results, inlier points) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 3) if args.impl == "cvgraft" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_cvgraft(args)


if __name__ == "__main__":
    main()
