"""SoundSequence::from_distances for SS_DTW_TARGET (DESIGN.md §3.1i), three ways in the same run, as tools/bench_latency.py's
walk_rows does for the cosine walk: the host loop of ss_dict_match(nq = 1, SS_DTW_TARGET) it replaces (the first --loop-steps
steps, wall clock), ss_dict_walk_dtw (host buffers, wall clock) and ss_dict_walk_dtw_dev (CUDA events). The three must agree
bit for bit on the common steps. Dictionaries: configs 3 and 4 (synth.segments(10 000 | 100 000, 13, seed=1234), every pair on
the lane-per-segment path) and 2 000 segments of 1-400 frames (the warp-per-pair path). The chain starts from the first
synthetic query (seed 5678, of the same length range); targets are uniform between the 10th and 90th percentile of the start's
D row ("mid"), or NULL (t = 0).
Per step: us, cells = Lq * sum(Ld) (the band is not counted), cells/s, and the fraction of an FP64-pipe FLOOR. The floor is a
MODEL, not a measurement: 42 f64 operations per cell (13 x subtract, multiply, add for the cost; two min and one add for the
recurrence), 64 f64 operations per clock per SM, at the SM clock NVML reports during the timed region (bench.py's ClockSampler).
  python tools/bench_walk_dtw.py [--out profiles/bench/walk_dtw.json] [--steps 300] [--loop-steps 100]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import ClockSampler  # noqa: E402
from oracle import oracle as O  # noqa: E402
from soundsym_b200 import api, synth  # noqa: E402
from soundsym_b200._lib import SS_DTW, SS_DTW_TARGET  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="")
ap.add_argument("--steps", type=int, default=300)
ap.add_argument("--loop-steps", type=int, default=100)
ap.add_argument("--mixed-steps", type=int, default=40)
ap.add_argument("--reps", type=int, default=3)
args = ap.parse_args()
ctx = api.Context(0)
res = {"floor_model": "42 f64 operations per cell at 64 per clock per SM, SM clock from NVML during the timed region (a model, not a measurement)"}
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    gpu = ""
res["gpu"] = gpu
print("GPU (name, power limit): %s" % gpu, flush=True)
F64_OPS_PER_CELL, F64_PER_CLK_SM = 42, 64
NONE = 0xFFFFFFFF


def one(a):
    return np.array([0, a.shape[0]], dtype=np.uint64)


def walk_dtw_rows(dev, d, doff, start, steps, n, name):
    import torch
    lens = np.diff(doff).astype(np.int64)
    mode = SS_DTW if steps is None else SS_DTW_TARGET
    dev.walk_dtw(start, None if steps is None else steps[:4], 4)  # warm-up (workspaces, module load)
    nloop = min(args.loop_steps, n)
    cur, li, ld = start, [], []
    t0 = time.perf_counter()
    for s in range(nloop):
        i, dd = dev.match(cur, one(cur), mode, 1, None if steps is None else [steps[s]])
        li.append(int(i[0, 0]))
        ld.append(float(dd[0, 0]))
        cur = d[int(doff[li[-1]]):int(doff[li[-1] + 1])] if li[-1] != NONE else np.zeros((0, d.shape[1]))
    loop_s = time.perf_counter() - t0
    wall = []
    for _ in range(args.reps):
        t0 = time.perf_counter()
        wi, wd = dev.walk_dtw(start, steps, n)
        wall.append(time.perf_counter() - t0)
    assert np.array_equal(wi[:nloop], np.array(li, dtype=np.uint32)), "walk indices differ from the nq = 1 loop"
    assert np.array_equal(wd[:nloop].view(np.uint64), np.array(ld).view(np.uint64)), "walk distances differ from the nq = 1 loop"
    stream = torch.cuda.ExternalStream(ctx.stream)
    sq = api.DeviceQueries(ctx, start, one(start))
    d_t = torch.from_numpy(np.ascontiguousarray(steps)).cuda() if steps is not None else None
    d_i = torch.empty(n, dtype=torch.int32, device="cuda")
    d_d = torch.empty(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    clk = ClockSampler(0)
    clk.prepare()
    ev = []
    clk.start()
    for _ in range(args.reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.check(ctx.lib.ss_dict_walk_dtw_dev(dev.h, sq.h, d_t.data_ptr() if d_t is not None else None, n, d_i.data_ptr(), d_d.data_ptr()))
        e1.record(stream)
        e1.synchronize()
        ev.append(e0.elapsed_time(e1) * 1e-3)
    clocks = clk.stop()
    assert np.array_equal(d_i.cpu().numpy().view(np.uint32), wi) and np.array_equal(d_d.cpu().numpy().view(np.uint64), wd.view(np.uint64))
    lq = np.concatenate([[start.shape[0]], np.where(wi[:-1] != NONE, lens[np.minimum(wi[:-1], len(lens) - 1).astype(np.int64)], 0)])
    cells = float(lq.mean()) * float(lens.sum())
    sm_mhz = clocks.get("sm_mhz") or 1965.0
    floor_s = cells * F64_OPS_PER_CELL / (F64_PER_CLK_SM * ctx_sms * sm_mhz * 1e6)
    dev_us, wall_us, loop_us = np.median(ev) / n * 1e6, np.median(wall) / n * 1e6, loop_s / nloop * 1e6
    row = {"steps": n, "loop_steps": nloop, "nseg": len(lens), "dev_us_per_step": dev_us, "walk_wall_us_per_step": wall_us,
           "loop_nq1_us_per_step": loop_us, "gain_wall_vs_loop": loop_us / wall_us, "cells_per_step": cells,
           "cells_per_s": cells / (dev_us * 1e-6), "fp64_floor_model_us": floor_s * 1e6, "frac_of_fp64_floor_model": floor_s / (dev_us * 1e-6),
           "clocks": clocks, "identical_to_loop": True}
    res["walk_dtw_%s" % name] = row
    print("walk_dtw %-24s steps=%d: dev %8.1f us/step  ss_dict_walk_dtw %8.1f us/step  nq=1 loop %8.1f us/step (x%.1f)  %.3g cells/step "
          "%.3g cells/s  FP64 floor model %.1f us = %.2f of the step  (SM %s MHz)" % (name, n, dev_us, wall_us, loop_us, loop_us / wall_us, cells,
                                                                                 row["cells_per_s"], floor_s * 1e6, row["frac_of_fp64_floor_model"],
                                                                                 clocks.get("sm_mhz")), flush=True)


import torch  # noqa: E402

ctx_sms = torch.cuda.get_device_properties(0).multi_processor_count
for nd, lmin, lmax, n, name in ((10000, 4, 32, args.steps, "config3"), (100000, 4, 32, args.steps, "config4"),
                                (2000, 1, 400, args.mixed_steps, "mixed_1_400")):
    d, doff = synth.segments(nd, 13, lmin=lmin, lmax=lmax, seed=1234)
    q, qoff = synth.segments(8, 13, lmin=lmin, lmax=lmax, seed=5678)
    start = np.ascontiguousarray(q[int(qoff[0]):int(qoff[1])])
    row = O.dtw_matrix(d, doff, start, one(start), 13)[0]
    lo, hi = np.nanquantile(row, [0.1, 0.9])
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    walk_dtw_rows(dev, d, doff, start, np.random.default_rng(nd).uniform(lo, hi, n), n, name + "_mid")
    walk_dtw_rows(dev, d, doff, start, None, n, name + "_t0")
    dev.close()
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
