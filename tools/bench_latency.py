"""Latency of the nq = 1 path (SURVEY.md 8f row 3): SoundDictionary::at_distance / match_sound issue ONE query per call
(examples/matcher.rs:39-48, SoundSequence::from_distances src/sound.rs:405-417). Wall clock of ss_dict_match(nq = 1) with host
buffers against the 100k-segment dictionary of config 4 (and the 10k one of config 3), both matchers; also nq = 8 and 128.
Then the from_distances chain of --walk-steps steps three ways in the same run: the host loop of ss_dict_match(nq = 1) it
replaces, ss_dict_walk (host buffers, wall clock) and ss_dict_walk_dev (CUDA events); the three must agree bit for bit.
  python tools/bench_latency.py [--out profiles/bench/latency.json] [--walk-steps 1000]"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from soundsym_b200 import api, synth  # noqa: E402
from soundsym_b200._lib import SS_COSINE_REF, SS_DTW  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--out", default="")
ap.add_argument("--reps", type=int, default=50)
ap.add_argument("--walk-steps", type=int, default=1000)
ap.add_argument("--walk-reps", type=int, default=5)
args = ap.parse_args()
ctx = api.Context(0)
res = {}
L2_BYTES = 126e6  # B200
try:
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True,
                         timeout=30).stdout.strip()
except (OSError, subprocess.SubprocessError):
    gpu = ""
res["gpu"] = gpu
print("GPU (name, power limit): %s" % gpu, flush=True)


def walk_rows(dev, d, doff, nd, start, steps, name):
    """from_distances over `dev`: host loop of nq = 1 matches vs ss_dict_walk vs ss_dict_walk_dev, same targets"""
    import torch
    n = len(steps)
    lens = np.diff(doff).astype(np.int64)
    one = lambda a: np.array([0, a.shape[0]], dtype=np.uint64)  # noqa: E731
    dev.walk(start, steps[:8])  # warm-up (workspaces, module load)
    cur, li, ld = start, [], []
    t0 = time.perf_counter()
    for t in steps:
        i, dd = dev.match(cur, one(cur), SS_COSINE_REF, 1, [t])
        li.append(int(i[0, 0]))
        ld.append(float(dd[0, 0]))
        cur = d[int(doff[li[-1]]):int(doff[li[-1] + 1])]
    loop_s = time.perf_counter() - t0
    wall = []
    for _ in range(args.walk_reps):
        t0 = time.perf_counter()
        wi, wd = dev.walk(start, steps)
        wall.append(time.perf_counter() - t0)
    assert np.array_equal(wi, np.array(li, dtype=np.uint32)), "walk indices differ from the nq = 1 loop"
    assert np.array_equal(wd.view(np.uint64), np.array(ld).view(np.uint64)), "walk distances differ from the nq = 1 loop"
    stream = torch.cuda.ExternalStream(ctx.stream)
    sq = api.DeviceQueries(ctx, start, one(start))
    d_t = torch.from_numpy(steps).cuda()
    d_i = torch.empty(n, dtype=torch.int32, device="cuda")
    d_d = torch.empty(n, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    ev = []
    for _ in range(args.walk_reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctx.check(ctx.lib.ss_dict_walk_dev(dev.h, sq.h, d_t.data_ptr(), n, d_i.data_ptr(), d_d.data_ptr()))
        e1.record(stream)
        e1.synchronize()
        ev.append(e0.elapsed_time(e1) * 1e-3)
    assert np.array_equal(d_i.cpu().numpy().view(np.uint32), wi) and np.array_equal(d_d.cpu().numpy().view(np.uint64), wd.view(np.uint64))
    # bytes a step must read: sum over segments of min(Kq, Kd) f64 values, plus the query (Kq = frames x C of the step's query)
    kq = np.concatenate([[start.shape[0]], lens[wi[:-1].astype(np.int64)]])
    srt = np.sort(lens)
    pre = np.concatenate([[0], np.cumsum(srt)])
    pos = np.searchsorted(srt, kq, side="right")
    frames = pre[pos] + (len(srt) - pos) * kq + kq
    step_bytes = float(frames.mean()) * d.shape[1] * 8
    dict_bytes = float(d.shape[0] * d.shape[1] * 8)
    dev_us, wall_us, loop_us = np.median(ev) / n * 1e6, np.median(wall) / n * 1e6, loop_s / n * 1e6
    row = {"steps": n, "dev_us_per_step": dev_us, "walk_wall_us_per_step": wall_us, "loop_nq1_us_per_step": loop_us,
           "gain_wall_vs_loop": loop_us / wall_us, "bytes_per_step": step_bytes, "achieved_GBps_dev": step_bytes / (dev_us * 1e-6) / 1e9,
           "dict_bytes": dict_bytes, "dict_fits_l2": dict_bytes <= L2_BYTES, "identical_to_loop": True}
    res["walk_cosine_ref_%s_nd%d" % (name, nd)] = row
    print("walk %-5s nd=%6d steps=%d: dev %7.1f us/step  ss_dict_walk %7.1f us/step  nq=1 loop %7.1f us/step  (x%.1f)  %.1f MB/step -> %.0f GB/s; "
          "dictionary %.0f MB (%s the 126 MB L2)" % (name, nd, n, dev_us, wall_us, loop_us, loop_us / wall_us, step_bytes / 1e6,
                                                    row["achieved_GBps_dev"], dict_bytes / 1e6, "fits" if row["dict_fits_l2"] else "exceeds"), flush=True)

q, qoff = synth.segments(256, 13, seed=5678)
for nd in (10000, 100000):
    d, doff = synth.segments(nd, 13, seed=1234)
    dev = api.DeviceDictionary(ctx, d, doff)
    for mode, name in ((SS_DTW, "dtw"), (SS_COSINE_REF, "cosine_ref")):
        for nq in (1, 8, 128):
            subs = []
            for r in range(args.reps + 5):
                i0 = (r * nq) % (256 - nq + 1)
                off = (qoff[i0:i0 + nq + 1] - qoff[i0]).astype(np.uint64)
                subs.append((np.ascontiguousarray(q[int(qoff[i0]):int(qoff[i0 + nq])]), off))
            for s, o in subs[:5]:
                dev.match(s, o, mode, 1)
            ts = []
            for s, o in subs[5:]:
                t0 = time.perf_counter()
                dev.match(s, o, mode, 1)
                ts.append((time.perf_counter() - t0) * 1e6)
            ts = np.array(ts)
            res["%s_nd%d_nq%d" % (name, nd, nq)] = {"median_us": float(np.median(ts)), "p10_us": float(np.percentile(ts, 10)), "p90_us": float(np.percentile(ts, 90)),
                                                    "calls_per_s": float(1e6 / np.median(ts))}
            print("%-10s nd=%6d nq=%3d: median %8.1f us  (p10 %8.1f, p90 %8.1f)" % (name, nd, nq, np.median(ts), np.percentile(ts, 10), np.percentile(ts, 90)), flush=True)
    if args.walk_steps > 0:
        # targets uniform in [-1, 1] from the first synthetic query: the chain drifts to short segments
        walk_rows(dev, d, doff, nd, np.ascontiguousarray(q[int(qoff[0]):int(qoff[1])]),
                  np.random.default_rng(nd).uniform(-1.0, 1.0, args.walk_steps), "mixed")
        # the most a step can read: from the first of the longest segments at target 1.0 the chain stays on that segment, and
        # every step reads min(Kq, Kd) = the whole of every segment
        li = int(np.argmax(np.diff(doff)))
        walk_rows(dev, d, doff, nd, np.ascontiguousarray(d[int(doff[li]):int(doff[li + 1])]), np.ones(args.walk_steps), "long")
    dev.close()
if args.out:
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    json.dump(res, open(args.out, "w"), indent=1)
