"""ss_dict_locate_dev (subsequence DTW, DESIGN.md §3.1g) timed with CUDA events.

  python tools/bench_locate.py [--reps 5] [--seconds 3600] [--out profiles/bench/locate.json]

Cases (k = 1; cells = sum over (query, segment) pairs of Lq * Ld, computed here from the offsets):
  config3        synth.segments(10 000, seed=1234) x the 1 000 queries of synth.segments(1 000, seed=5678)
  config5        config 5's target segments (tools/config5.py: synthetic audio, source = first half, target = second half,
                 Partitioner threshold 4 / depth 3, model seed 3) against the UNSEGMENTED source as one dictionary sound
  config5_nq1    the first non-empty target segment alone against that source: the latency of one warp walking every column
Each is the median of `reps` event-timed calls with the L2 overwritten before every call (256 MB > 126 MB), after one warm-up
call. One JSON document with the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except Exception as e:  # the name then comes from torch alone
        return "nvidia-smi unavailable (%s)" % e


def config5_inputs(seconds):
    from soundsym_b200 import api, synth
    ctx = api.default_context()
    audio = synth.audio(seconds, seed=42)
    half = (len(audio) // 2 // 256) * 256
    src = api.Sound.from_samples(audio[:half], 44100.0, ctx=ctx)
    part = api.Partitioner(src, ctx).set_threshold(4).set_depth(3)  # examples/reconstruction.rs:43-45
    part.train(seed=3)
    part.sound = api.Sound.from_samples(audio[half:], 44100.0, ctx=ctx)
    tsplits = part.partition()
    qoff = np.zeros(len(tsplits) + 1, dtype=np.uint64)
    qoff[1:] = np.cumsum(np.asarray(tsplits, dtype=np.uint64) // np.uint64(256))
    dm = src.mfcc_arrays()
    return dm, np.array([0, dm.shape[0]], dtype=np.uint64), part.sound.mfcc_arrays()[:int(qoff[-1])], qoff


def time_case(name, d, doff, q, qoff, reps):
    import torch
    from soundsym_b200 import api
    ctx = api.default_context()
    dev = api.DeviceDictionary(ctx, d, doff, d.shape[1])
    qs = api.DeviceQueries(ctx, q, qoff, d.shape[1])
    nq = qoff.shape[0] - 1
    stream = torch.cuda.ExternalStream(ctx.stream)
    out = [torch.empty(nq, dtype=torch.int32, device="cuda") for _ in range(3)] + [torch.empty(nq, dtype=torch.float64, device="cuda")]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def call():
        ctx.check(ctx.lib.ss_dict_locate_dev(dev.h, qs.h, 1, *[t.data_ptr() for t in out]))

    with torch.cuda.stream(stream):
        n0 = ctx.launches
        call()
        launches = ctx.launches - n0
        ctx.sync()
        ms = []
        for _ in range(reps):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            call()
            e1.record(stream)
            ctx.sync()
            torch.cuda.synchronize()
            ms.append(e0.elapsed_time(e1))
    lq = np.diff(qoff).astype(np.float64)
    ld = np.diff(doff).astype(np.float64)
    cells = float(lq.sum() * ld.sum())
    med = float(np.median(ms))
    cost = out[3].cpu().numpy()
    return {"case": name, "nq": int(nq), "nseg": int(doff.shape[0] - 1), "query_frames": int(lq.sum()), "dict_frames": int(ld.sum()),
            "cells": cells, "median_ms": med, "ms": [round(x, 4) for x in ms], "cells_per_s": cells / (med * 1e-3), "launches": int(launches),
            "hits": int(np.isfinite(cost).sum())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--seconds", type=float, default=3600.0, help="config 5's audio length (source = first half)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench", "locate.json"))
    args = ap.parse_args()
    import torch
    from soundsym_b200 import synth
    res = {"gpu": gpu_name(), "torch_device": torch.cuda.get_device_name(0), "reps": args.reps, "cases": []}
    d, doff = synth.segments(10000, 13, seed=1234)
    q, qoff = synth.segments(1000, 13, seed=5678)
    res["cases"].append(time_case("config3", d, doff, q, qoff, args.reps))
    print(json.dumps(res["cases"][-1]), flush=True)
    dm, dmoff, qm, qmoff = config5_inputs(args.seconds)
    res["cases"].append(time_case("config5", dm, dmoff, qm, qmoff, args.reps))
    print(json.dumps(res["cases"][-1]), flush=True)
    first = int(np.flatnonzero(np.diff(qmoff) > 0)[0])
    one = qm[int(qmoff[first]):int(qmoff[first + 1])]
    res["cases"].append(time_case("config5_nq1", dm, dmoff, one, np.array([0, one.shape[0]], dtype=np.uint64), args.reps))
    print(json.dumps(res["cases"][-1]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "out": args.out}))


if __name__ == "__main__":
    main()
