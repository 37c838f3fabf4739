"""SS_DTW_TARGET (DESIGN.md §3.1h) timed with CUDA events beside SS_DTW and SS_COSINE_REF.

  python tools/bench_target.py [--reps 3] [--seconds 3600] [--out profiles/bench/target.json]

Workloads (k = 1):
  config3   synth.segments(10 000, seed=1234) x the 1 000 queries of synth.segments(1 000, seed=5678)
  config4   synth.segments(100 000, seed=1234) x the 10 000 queries of synth.segments(10 000, seed=5678) (bench.py's workload)
  config5   examples/reconstruction.rs' match on `--seconds` of synthetic audio (tools/config5.py's flow: source = first half,
            target = second half, Partitioner threshold 4 / depth 3, model seed 3): target segments x source segments, 12 coefficients
Cases per workload:
  dtw                SS_DTW (the targets passed are ignored)
  cosine_ref         SS_COSINE_REF with targets 1.0
  target_t0          SS_DTW_TARGET, t = 0
  target_c1.5, _c3   SS_DTW_TARGET, t = c x the query's nearest SS_DTW distance
  target_median      SS_DTW_TARGET, t = the median of the exact distances of 8 queries x 2 000 segments (oracle, f64)
Each time is the median of `reps` event-timed calls of ss_dict_match_dev + ss_dict_match_finish, the L2 overwritten (256 MB >
126 MB) before every call, after one warm-up call; last_exhaustive is the number of queries the call sent to the exhaustive f64
stage. One JSON document with the card's name and power limit, read in the same run.
"""
import argparse
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from bench_locate import gpu_name  # noqa: E402


def config5_inputs(seconds):
    from soundsym_b200 import api, synth
    ctx = api.default_context()
    audio = synth.audio(seconds, seed=42)
    half = (len(audio) // 2 // 256) * 256
    src = api.Sound.from_samples(audio[:half], 44100.0, ctx=ctx)
    part = api.Partitioner(src, ctx).set_threshold(4).set_depth(3)  # examples/reconstruction.rs:43-45
    part.train(seed=3)

    def cut(snd):
        part.sound = snd
        off = np.zeros(1, dtype=np.uint64)
        off = np.concatenate([off, np.cumsum(np.asarray(part.partition(), dtype=np.uint64) // np.uint64(256))])
        return snd.mfcc_arrays()[:int(off[-1])], off

    d, doff = cut(src)
    q, qoff = cut(api.Sound.from_samples(audio[half:], 44100.0, ctx=ctx))
    return d, doff, q, qoff


def median_target(d, doff, q, qoff):
    from oracle import oracle as O
    rng = np.random.default_rng(11)
    nq, nseg = len(qoff) - 1, len(doff) - 1
    qs = rng.choice(nq, size=min(8, nq), replace=False)
    segs = np.sort(rng.choice(nseg, size=min(2000, nseg), replace=False))
    qparts = [q[int(qoff[i]):int(qoff[i + 1])] for i in qs]
    dparts = [d[int(doff[j]):int(doff[j + 1])] for j in segs]

    def pack(parts):
        off = np.zeros(len(parts) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([p.shape[0] for p in parts])
        return np.concatenate(parts, axis=0), off

    dd, ddo = pack(dparts)
    qq, qqo = pack(qparts)
    D = O.dtw_matrix(dd, ddo, qq, qqo, d.shape[1])
    return float(np.nanmedian(D[np.isfinite(D)]))


def run_workload(name, d, doff, q, qoff, reps):
    import torch
    from soundsym_b200 import api
    from soundsym_b200._lib import SS_COSINE_REF, SS_DTW, SS_DTW_TARGET
    ctx = api.default_context()
    c = d.shape[1]
    dev = api.DeviceDictionary(ctx, d, doff, c)
    qs = api.DeviceQueries(ctx, q, qoff, c)
    nq = len(qoff) - 1
    stream = torch.cuda.ExternalStream(ctx.stream)
    o_idx = torch.empty(max(nq, 1), dtype=torch.int32, device="cuda")
    o_dist = torch.empty(max(nq, 1), dtype=torch.float64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def timed(mode, t):
        td = torch.from_numpy(np.ascontiguousarray(t, dtype=np.float64)).cuda()
        torch.cuda.synchronize()

        def call():
            ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, mode, td.data_ptr(), 1, o_idx.data_ptr(), o_dist.data_ptr()))
            ctx.check(ctx.lib.ss_dict_match_finish(dev.h))

        ms, exh = [], []
        with torch.cuda.stream(stream):
            call()
            ctx.sync()
            for _ in range(reps):
                flush.zero_()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(stream)
                call()
                e1.record(stream)
                ctx.sync()
                torch.cuda.synchronize()
                ms.append(e0.elapsed_time(e1))
                exh.append(int(dev.last_exhaustive))
        return {"median_ms": float(np.median(ms)), "ms": [round(x, 3) for x in ms], "last_exhaustive": exh,
                "last_scan_kind": int(dev.last_scan_kind)}, o_dist.cpu().numpy()[:nq].copy()

    res = {"workload": name, "nq": int(nq), "nseg": int(len(doff) - 1), "dict_frames": int(doff[-1]), "query_frames": int(qoff[-1]),
           "cells": float(np.diff(qoff).astype(np.float64).sum() * float(doff[-1])), "cases": {}}
    res["cases"]["dtw"], nearest = timed(SS_DTW, np.zeros(nq))
    res["cases"]["cosine_ref"], _ = timed(SS_COSINE_REF, np.ones(nq))
    res["cases"]["target_t0"], _ = timed(SS_DTW_TARGET, np.zeros(nq))
    near = np.where(np.isfinite(nearest), nearest, 0.0)
    for cf in (1.5, 3.0):
        res["cases"]["target_c%g" % cf], _ = timed(SS_DTW_TARGET, cf * near)
    tm = median_target(d, doff, q, qoff)
    res["median_target"] = tm
    res["cases"]["target_median"], _ = timed(SS_DTW_TARGET, np.full(nq, tm))
    print(json.dumps(res), flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--seconds", type=float, default=3600.0, help="config 5's audio length (source = first half)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "bench", "target.json"))
    args = ap.parse_args()
    import torch
    from soundsym_b200 import synth
    res = {"gpu": gpu_name(), "torch_device": torch.cuda.get_device_name(0), "reps": args.reps, "l2": "overwritten before every call",
           "workloads": []}
    for name, nd, nq in (("config3", 10000, 1000), ("config4", 100000, 10000)):
        d, doff = synth.segments(nd, 13, seed=1234)
        q, qoff = synth.segments(nq, 13, seed=5678)
        res["workloads"].append(run_workload(name, d, doff, q, qoff, args.reps))
    d, doff, q, qoff = config5_inputs(args.seconds)
    res["workloads"].append(run_workload("config5", d, doff, q, qoff, args.reps))
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps({"gpu": res["gpu"], "out": args.out}))


if __name__ == "__main__":
    main()
