"""SS_DTW matches and ss_dict_align_dev under a Sakoe-Chiba band (ss_dict_set_dtw_band), timed with CUDA events on one GPU.

  python tools/bench_band.py [--radii 0,1,2,4,8,32,2048] [--cases config3,config4,config5,align] [--seconds 600] [--out path.json]

Cases (C = 13):
  config3   synthetic 10 000-segment dictionary x 1 000 queries, L ~ U{4..32} (soundsym_b200.synth, seeds 1234 / 5678)
  config4   synthetic 100 000-segment dictionary x 10 000 queries, L ~ U{4..32}
  config5   examples/reconstruction.rs' match on `--seconds` of synthetic 44.1 kHz audio (tools/config5.py's front end: source =
            first half, target = second half, Partitioner threshold 4, depth 3); segments of up to several hundred frames
  align     ss_dict_align_dev on 1 000 fixed pairs (query p, segment p) of 33-400 frames
Per radius, a match case records the median of `reps` event-timed ss_dict_match_dev + ss_dict_match_finish calls (k = 1, after
one warm-up call) and the stage counters of the last call; r = 2048 is checked bit for bit against r = 0 (it covers every
pair of these workloads). The align case records the median of `reps` calls with L2 overwritten before each (256 MB), the
cells inside the band and the cells the kernels visit (32-row step blocks x 32 lanes per strip, DESIGN.md §3.1f).
One JSON line per case, with the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

MATCH_REPS = {"config3": 10, "config4": 3, "config5": 3}


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except Exception as e:
        return "nvidia-smi unavailable (%s)" % e


def band_rows(j, la, lb, r):
    """rows [lo, hi] of column j inside the band of radius r >= 1 (exact.cu band_rows)"""
    A, B = lb - 1, la - 1
    if A == 0:
        return 0, la - 1
    w, x = min(r, max(la, lb)) * max(A, B), j * B
    lo = 0 if x - w <= 0 else (x - w + A - 1) // A
    return lo, min(la - 1, (x + w) // A)


def cell_counts(la, lb, r):
    """(cells inside the band, cells the exact kernels visit) of one pair"""
    if r == 0:
        inside = la * lb
    else:
        inside = sum(hi - lo + 1 for lo, hi in (band_rows(j, la, lb, r) for j in range(lb)))
    if la <= 32 and lb <= 32:
        return inside, la * lb  # one warp: every cell of the wavefront
    visited, nsteps = 0, la + 31
    for s in range((lb + 31) // 32):
        t0b, t0e = 0, nsteps
        if r:
            t0b = band_rows(32 * s, la, lb, r)[0] & ~31
            t0e = min(nsteps, band_rows(min(32 * s + 31, lb - 1), la, lb, r)[1] + 32)
        visited += ((t0e - t0b + 31) // 32) * 32 * 32
    return inside, visited


def config5_workload(seconds, ctx):
    from soundsym_b200 import api, synth
    audio = synth.audio(seconds, seed=42)
    half = (len(audio) // 2 // 256) * 256
    src = api.Sound.from_samples(audio[:half], 44100.0, ctx=ctx)
    part = api.Partitioner(src, ctx).set_threshold(4).set_depth(3)
    part.train(seed=3)
    splits = part.partition()
    tgt = api.Sound.from_samples(audio[half:], 44100.0, ctx=ctx)
    part.sound = tgt
    tsplits = part.partition()
    doff = np.zeros(len(splits) + 1, dtype=np.uint64)
    doff[1:] = np.cumsum(np.asarray(splits, dtype=np.uint64) // np.uint64(256))
    qoff = np.zeros(len(tsplits) + 1, dtype=np.uint64)
    qoff[1:] = np.cumsum(np.asarray(tsplits, dtype=np.uint64) // np.uint64(256))
    return src.mfcc_arrays()[: int(doff[-1])], doff, tgt.mfcc_arrays()[: int(qoff[-1])], qoff


def match_case(name, radii, seconds, gpu):
    import torch
    from soundsym_b200 import api, synth
    from soundsym_b200._lib import SS_DTW
    ctx = api.Context(0)
    if name == "config5":
        d, doff, q, qoff = config5_workload(seconds, ctx)
        workload = "examples/reconstruction.rs match on %.0f s of synthetic audio (config 5 front end)" % seconds
    else:
        nd, nq = (10000, 1000) if name == "config3" else (100000, 10000)
        d, doff = synth.segments(nd, 13, seed=1234)
        q, qoff = synth.segments(nq, 13, seed=5678)
        workload = "synthetic %d-segment dictionary x %d queries, L ~ U{4..32}" % (nd, nq)
    c = d.shape[1]
    nq = len(qoff) - 1
    dev = api.DeviceDictionary(ctx, d, doff, c)
    qs = api.DeviceQueries(ctx, q, qoff, c)
    stream = torch.cuda.ExternalStream(ctx.stream)
    o_idx = torch.empty((nq, 1), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((nq, 1), dtype=torch.float64, device="cuda")
    L = ctx.lib

    def match():
        ctx.check(L.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 1, o_idx.data_ptr(), o_dist.data_ptr()))
        ctx.check(L.ss_dict_match_finish(dev.h))

    rows, ref = [], None
    for r in radii:
        dev.set_dtw_band(r)
        match()
        ctx.sync()
        out = (o_idx.cpu().numpy().copy(), o_dist.cpu().numpy().copy())
        if r == 0:
            ref = out
        times = []
        for _ in range(MATCH_REPS[name]):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            match()
            e1.record(stream)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        row = {"r": r, "match_ms": {"median": float(np.median(times)), "min": float(np.min(times)), "max": float(np.max(times))},
               "last_tc_fallback": dev.last_tc_fallback, "last_exhaustive": dev.last_exhaustive, "last_uncertified": dev.last_uncertified}
        if ref is not None and r >= 2048:
            row["equals_r0_bit_for_bit"] = bool(np.array_equal(out[0], ref[0]) and np.array_equal(out[1].view(np.uint64), ref[1].view(np.uint64)))
        if ref is not None and 0 < r < 2048:
            row["top1_differs_from_r0"] = int(np.sum(out[0] != ref[0]))
        rows.append(row)
        print(json.dumps({"case": name, **row}), file=sys.stderr, flush=True)
    return {"case": name, "gpu": gpu, "workload": workload, "nd": len(doff) - 1, "nq": nq, "max_len": [int(np.diff(doff).max()), int(np.diff(qoff).max())],
            "k": 1, "reps": MATCH_REPS[name], "l2": "not flushed (the match's working set is its own)", "radii": rows}


def align_case(radii, reps, gpu):
    import torch
    from soundsym_b200 import api, synth
    n = 1000
    d, doff = synth.segments(n, 13, lmin=33, lmax=400, seed=1234)
    q, qoff = synth.segments(n, 13, lmin=33, lmax=400, seed=5678)
    ctx = api.Context(0)
    L = ctx.lib
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    stream = torch.cuda.ExternalStream(ctx.stream)
    lq, ld = np.diff(qoff).astype(np.int64), np.diff(doff).astype(np.int64)
    cap = int(np.sum(lq + dev.max_len - 1))
    seg = torch.arange(n, dtype=torch.int32, device="cuda")
    d_path = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    d_off = torch.empty(n + 1, dtype=torch.int64, device="cuda")
    d_dist = torch.empty(n, dtype=torch.float64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def align():
        ctx.check(L.ss_dict_align_dev(dev.h, qs.h, seg.data_ptr(), d_path.data_ptr(), cap, d_off.data_ptr(), d_dist.data_ptr()))

    rows = []
    for r in radii:
        dev.set_dtw_band(r)
        align()
        ctx.sync()
        times = []
        for _ in range(reps):
            with torch.cuda.stream(stream):
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            align()
            e1.record(stream)
            e1.synchronize()
            times.append(e0.elapsed_time(e1))
        inside = visited = 0
        for p in range(n):
            a, b = cell_counts(int(lq[p]), int(ld[p]), r)
            inside += a
            visited += b
        rows.append({"r": r, "align_ms": {"median": float(np.median(times)), "min": float(np.min(times)), "max": float(np.max(times))},
                     "cells_inside_band": inside, "cells_visited": visited, "path_cells": int(d_off[-1].item()),
                     "finite_distances": int(np.isfinite(d_dist.cpu().numpy()).sum())})
        print(json.dumps({"case": "align", **rows[-1]}), file=sys.stderr, flush=True)
    return {"case": "align", "gpu": gpu, "pairs": n, "lengths": [33, 400], "reps": reps, "l2": "overwritten before every call",
            "dp_cells_unbanded": int(np.sum(lq * ld)), "radii": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--radii", default="0,1,2,4,8,32,2048")
    ap.add_argument("--cases", default="config3,config4,config5,align")
    ap.add_argument("--seconds", type=float, default=600.0, help="config 5: seconds of synthetic audio")
    ap.add_argument("--reps", type=int, default=20, help="align: timed calls per radius")
    ap.add_argument("--out", default=None, help="also write the lines as one JSON list here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_band.py needs a CUDA device")
    radii = [int(x) for x in args.radii.split(",")]
    gpu = gpu_name()
    lines = []
    for name in args.cases.split(","):
        r = align_case(radii, args.reps, gpu) if name == "align" else match_case(name, radii, args.seconds, gpu)
        print(json.dumps(r), flush=True)
        lines.append(r)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, "w") as f:
                json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
