"""The config-5 flow with the warped resynthesis (ss_resynth_warped) next to the plain one (ss_resynth) on one B200.

  python tools/bench_resynth_warp.py [--seconds 3600] [--mode cosine|dtw] [--reps 5] [--out profiles/bench/resynth_warp.json]

examples/reconstruction.rs on synthetic 44.1 kHz audio (source = first half, target = second half), then on the same
target segments and indices:
  match      ss_dict_match (host buffers, k = 1) in the chosen mode
  align      ss_dict_align of those indices (the DTW path, whatever matcher chose them)
  resynth    ss_resynth          (host buffers: dictionary samples up, output down, one kernel)
  warped     ss_resynth_warped   (the same plus the paths)
Wall clock: the median of `reps` calls, each ending in a stream synchronisation. Kernel time: a separate torch.profiler run
of the two resynthesis calls (k_resynth, k_resynth_warped), median over `reps` launches. Also reported: the bytes each kernel
must move per output sample, how many target samples the plain resynthesis zero-padded or cut, and how many output blocks
the warped one crossfades. The warped output is checked against the numpy twin (tests/warp_reference.py).
The card's name and power limit are read in the same run. Needs a CUDA device.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
H = 256


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except Exception as e:
        return "nvidia-smi unavailable (%s)" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--seconds", type=float, default=3600.0)
    ap.add_argument("--mode", default="cosine", choices=["cosine", "dtw"])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write the JSON record here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_resynth_warp.py needs a CUDA device")
    import warp_reference as W
    from soundsym_b200 import api, synth
    from soundsym_b200._lib import SS_COSINE_REF, SS_DTW
    gpu = gpu_name()
    ctx = api.Context(0)
    mode = SS_DTW if args.mode == "dtw" else SS_COSINE_REF

    audio = synth.audio(args.seconds, seed=42)
    half = (len(audio) // 2 // H) * H
    src = api.Sound.from_samples(audio[:half], 44100.0, ctx=ctx)
    part = api.Partitioner(src, ctx).set_threshold(4).set_depth(3)  # examples/reconstruction.rs:43-45
    part.train(seed=3)
    splits = part.partition()
    tgt = api.Sound.from_samples(audio[half:], 44100.0, ctx=ctx)
    part.sound = tgt
    tsplits = part.partition()
    doff = np.zeros(len(splits) + 1, dtype=np.uint64)
    doff[1:] = np.cumsum(np.asarray(splits, dtype=np.uint64) // np.uint64(H))
    qoff = np.zeros(len(tsplits) + 1, dtype=np.uint64)
    qoff[1:] = np.cumsum(np.asarray(tsplits, dtype=np.uint64) // np.uint64(H))
    dm, qm = src.mfcc_arrays()[: int(doff[-1])], tgt.mfcc_arrays()[: int(qoff[-1])]
    soff = np.zeros(len(splits) + 1, dtype=np.uint64)
    soff[1:] = np.cumsum(np.asarray(splits, dtype=np.uint64))
    ds = np.ascontiguousarray(src.samples()[: int(soff[-1])])
    tl = np.asarray(tsplits, dtype=np.uint64)
    dev = api.DeviceDictionary(ctx, dm, doff, api.NCOEFFS)

    def wall(fn):
        ts, r = [], None
        for _ in range(args.reps):
            ctx.sync()
            t = time.perf_counter()
            r = fn()
            ctx.sync()
            ts.append((time.perf_counter() - t) * 1e3)
        return r, {"median": float(np.median(ts)), "min": float(np.min(ts)), "max": float(np.max(ts))}

    (idx, _), match_ms = wall(lambda: dev.match(qm, qoff, mode, 1))
    idx = idx[:, 0]
    (paths, _), align_ms = wall(lambda: dev.align(qm, qoff, idx))
    cells, poff = W.flatten(paths)
    plain, resynth_ms = wall(lambda: ctx.resynth(ds, soff, idx, tl))
    warped, warped_ms = wall(lambda: ctx.resynth_warped(ds, soff, idx, cells, poff, tl))
    ooff = np.concatenate([[0], np.cumsum(tl.astype(np.int64))])
    for a in range(0, len(tl), 1000):  # the twin in slices of segments, to bound its memory
        b = min(a + 1000, len(tl))
        c, o = W.flatten(paths[a:b])
        assert np.array_equal(warped[ooff[a]:ooff[b]], W.resynth_warped(ds, soff, idx[a:b], c, o, tl[a:b])), "warped differs from the twin"

    # kernel time in a run of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(args.reps):
            ctx.resynth(ds, soff, idx, tl)
            ctx.resynth_warped(ds, soff, idx, cells, poff, tl)
        torch.cuda.synchronize()
    kern = {}
    for ev in prof.events():
        if "k_resynth(" in ev.name or ev.name.startswith("_ZN2ss9k_resynthE"):
            kern.setdefault("k_resynth", []).append(ev.device_time_total / 1e3)
        elif "k_resynth_warped" in ev.name:
            kern.setdefault("k_resynth_warped", []).append(ev.device_time_total / 1e3)
    kernel_ms = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "n": len(v)} for k, v in kern.items()}

    total = int(tl.sum())
    dlen = np.diff(soff).astype(np.int64)[idx]
    tl64 = tl.astype(np.int64)
    padded = int(np.sum(np.maximum(tl64 - dlen, 0)))
    cut = int(np.sum(np.maximum(dlen - tl64, 0)))
    nblocks = int(np.sum((tl64 + H - 1) // H))
    crossfaded = 0
    for t, p in enumerate(paths):  # blocks whose source frame is not one past the previous block's
        g = (int(tl64[t]) + H - 1) // H
        if len(p) == 0 or g < 2:
            continue
        first = np.ones(len(p), dtype=bool)
        first[1:] = p[1:, 0] != p[:-1, 0]
        rj = p[first, 1].astype(np.int64)
        b = np.arange(g)
        row = np.minimum(b, len(rj) - 1)
        j = rj[row] + (b - row)
        crossfaded += int(np.sum(np.diff(j) != 1))
    bytes_warped = 8 * total + 8 * total + 8 * H * crossfaded  # write + read a + read c where a block crossfades
    rec = {"tool": "bench_resynth_warp", "gpu": gpu, "config": "config 5: examples/reconstruction.rs on %.0f s synthetic 44.1 kHz audio, %s matcher"
           % (args.seconds, args.mode), "dictionary_segments": len(splits), "target_segments": len(tsplits), "output_samples": total,
           "path_cells": int(poff[-1]), "reps": args.reps,
           "wall_ms": {"match": match_ms, "align": align_ms, "resynth": resynth_ms, "resynth_warped": warped_ms},
           "kernel_ms": kernel_ms,
           "bytes_per_output_sample": {"k_resynth": 16.0, "k_resynth_warped": bytes_warped / max(total, 1)},
           "plain_resynth_zero_padded_samples": padded, "plain_resynth_cut_samples": cut,
           "plain_resynth_changed_fraction": (padded + cut) / max(total, 1),
           "warped_blocks": nblocks, "warped_crossfaded_blocks": crossfaded,
           "warped_differs_from_plain_samples": int(np.sum(warped != plain)), "warped_equals_twin": True}
    print(json.dumps(rec), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
