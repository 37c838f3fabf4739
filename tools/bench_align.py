"""ss_dict_align_dev timed with CUDA events on the top-1 results of a DTW match, next to the match itself in the same run.

  python tools/bench_align.py [--reps 20] [--out path.json]

Cases (synthetic inputs of soundsym_b200.synth, C = 13):
  config3   10 000-segment dictionary x 1 000 queries, L ~ U{4..32}
  config4   100 000-segment dictionary x 10 000 queries, L ~ U{4..32}
  long      2 000-segment dictionary x 1 000 queries, L ~ U{33..400} (every pair takes the strip kernel)
For each: the match (ss_dict_match_dev + ss_dict_match_finish, k = 1) and the align of its indices (ss_dict_align_dev), each the
median of `reps` event-timed calls with the L2 overwritten before every call (256 MB > 126 MB). The align's distances are
checked bit for bit against the match's. One JSON line per case, carrying the card's name and power limit.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

CASES = {"config3": (10000, 1000, 4, 32), "config4": (100000, 10000, 4, 32), "long": (2000, 1000, 33, 400)}


def gpu_name():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"], capture_output=True,
                              text=True, timeout=60).stdout.strip()
    except Exception as e:  # the name then comes from torch alone
        return "nvidia-smi unavailable (%s)" % e


def run_case(name, reps, gpu):
    import torch
    from soundsym_b200 import api, synth
    from soundsym_b200._lib import SS_DTW
    nd, nq, lmin, lmax = CASES[name]
    d, doff = synth.segments(nd, 13, lmin=lmin, lmax=lmax, seed=1234)
    q, qoff = synth.segments(nq, 13, lmin=lmin, lmax=lmax, seed=5678)
    ctx = api.Context(0)
    L = ctx.lib
    dev = api.DeviceDictionary(ctx, d, doff, 13)
    qs = api.DeviceQueries(ctx, q, qoff, 13)
    stream = torch.cuda.ExternalStream(ctx.stream)
    lq = np.diff(qoff).astype(np.int64)
    cap = int(np.sum(lq[lq > 0] + dev.max_len - 1))
    o_idx = torch.empty((nq, 1), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((nq, 1), dtype=torch.float64, device="cuda")
    d_path = torch.empty((cap, 2), dtype=torch.int32, device="cuda")
    d_off = torch.empty(nq + 1, dtype=torch.int64, device="cuda")
    d_dist = torch.empty(nq, dtype=torch.float64, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()

    def match():
        ctx.check(L.ss_dict_match_dev(dev.h, qs.h, SS_DTW, None, 1, o_idx.data_ptr(), o_dist.data_ptr()))
        ctx.check(L.ss_dict_match_finish(dev.h))

    def align():
        ctx.check(L.ss_dict_align_dev(dev.h, qs.h, o_idx.data_ptr(), d_path.data_ptr(), cap, d_off.data_ptr(), d_dist.data_ptr()))

    def timed(fn):
        out = []
        for _ in range(reps):
            with torch.cuda.stream(stream):
                flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            fn()
            e1.record(stream)
            e1.synchronize()
            out.append(e0.elapsed_time(e1))
        return float(np.median(out)), float(np.min(out)), float(np.max(out))

    match()
    align()  # warm-up of both shapes
    ctx.sync()
    n0 = ctx.launches
    align()
    launches = ctx.launches - n0
    ctx.sync()
    mdist, adist = o_dist.cpu().numpy()[:, 0], d_dist.cpu().numpy()
    assert np.array_equal(mdist.view(np.uint64), adist.view(np.uint64)), "align distances differ from the match's"
    cells = int(d_off[-1].item())
    m_med, m_min, m_max = timed(match)
    a_med, a_min, a_max = timed(align)
    return {"case": name, "gpu": gpu, "nd": nd, "nq": nq, "lengths": [lmin, lmax], "reps": reps, "l2": "overwritten before every call",
            "match_ms": {"median": m_med, "min": m_min, "max": m_max},
            "align_ms": {"median": a_med, "min": a_min, "max": a_max},
            "align_launches": launches, "path_cells": cells, "dp_cells": int(sum(int(lq[p]) * int(doff[i + 1] - doff[i])
                                                                              for p, i in enumerate(o_idx.cpu().numpy()[:, 0]) if lq[p])),
            "align_dist_equals_match_dist": True}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--cases", default="config3,config4,long")
    ap.add_argument("--out", default=None, help="also write the lines as one JSON list here")
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("bench_align.py needs a CUDA device")
    gpu = gpu_name()
    lines = []
    for name in args.cases.split(","):
        r = run_case(name, args.reps, gpu)
        print(json.dumps(r), flush=True)
        lines.append(r)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(lines, f, indent=1)


if __name__ == "__main__":
    main()
