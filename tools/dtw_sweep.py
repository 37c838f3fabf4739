"""Development sweep: DTW match throughput for a synthetic dictionary x query batch (device-resident).

  python tools/dtw_sweep.py [ND] [NQ] [dtw|cos] [FIRST_STAGE]

FIRST_STAGE is ss_dict_set_scan's argument: 0 = packed-half tensor-core scan (default), 1 = fp32-DP tensor-core scan,
2 = fp32 CUDA-core scan, 3 = packed-half scan without its second chance."""
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from soundsym_b200 import api, synth  # noqa: E402
from soundsym_b200._lib import SS_DTW, SS_COSINE_REF  # noqa: E402

nd = int(sys.argv[1]) if len(sys.argv) > 1 else 10000
nq = int(sys.argv[2]) if len(sys.argv) > 2 else 1000
mode = SS_COSINE_REF if (len(sys.argv) > 3 and sys.argv[3] == "cos") else SS_DTW
first_stage = int(sys.argv[4]) if len(sys.argv) > 4 else 0
k = 1
ctx = api.Context(0)
t = time.time()
d, doff = synth.segments(nd, 13, seed=1234)
q, qoff = synth.segments(nq, 13, seed=5678)
print("gen %.1fs" % (time.time() - t), flush=True)
dev = api.DeviceDictionary(ctx, d, doff)
dev.set_scan(first_stage)
qs = api.DeviceQueries(ctx, q, qoff)
oi = torch.empty((nq, k), dtype=torch.int32, device="cuda")
od = torch.empty((nq, k), dtype=torch.float64, device="cuda")
stream = torch.cuda.ExternalStream(ctx.stream)
cells = int(doff[-1]) * int(qoff[-1])


def run():
    ctx.check(ctx.lib.ss_dict_match_dev(dev.h, qs.h, mode, None, k, oi.data_ptr(), od.data_ptr()))


for it in range(2):
    run()
ctx.sync()
with torch.cuda.stream(stream):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    n = 3
    for it in range(n):
        run()
    e1.record(stream)
ctx.sync()
ms = e0.elapsed_time(e1) / n
work = dev.last_work
print("first_stage=%d scan_kind=%d scan_ms=%.3f mode=%d nd=%d nq=%d: %.3f ms/step, %.3e work-units/s (work %.3e, cells %.3e), uncertified %d" %
      (first_stage, dev.last_scan_kind, float(ctx.lib.ss_dict_last_scan_ms(dev.h)), mode, nd, nq, ms, work / (ms * 1e-3), work, cells,
       dev.last_uncertified if mode == SS_DTW else 0), "tc_fallback", dev.last_tc_fallback)

# result fingerprint: identical for every first stage (indices are the f64 argmin, distances f64-rescored)
import hashlib  # noqa: E402
ctx.sync()
print("fingerprint idx=%s dist=%s exhaustive=%d" % (hashlib.sha1(oi.cpu().numpy().tobytes()).hexdigest()[:16],
                                                  hashlib.sha1(od.cpu().numpy().tobytes()).hexdigest()[:16], dev.last_exhaustive))
