#!/usr/bin/env python
"""bench.py — benchmarks of the soundsym hot path on B200 (contract in the build brief, section 4).

Default (what the driver runs) = the headline: BASELINE.json's metric "DTW cell-updates/s and queries/s, 100k-segment
dictionary, on 1/2/4/8 B200" on config 4 (SURVEY.md §8d): synthetic dictionary of 100 000 segments x 10 000 query segments,
13-coefficient MFCC frames, lengths ~ U{4..32}; a STEP = one match of the whole query batch against the whole dictionary
(top-1, SS_DTW). With N GPUs the dictionary is partitioned into N contiguous shards (balanced by frames), the exchange
(query all-gather over NVLink, one ncclAllGather of the per-shard top-k, merge) runs INSIDE the library
(ss_dict_match_sharded*)  ->  "scaling": "strong". torch.distributed is only used for the barrier, for shipping the 128-byte
communicator id and for the max-over-ranks of the timings.

  value      cells/s with the queries' f64 MFCCs already in HBM: layout kernel + tensor-core scan + merge + f64 refine
             (+ exchange for N > 1), CUDA events on the library's stream around the K steps, max over ranks. The L2 flush
             (a 256 MB fill) at the start of every step is INSIDE the bracket.
  e2e        the same through the reference-facing call ss_dict_match / ss_dict_match_sharded with pinned HOST buffers:
             H2D of the queries and D2H of the results inside the timed region, every step.
  roofline   the dominant kernel (k_dtw_scan_tc), timed live with CUDA events around its launch (ss_dict_last_scan_ms).
             It is bound by CUDA-core ISSUE of the DP recurrence (one FMNMX3 + one FADD per cell), not by HBM or the tensor
             pipe: achieved = useful DP cells / clk / SM, peak = the ALU pipe's FMNMX3 rate measured on this chip
             (tools/microbench_band2.cu: 63.9 lanes / clk / SM; the register-resident band alone reaches 47.3).
             The pairwise-streaming byte model of SURVEY.md §8d is kept as `effective_hbm_gbs` WITHOUT a fraction.
  cpu_baseline / --impl reference   the f64 CPU oracle ("port": the Rust reference cannot be built here) on a bounded
             sample of the same workload, on the box's host cores.

Other lines (not run by the driver; committed under profiles/bench/):  --config 3 (10k x 1k on 1 GPU, DTW and cosine-ref),
--config 2 (MFCC + partition of the Section_7_1 fixture, and the MFCC kernel on 1 h of audio against both of its roofs),
--config 5 (examples/reconstruction.rs on 1 h of synthetic audio, N GPUs).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

ND, NQ, C, K = 100000, 10000, 13, 1


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--nd", type=int, default=ND)
    ap.add_argument("--nq", type=int, default=NQ)
    ap.add_argument("--cpu-sample-queries", type=int, default=0, help="queries in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--config", type=int, default=4, choices=[2, 3, 4, 5], help="BASELINE.json config (default 4 = the headline)")
    ap.add_argument("--probe-queries", type=int, default=256, help="random queries checked against the f64 oracle after the run")
    ap.add_argument("--seconds", type=float, default=3600.0, help="configs 2 / 5: seconds of synthetic audio")
    ap.add_argument("--mode", default="dtw", choices=["dtw", "cosine"], help="config 5: matcher")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="configs 3 / 4: write the match result of the last timed step to DIR/*.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl != "ours" or args.config not in (3, 4)):
        ap.error("--dump-outputs is available for --impl ours with --config 3 or 4")
    return args


class ClockSampler:
    """samples SM clock, power and throttle reasons DURING the timed region through NVML (the same counters as the
    `nvidia-smi --query-gpu=clocks.sm,...,clocks_event_reasons.*` line of B200_PROFILING.md). An in-process NVML thread
    is used instead of an `nvidia-smi -lms` child because starting nvidia-smi next to a ~1 s timed region stalled the
    driver and inflated the measured step by 30-60 % (measured; see DESIGN.md "Measurement")."""

    def __init__(self, gpu_index, period_s=0.01):
        self.gpu, self.period = gpu_index, period_s
        self.rows, self.on, self.t, self.h = [], False, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            # NVML enumerates physical devices; honour CUDA_VISIBLE_DEVICES when it lists indices
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = gpu_index
            if vis:
                try:
                    phys = int(vis.split(",")[gpu_index])
                except Exception:
                    phys = gpu_index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    def _sample(self):
        nv = self.nv
        try:
            sm = nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)
            pw = nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0
            try:
                rs = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
            except Exception:
                rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
            self.rows.append((sm, pw, rs))
        except Exception:
            pass

    def _loop(self):
        # the timed region of an 8-GPU run is ~40 ms: sample every 10 ms while it is on
        while self.alive:
            if self.on:
                self._sample()
            time.sleep(self.period)

    def prepare(self):
        """start the thread (idle) before warm-up so that no start-up cost lands in the timed region"""
        if self.h is None:
            return
        self.alive = True
        self.t = threading.Thread(target=self._loop, daemon=True)
        self.t.start()

    def start(self):
        self.on = True

    def stop(self):
        if self.h is not None and self.on and not self.rows:
            self._sample()  # region shorter than one period: one reading while the last step is still in flight
        self.on = False
        self.alive = False
        if self.h is None or not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"], "samples": 0}
        nv = self.nv
        names = {"hw_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4)}
        reasons = sorted(k for k, bit in names.items() if any(r[2] & bit for r in self.rows))
        return {"sm_mhz": float(np.median([r[0] for r in self.rows])), "sm_max_mhz": float(self.max_sm), "reasons": reasons,
                "power_w_max": max(r[1] for r in self.rows), "samples": len(self.rows)}


def workload(nd, nq):
    from soundsym_b200 import synth
    d, doff = synth.segments(nd, C, seed=1234)
    q, qoff = synth.segments(nq, C, seed=5678)
    return d, doff, q, qoff


def shard_bounds(doff, n):
    """contiguous segment ranges balanced by frames (SURVEY.md §8e)."""
    total = int(doff[-1])
    cuts = [0]
    for r in range(1, n):
        cuts.append(int(np.searchsorted(doff, total * r // n, side="left")))
    cuts.append(len(doff) - 1)
    return cuts


def algorithmic_bytes(doff, qoff, s0, s1):
    """sum over (query, dict segment in [s0, s1)) of (Lq + Ld) * C * 4 B."""
    ld = int(doff[s1] - doff[s0])
    lq = int(qoff[-1])
    nq, nd = len(qoff) - 1, s1 - s0
    return (nd * lq + nq * ld) * C * 4


DUMP_BYTES = 64_000_000


def dump_outputs(out_dir, idx, dist):
    """Writes a match result as the caller of ss_dict_match_dev receives it, in float64: indices.npy (u32 segment indices,
    0xFFFFFFFF = empty slot) and distances.npy, both [queries, k], and query_ids.npy, the query each row belongs to.
    A result larger than DUMP_BYTES is cut to a fixed, seeded sample of queries, so that two builds run with the same
    arguments write the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    nq, k = idx.shape
    row_bytes = 8 * (2 * k + 1)
    rows = np.arange(nq)
    if nq * row_bytes > DUMP_BYTES - 3 * 4096:  # room for the three .npy headers
        rows = np.sort(np.random.default_rng(2026).choice(nq, size=(DUMP_BYTES - 3 * 4096) // row_bytes, replace=False))
    np.save(os.path.join(out_dir, "query_ids.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "indices.npy"), idx[rows].astype(np.float64))
    np.save(os.path.join(out_dir, "distances.npy"), dist[rows].astype(np.float64))


def cpu_sample(d, doff, q, qoff, nsample, threads):
    from oracle import oracle as O
    O.set_threads(threads)
    sub_off = qoff[: nsample + 1]
    sub = q[: int(sub_off[-1])]
    t0 = time.perf_counter()
    O.dtw_topk(d, doff, sub, sub_off, C, K)
    dt = time.perf_counter() - t0
    cells = int(doff[-1]) * int(sub_off[-1])
    return cells / dt, dt, cells


WORKLOADS = {
    4: "synthetic 100k-segment dictionary x 10k queries, C=13, L~U{4..32}, DTW top-1 (config 4)",
    3: "synthetic 10k-segment dictionary x 1k queries, C=13, L~U{4..32}, DTW top-1 (config 3)",
}
# measured on B200 by tools/microbench_band2.cu (profiles/r2_microbench_band2.log). Every DP cell needs one three-input min
# on the ALU pipe, which issues FMNMX3 (fp32: one cell) and VHMNMX (half2: two cells) at 63.9 lanes / clk / SM; the
# register-resident band alone (min + add per cell, costs already in registers) reaches 47.3 / 83.1 cells / clk / SM.
SCAN_KERNELS = {
    1: ("k_dtw_scan_h2 (tcgen05 fp16 cost matrix, F16 accumulator in TMEM + packed-half DP: VHMNMX + HADD2 per two cells)", 2 * 63.9, 83.1,
        "f16 (packed-half DP scan on f16 tensor-core costs; winners refined in f64)"),
    2: ("k_dtw_scan_tc (tcgen05 fp16 cost matrix, F32 accumulator in TMEM + fp32 DP: FMNMX3 + FADD per cell)", 63.9, 47.3,
        "f32 (DP scan; local costs from f16 tensor-core products accumulated in f32; winners refined in f64)"),
    3: ("k_dtw_scan (fp32 CUDA-core scan)", 63.9, 47.3, "f32 (winners refined in f64)"),
}


def config_dict(args):
    """the same object on both arms (the driver compares them): workload, sizes, and how the GPU arm treats L2"""
    std = (args.nd, args.nq) in ((ND, NQ), (10000, 1000))
    return {"workload": WORKLOADS.get(args.config, WORKLOADS[4]) if std else
            "synthetic %d-segment dictionary x %d queries, C=13, L~U{4..32}, DTW top-1" % (args.nd, args.nq),
            "nd": args.nd, "nq": args.nq, "ncoeffs": C, "k": K,
            "l2": "GPU arm: flushed, a 256 MB buffer is overwritten at the start of every timed step (inside the bracket)"}


def run_reference(args):
    """the reference arm: the CPU path (oracle port; the Rust crate cannot be built in this image) with all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import oracle as O
    d, doff, q, qoff = workload(args.nd, args.nq)
    threads = O.hardware_threads()
    nsample = args.cpu_sample_queries or max(threads, 32)
    # calibrate so one step is a few seconds
    rate, dt, _ = cpu_sample(d, doff, q, qoff, min(nsample, 8), threads)
    for _ in range(args.warmup):
        pass  # CPU path has no warm-up state beyond the calibration pass above
    times, cells = [], 0
    for _ in range(args.steps):
        r, dt, cells = cpu_sample(d, doff, q, qoff, nsample, threads)
        times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = cells / (ms * 1e-3)
    sample = "%d of %d queries x full %d-segment dictionary per step (%.3e cells), f64 oracle port, %d threads" % (
        nsample, args.nq, args.nd, cells, threads)
    line = {"impl": "reference", "metric": "dtw_cell_updates_per_s", "value": value, "unit": "cells/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": config_dict(args),
            "queries_per_s": nsample / (ms * 1e-3),
            "cpu_baseline": {"value": value, "unit": "cells/s", "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": "cells/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def run_match(args):
    import ctypes as CT
    import torch
    import torch.distributed as dist
    from soundsym_b200 import api
    from soundsym_b200._lib import SS_DTW

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    n_gpus = world

    d, doff, q, qoff = workload(args.nd, args.nq)
    nq = len(qoff) - 1
    ctx = api.Context(local)
    lib = ctx.lib
    cuts = api.shard_bounds(doff, world)
    assert cuts == shard_bounds(doff, world)
    s0, s1 = cuts[rank], cuts[rank + 1]
    stream = torch.cuda.ExternalStream(ctx.stream, device=torch.device("cuda", local))
    shard = api.DeviceDictionary(ctx, d, doff[s0:s1 + 1], C, index_base=s0)
    total_cells = int(doff[-1]) * int(qoff[-1])
    shard_cells = int(doff[s1] - doff[s0]) * int(qoff[-1])

    comm = None
    if world > 1:
        # the library owns the NCCL communicator of the data path; torch only carries its 128-byte id to the other ranks
        idt = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            idt.copy_(torch.frombuffer(bytearray(api.Comm.unique_id()), dtype=torch.uint8))
        dist.broadcast(idt, 0)
        comm = api.Comm(ctx, world, rank, idt.cpu().numpy().tobytes())

    # device-resident queries + outputs
    if world > 1:
        qh = CT.c_void_p()
        ctx.check(lib.ss_queries_create_sharded(comm.h, q.ctypes.data, qoff.ctypes.data, nq, C, CT.byref(qh)))
    else:
        qdev = api.DeviceQueries(ctx, q, qoff, C)
        qh = qdev.h
    o_idx = torch.empty((nq, K), dtype=torch.int32, device="cuda")
    o_dist = torch.empty((nq, K), dtype=torch.float64, device="cuda")
    # pinned host buffers for the e2e leg
    hq = torch.from_numpy(q).pin_memory()
    hqoff = torch.from_numpy(qoff.astype(np.int64)).pin_memory()
    h_idx = torch.empty((nq, K), dtype=torch.int32).pin_memory()
    h_dist = torch.empty((nq, K), dtype=torch.float64).pin_memory()

    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")  # > 126 MB L2

    def step_resident():
        flush.zero_()
        ctx.check(lib.ss_queries_invalidate(qh))  # the layout kernel runs inside the step
        if world > 1:
            ctx.check(lib.ss_dict_match_sharded_dev(shard.h, comm.h, qh, SS_DTW, None, K, o_idx.data_ptr(), o_dist.data_ptr()))
        else:
            ctx.check(lib.ss_dict_match_dev(shard.h, qh, SS_DTW, None, K, o_idx.data_ptr(), o_dist.data_ptr()))

    def step_e2e():
        flush.zero_()
        # the reference-facing call: HOST buffers in, HOST buffers out (H2D + D2H inside; 1/N of the query bytes per GPU)
        if world > 1:
            ctx.check(lib.ss_dict_match_sharded(shard.h, comm.h, hq.data_ptr(), hqoff.data_ptr(), nq, SS_DTW, None, K, h_idx.data_ptr(), h_dist.data_ptr()))
        else:
            ctx.check(lib.ss_dict_match(shard.h, hq.data_ptr(), hqoff.data_ptr(), nq, SS_DTW, None, K, h_idx.data_ptr(), h_dist.data_ptr()))

    def barrier():
        ctx.sync()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record(stream)
        for _ in range(steps):
            fn()
        ctx.check(lib.ss_dict_match_finish(shard.h))  # the last step's fallback decision belongs to the step
        e1.record(stream)
        barrier()
        wall = (time.perf_counter() - t0) * 1e3
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms, wall], dtype=torch.float64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms, wall = float(t[0]), float(t[1])
        return ms / steps, wall / steps

    with torch.cuda.stream(stream):
        sampler = ClockSampler(local)
        if rank == 0 and not os.environ.get("BENCH_NO_SAMPLER"):
            sampler.prepare()
        for _ in range(max(args.warmup, 3)):
            step_resident()
        sampler.start()
        launches0 = ctx.launches
        ms_step, _ = timed(step_resident, args.steps)
        launches = ctx.launches - launches0
        scan_ms = float(lib.ss_dict_last_scan_ms(shard.h))
        tc_fallback, exhaustive, uncert = shard.last_tc_fallback, shard.last_exhaustive, shard.last_uncertified
        clocks = sampler.stop() if rank == 0 else None
        if args.dump_outputs and rank == 0:  # every rank holds the merged result of the last timed step
            dump_outputs(args.dump_outputs, o_idx.cpu().numpy().view(np.uint32), o_dist.cpu().numpy())
        for _ in range(2):
            step_e2e()
        # e2e blocks on the host every step (the call returns results in host memory): wall clock == device time here
        _, ms_e2e = timed(step_e2e, args.steps)
        # one more untimed step with the scan's per-CTA timeline hook on (SS_DTW_H2_TIMELINE): clock64 cycles over globaltimer ns
        # of every CTA's DP phase = the SM clock the scan actually runs at. NVML reports 1 965 MHz under this load while the
        # SMs count 1 842 MHz (15/16 of it); the ceilings of the roofline block are in clock64 cycles (tools/microbench_band2.cu),
        # so the achieved rate has to be, too.
        # (one GPU only: the N > 1 lines keep NVML's clock - the hook synchronises inside the match, between scan and exchange)
        sm_mhz_kernel = None
        tl_path = os.path.join(tempfile.gettempdir(), "ss_h2_timeline_%d_%d.txt" % (os.getpid(), rank))
        if world == 1:
            os.environ["SS_DTW_H2_TIMELINE"] = tl_path
            try:
                step_resident()
                ctx.check(lib.ss_dict_match_finish(shard.h))
                barrier()
            finally:
                del os.environ["SS_DTW_H2_TIMELINE"]
        if os.path.exists(tl_path):
            try:
                tl = np.loadtxt(tl_path, dtype=np.int64, comments="#", ndmin=2)
                tl = tl[(tl[:, 1] > 0) & (tl[:, 3] > tl[:, 2])] if tl.shape[1] >= 12 else tl[:0]
                if len(tl):
                    sm_mhz_kernel = float(np.median(tl[:, 10] / (tl[:, 3] - tl[:, 2])) * 1e3)
            finally:
                os.remove(tl_path)
    res_idx = o_idx.cpu().numpy().view(np.uint32)
    res_dist = o_dist.cpu().numpy()
    assert np.array_equal(res_idx, h_idx.numpy().view(np.uint32)) and np.array_equal(res_dist, h_dist.numpy()), "e2e and resident paths disagree"
    assert uncert == 0, "%d queries left uncertified" % uncert

    # correctness gate against the oracle on a random sample of queries (outside every timed region); a wrong match must not
    # produce a normal bench line
    probe = None
    if rank == 0 and not args.no_cpu_baseline:
        from oracle import oracle as O
        O.set_threads(O.hardware_threads())
        ids = np.sort(np.random.default_rng(2026).choice(nq, size=min(args.probe_queries, nq), replace=False))
        rows = np.concatenate([np.arange(int(qoff[i]), int(qoff[i + 1])) for i in ids])
        so = np.zeros(len(ids) + 1, dtype=np.uint64)
        so[1:] = np.cumsum((qoff[1:] - qoff[:-1])[ids])
        oi, od = O.dtw_topk(d, doff, np.ascontiguousarray(q[rows]), so, C, K)
        ok = bool(np.array_equal(oi, res_idx[ids]) and np.allclose(od, res_dist[ids], rtol=1e-12, atol=0))
        assert ok, "GPU match differs from the f64 oracle on the probe sample"
        probe = {"queries": int(len(ids)), "indices_equal": True, "max_rel_dist_err": float(np.max(np.abs(od - res_dist[ids]) / od))}

    if rank == 0:
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        if os.path.exists(peaks_path):
            hbm_peak, hbm_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        else:
            hbm_peak, hbm_src = 6650.0, "fallback (B200_PROFILING.md)"
        alg = algorithmic_bytes(doff, qoff, s0, s1)
        kind = shard.last_scan_kind
        scan_kernel, alu_peak, band_ceiling, dtype = SCAN_KERNELS.get(kind, SCAN_KERNELS[3])
        traffic, traffic_src = None, None
        tp = os.path.join(ROOT, "profiles", "dtw_scan_traffic.json")
        if os.path.exists(tp) and world == 1 and args.nd == ND and args.nq == NQ:
            tj = json.load(open(tp)).get({1: "h2", 2: "tc"}.get(kind, "fp32"), {})
            traffic, traffic_src = tj.get("dram_bytes_per_launch"), tj.get("source")
        if clocks is not None:
            clocks["sm_mhz_in_kernel"] = sm_mhz_kernel
        sm_mhz = sm_mhz_kernel or ((clocks or {}).get("sm_mhz") or 1965.0)
        sms = 148.0
        cells_clk_sm = shard_cells / (scan_ms * 1e-3) / sms / (sm_mhz * 1e6) if scan_ms > 0 else None
        cpu = None
        if not args.no_cpu_baseline:
            from oracle import oracle as O
            threads = O.hardware_threads()
            nsample = args.cpu_sample_queries or max(4 * threads, 64)
            rate, dt, cells = cpu_sample(d, doff, q, qoff, nsample, threads)
            cpu = {"value": rate, "unit": "cells/s", "cores": threads, "kind": "port",
                   "sample": "%d of %d queries x full %d-segment dictionary (%.3e cells, %.1f s), scalar f64 oracle port" % (nsample, nq, args.nd, cells, dt)}
        line = {
            "metric": "dtw_cell_updates_per_s", "value": total_cells / (ms_step * 1e-3), "unit": "cells/s", "n_gpus": n_gpus,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None,
            "dtype": dtype, "data": "synthetic",
            "config": config_dict(args),
            "parallelism": "dictionary sharded x%d inside the library: queries 1/N per GPU over PCIe + NVLink all-gather, one ncclAllGather of the "
                           "per-shard top-k, merge on every rank" % world,
            "resident_per_gpu_mb": {"fp16_tiles": int(doff[s1] - doff[s0]) * 32 * 1.4 / 1e6, "f64_frames": int(doff[s1] - doff[s0]) * C * 8 / 1e6},
            "queries_per_s": nq / (ms_step * 1e-3),
            "e2e": {"value": total_cells / (ms_e2e * 1e-3), "unit": "cells/s", "ms_per_step": ms_e2e,
                    "h2d_bytes_per_step": int((q.nbytes + world - 1) // world + qoff.nbytes), "d2h_bytes_per_step": int(nq * K * 12),
                    "queries_per_s": nq / (ms_e2e * 1e-3)},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "issue", "kernel": scan_kernel, "achieved": cells_clk_sm, "peak": alu_peak,
                         "unit": "DP cells/clk/SM", "frac": (cells_clk_sm / alu_peak) if cells_clk_sm else None,
                         "traffic": traffic, "traffic_source": traffic_src,
                         "peak_source": "measured on B200: every DP cell needs one three-input min on the ALU pipe, which issues FMNMX3 (1 cell) / VHMNMX "
                                        "(2 cells) at 63.9 lanes/clk/SM (tools/microbench_band2.cu, profiles/r2_microbench_band2.log) per clock64 cycle; SM clock = "
                                        "clocks.sm_mhz_in_kernel: clock64 cycles / globaltimer ns over the DP phase of every CTA of one untimed step "
                                        "(NVML's sm clock when that is unavailable)",
                         "band_ceiling": band_ceiling,
                         "frac_of_band_ceiling": (cells_clk_sm / band_ceiling) if cells_clk_sm else None,
                         "kernel_ms": scan_ms, "kernel_share_of_step": scan_ms / ms_step if ms_step else None,
                         "cells_per_s_kernel": shard_cells / (scan_ms * 1e-3) if scan_ms > 0 else None,
                         "effective_hbm_gbs": alg / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else None, "hbm_peak_gbs": hbm_peak, "hbm_peak_source": hbm_src,
                         "algorithmic_bytes_per_launch": alg,
                         "note": "effective_hbm_gbs is the pairwise-streaming model of SURVEY.md 8d (bytes the CPU path streams per pair): operands stay "
                                 "on chip (one dictionary tile serves 128 queries from shared memory / TMEM), so it is NOT a roofline fraction; "
                                 "`traffic` is the physical DRAM traffic of one launch from ncu"},
            "cpu_baseline": cpu,
            "uncertified_queries": int(uncert), "tc_fallback_queries": int(tc_fallback), "exhaustive_queries": int(exhaustive),
            "oracle_probe": probe,
        }
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        comm.close()
        dist.destroy_process_group()


def main():
    args = parse()
    if args.config == 3 and (args.nd, args.nq) == (ND, NQ):
        args.nd, args.nq = 10000, 1000
    if args.impl == "reference":
        return run_reference(args)
    if args.config in (3, 4):
        return run_match(args)
    from tools import bench_configs
    return bench_configs.run(args)


if __name__ == "__main__":
    main()
