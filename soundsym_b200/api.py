"""Host-side mirror of the reference crate's public API for the hot path, on top of the C ABI.

Rust is not installed in this image, so instead of the `extern "C"` shim shown in INTEGRATION.md this module plays the
host role: same type names, method names, argument meaning and error behaviour as src/lib.rs / src/sound.rs, so the
parity tests read like the reference's own tests. All numerics happen in libsoundsym_b200.so on the GPU; this file
only owns host buffers (numpy f64, like the reference's Vec<f64>) and calls through ctypes.

    Sound::from_samples / from_path / push_samples / max_power / mfccs / mean_mfccs / num_frames   src/sound.rs:92-212
    SoundDictionary::{new, from_segments, add_segments, match_sound, at_distance}                  src/sound.rs:290-370
    SoundSequence::{new, clone_from_dictionary, to_sound, morph_to, from_distances, distances}     src/sound.rs:390-483
    Partitioner::{new, depth, threshold, train(model), partition, partition_other}                 src/lib.rs:67-151
"""
import ctypes as C
import struct

import numpy as np

from . import _lib
from ._lib import SS_COSINE_REF, SS_DTW, SS_DTW_TARGET, SoundsymError

NCOEFFS, NCLUSTERS, HOP, BIN = 12, 26, 256, 1024  # src/lib.rs:22-25


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


class Context:
    """ss_ctx: one device, one stream. Not thread-safe (like the reference, which is single-threaded)."""

    def __init__(self, device=0):
        self.lib = _lib.load()
        h = C.c_void_p()
        rc = self.lib.ss_ctx_create(int(device), C.byref(h))
        if rc != 0:
            raise SoundsymError(rc, self.lib.ss_last_error(None).decode())
        self.h = h
        self.device = int(device)

    def close(self):
        if getattr(self, "h", None):
            self.lib.ss_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, rc):
        if rc != 0:
            raise SoundsymError(rc, self.lib.ss_last_error(self.h).decode())

    @property
    def stream(self):
        return self.lib.ss_ctx_stream(self.h)

    def sync(self):
        self.check(self.lib.ss_ctx_sync(self.h))

    @property
    def launches(self):
        return int(self.lib.ss_ctx_launch_count(self.h))

    # ---- MFCC subsystem ------------------------------------------------------------------------------------------
    def decode_pcm(self, pcm, bits):
        pcm = np.ascontiguousarray(pcm, dtype=np.int32)
        out = np.empty(pcm.shape[0], dtype=np.float64)
        self.check(self.lib.ss_decode_pcm(self.h, _ptr(pcm), pcm.shape[0], int(bits), _ptr(out)))
        return out

    def analyze(self, samples, sample_rate=44100.0, ncoeffs=NCOEFFS):
        """Sound::from_samples' three analyses in one call -> (mfcc [frames, C], max_power, mean_mfccs [C])."""
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        n = samples.shape[0]
        frames = C.c_size_t()
        self.check(self.lib.ss_frame_count(n, C.byref(frames)))
        mfcc = np.empty((frames.value, ncoeffs), dtype=np.float64)
        mean = np.empty(ncoeffs, dtype=np.float64)
        mp = C.c_double()
        self.check(self.lib.ss_sound_analyze(self.h, _ptr(samples), n, float(sample_rate), int(ncoeffs), _ptr(mfcc),
                                             C.byref(frames), C.byref(mp), _ptr(mean)))
        return mfcc, float(mp.value), mean

    def analyze_pcm(self, pcm, bits, sample_rate=44100.0, ncoeffs=NCOEFFS):
        """Sound::from_path's decode + the three analyses with integer PCM crossing PCIe (2 or 4 bytes per sample)
        -> (samples f64, mfcc, max_power, mean_mfccs)."""
        pcm = np.ascontiguousarray(pcm, dtype=np.int16 if bits == 16 else np.int32)
        n = pcm.shape[0]
        frames = C.c_size_t()
        self.check(self.lib.ss_frame_count(n, C.byref(frames)))
        samples = np.empty(n, dtype=np.float64)
        mfcc = np.empty((frames.value, ncoeffs), dtype=np.float64)
        mean = np.empty(ncoeffs, dtype=np.float64)
        mp = C.c_double()
        self.check(self.lib.ss_sound_analyze_pcm(self.h, _ptr(pcm), n, int(bits), float(sample_rate), int(ncoeffs), _ptr(samples), _ptr(mfcc),
                                                 C.byref(frames), C.byref(mp), _ptr(mean)))
        return samples, mfcc, float(mp.value), mean

    def analyze_batch(self, samples, sample_offsets, sample_rate=44100.0, ncoeffs=NCOEFFS):
        """Many sounds back to back, analysed in one upload / one MFCC launch (ss_sound_analyze_batch)
        -> (mfcc [sum frames, C], frame_offsets [n + 1], max_power [n], mean_mfccs [n, C])."""
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        off = np.ascontiguousarray(sample_offsets, dtype=np.uint64)
        n = off.shape[0] - 1
        foff = np.zeros(n + 1, dtype=np.uint64)
        frames = 0
        for i in range(n):
            ln = int(off[i + 1]) - int(off[i])
            frames += (ln - BIN) // HOP + 1 if ln >= BIN else 0
        mfcc = np.empty((frames, ncoeffs), dtype=np.float64)
        mp = np.zeros(n, dtype=np.float64)
        mean = np.empty((n, ncoeffs), dtype=np.float64)
        self.check(self.lib.ss_sound_analyze_batch(self.h, _ptr(samples), _ptr(off), n, float(sample_rate), int(ncoeffs), _ptr(mfcc),
                                                   _ptr(foff), _ptr(mp), _ptr(mean)))
        return mfcc, foff, mp, mean

    def max_power_batch(self, samples, sample_offsets):
        """analyze_max_power (src/sound.rs:244-256) of many cuts of one buffer in one launch -> f64 [ncuts]."""
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        off = np.ascontiguousarray(sample_offsets, dtype=np.uint64)
        n = off.shape[0] - 1
        mp = np.zeros(n, dtype=np.float64)
        foff = np.zeros(n + 1, dtype=np.uint64)
        if n:
            self.check(self.lib.ss_sound_analyze_batch(self.h, _ptr(samples), _ptr(off), n, 44100.0, NCOEFFS, None, _ptr(foff), _ptr(mp), None))
        return mp

    def mfcc(self, samples, sample_rate=44100.0, ncoeffs=NCOEFFS):
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        frames = C.c_size_t()
        self.check(self.lib.ss_frame_count(samples.shape[0], C.byref(frames)))
        out = np.empty((frames.value, ncoeffs), dtype=np.float64)
        self.check(self.lib.ss_mfcc(self.h, _ptr(samples), samples.shape[0], float(sample_rate), int(ncoeffs), _ptr(out), C.byref(frames)))
        return out

    def max_power(self, samples):
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        out = C.c_double()
        self.check(self.lib.ss_max_power(self.h, _ptr(samples), samples.shape[0], C.byref(out)))
        return float(out.value)

    # ---- segmentation subsystem ------------------------------------------------------------------------------------
    @staticmethod
    def _gmm(model):
        if model is None:
            return None, None
        means, covs, weights = (np.ascontiguousarray(m, dtype=np.float64) for m in model)
        g = _lib.ss_gmm(int(means.shape[0]), int(means.shape[1]), means.ctypes.data, covs.ctypes.data, weights.ctypes.data)
        return g, (means, covs, weights)

    def symbols(self, mfcc, model, want_posteriors=False):
        mfcc = np.ascontiguousarray(mfcc, dtype=np.float64)
        g, keep = self._gmm(model)
        out = np.empty(mfcc.shape[0], dtype=np.uint8)
        post = np.empty((mfcc.shape[0], keep[0].shape[0]), dtype=np.float64) if (want_posteriors and keep) else None
        self.check(self.lib.ss_symbols(self.h, _ptr(mfcc), mfcc.shape[0], C.byref(g) if g else None, _ptr(out), _ptr(post)))
        return (out, post) if want_posteriors else out

    def gmm_train(self, mfcc, ncomp=NCLUSTERS, iters=5, reg=0.1, seed=0):
        """train_model (src/lib.rs:44-54) on the GPU; retries with seed+1, ... like the reference's `while let Err` loop."""
        mfcc = np.ascontiguousarray(mfcc, dtype=np.float64)
        c = mfcc.shape[1]
        means, covs, weights = np.empty((ncomp, c)), np.empty((ncomp, c, c)), np.empty(ncomp)
        err = None
        for attempt in range(64):
            rc = self.lib.ss_gmm_train(self.h, _ptr(mfcc), mfcc.shape[0], c, int(ncomp), int(iters), float(reg), int(seed) + attempt,
                                       _ptr(means), _ptr(covs), _ptr(weights))
            if rc == 0:
                return means, covs, weights
            err = SoundsymError(rc, self.lib.ss_last_error(self.h).decode())
            if rc != _lib.SS_ERR_INVALID or "EM failed" not in err.message:
                break
        raise err

    def vote_split(self, symbols, depth, threshold):
        symbols = np.ascontiguousarray(symbols, dtype=np.uint8)
        n = symbols.shape[0]
        votes = np.zeros(n + 1, dtype=np.uint32)
        lens = np.empty(max(n, 1), dtype=np.uint64)
        nseg = C.c_size_t()
        self.check(self.lib.ss_vote_split(self.h, _ptr(symbols), n, int(depth), int(threshold), _ptr(votes), _ptr(lens), C.byref(nseg)))
        return votes, lens[: nseg.value].copy()

    def partition(self, mfcc, model, depth, threshold):
        mfcc = np.ascontiguousarray(mfcc, dtype=np.float64)
        g, keep = self._gmm(model)
        lens = np.empty(max(mfcc.shape[0], 1), dtype=np.uint64)
        nseg = C.c_size_t()
        self.check(self.lib.ss_partition(self.h, _ptr(mfcc), mfcc.shape[0], C.byref(g) if g else None, int(depth), int(threshold),
                                         _ptr(lens), C.byref(nseg)))
        return lens[: nseg.value].copy()

    # ---- matcher subsystem -----------------------------------------------------------------------------------------
    def resynth(self, dict_samples, dict_sample_offsets, match_idx, target_lens):
        ds = np.ascontiguousarray(dict_samples, dtype=np.float64)
        do = np.ascontiguousarray(dict_sample_offsets, dtype=np.uint64)
        mi = np.ascontiguousarray(match_idx, dtype=np.uint32)
        tl = np.ascontiguousarray(target_lens, dtype=np.uint64)
        out = np.empty(int(tl.sum()), dtype=np.float64)
        self.check(self.lib.ss_resynth(self.h, _ptr(ds), _ptr(do), do.shape[0] - 1, _ptr(mi), _ptr(tl), mi.shape[0], _ptr(out)))
        return out

    def resynth_warped(self, dict_samples, dict_sample_offsets, match_idx, paths, path_offsets, target_lens):
        """ss_resynth_warped: resynth along the DTW warping paths (A11, DESIGN.md §3.5). paths: uint32 [cells, 2] of (i, j),
        path t = paths[path_offsets[t]:path_offsets[t + 1]] (what DeviceDictionary.align returns, concatenated)."""
        ds = np.ascontiguousarray(dict_samples, dtype=np.float64)
        do = np.ascontiguousarray(dict_sample_offsets, dtype=np.uint64)
        mi = np.ascontiguousarray(match_idx, dtype=np.uint32)
        pa = np.ascontiguousarray(paths, dtype=np.uint32).reshape(-1, 2)
        po = np.ascontiguousarray(path_offsets, dtype=np.uint64)
        tl = np.ascontiguousarray(target_lens, dtype=np.uint64)
        if po.shape[0] != mi.shape[0] + 1 or tl.shape[0] != mi.shape[0]:
            raise SoundsymError(_lib.SS_ERR_INVALID, "one path and one target length per segment (%d indices, %d path offsets, %d lengths)"
                                % (mi.shape[0], po.shape[0], tl.shape[0]))
        out = np.empty(int(tl.sum()), dtype=np.float64)
        self.check(self.lib.ss_resynth_warped(self.h, _ptr(ds), _ptr(do), do.shape[0] - 1, _ptr(mi), _ptr(pa), _ptr(po), _ptr(tl), mi.shape[0],
                                              _ptr(out)))
        return out

    def sequence_distances(self, mean_rows):
        m = np.ascontiguousarray(mean_rows, dtype=np.float64)
        out = np.empty(max(m.shape[0] - 1, 0), dtype=np.float64)
        self.check(self.lib.ss_sequence_distances(self.h, _ptr(m), m.shape[0], m.shape[1], _ptr(out)))
        return out


class DeviceDictionary:
    """ss_dict: a dictionary (or one shard) resident in HBM. Offsets are in FRAMES."""

    def __init__(self, ctx, mfcc_flat, frame_offsets, ncoeffs=None, index_base=0):
        self.ctx = ctx
        mfcc_flat = np.ascontiguousarray(mfcc_flat, dtype=np.float64)
        off = np.ascontiguousarray(frame_offsets, dtype=np.uint64)
        if ncoeffs is None:
            ncoeffs = mfcc_flat.shape[1]
        self.ncoeffs = int(ncoeffs)
        self.max_len = int(np.max(np.diff(off))) if off.shape[0] > 1 else 0
        h = C.c_void_p()
        ctx.check(ctx.lib.ss_dict_create(ctx.h, _ptr(mfcc_flat), _ptr(off), off.shape[0] - 1, self.ncoeffs, int(index_base), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.lib.ss_dict_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self.ctx.lib.ss_dict_len(self.h))

    def match(self, q_flat, q_frame_offsets, mode=SS_DTW, k=1, targets=None):
        """ss_dict_match with HOST buffers -> (idx u32 [nq, k], dist f64 [nq, k])."""
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        nq = qo.shape[0] - 1
        idx = np.empty((nq, k), dtype=np.uint32)
        dist = np.empty((nq, k), dtype=np.float64)
        t = np.ascontiguousarray(targets, dtype=np.float64) if targets is not None else None
        self.ctx.check(self.ctx.lib.ss_dict_match(self.h, _ptr(q), _ptr(qo), nq, int(mode), _ptr(t), int(k), _ptr(idx), _ptr(dist)))
        return idx, dist

    def walk(self, start_mfcc, distances):
        """ss_dict_walk: SoundSequence::from_distances for SS_COSINE_REF on the device -> (idx u32 [n], dist f64 [n]); step t
        matches the segment step t - 1 returned (step 0: start_mfcc, frames x ncoeffs) at target distances[t]."""
        s = np.ascontiguousarray(start_mfcc, dtype=np.float64).reshape(-1, self.ncoeffs)
        t = np.ascontiguousarray(distances, dtype=np.float64).reshape(-1)
        n = t.shape[0]
        idx = np.empty(n, dtype=np.uint32)
        dist = np.empty(n, dtype=np.float64)
        self.ctx.check(self.ctx.lib.ss_dict_walk(self.h, _ptr(s), s.shape[0], _ptr(t), n, _ptr(idx), _ptr(dist)))
        return idx, dist

    def walk_dtw(self, start_mfcc, distances=None, nsteps=None):
        """ss_dict_walk_dtw: SoundSequence::from_distances for SS_DTW_TARGET on the device -> (idx u32 [n], dist f64 [n]); step t
        matches the segment step t - 1 returned (step 0: start_mfcc) at target distances[t]. distances=None: t = 0 at each of
        `nsteps` steps (SS_DTW's chain). A step with no result gives (0xFFFFFFFF, inf), and so does every later one."""
        s = np.ascontiguousarray(start_mfcc, dtype=np.float64).reshape(-1, self.ncoeffs)
        t = None if distances is None else np.ascontiguousarray(distances, dtype=np.float64).reshape(-1)
        n = t.shape[0] if t is not None else int(nsteps or 0)
        idx = np.empty(n, dtype=np.uint32)
        dist = np.empty(n, dtype=np.float64)
        self.ctx.check(self.ctx.lib.ss_dict_walk_dtw(self.h, _ptr(s), s.shape[0], _ptr(t), n, _ptr(idx), _ptr(dist)))
        return idx, dist

    def align(self, q_flat, q_frame_offsets, seg_idx):
        """ss_dict_align: the DTW warping path (DESIGN.md §3.1e) of query p against segment seg_idx[p] (an index as
        match reports it; 0xFFFFFFFF -> empty path, inf) -> (paths: list of uint32 [n, 2] arrays of (i, j), dist f64 [nq])."""
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        seg = np.ascontiguousarray(seg_idx, dtype=np.uint32).reshape(-1)
        nq = qo.shape[0] - 1
        if seg.shape[0] != nq:
            raise SoundsymError(_lib.SS_ERR_INVALID, "one segment index per query (%d queries, %d indices)" % (nq, seg.shape[0]))
        lq = np.diff(qo).astype(np.int64)
        cap = int(np.sum(lq[lq > 0] + max(self.max_len, 1) - 1))  # >= the sum of Lq + Ld - 1 the call requires
        path = np.empty((max(cap, 1), 2), dtype=np.uint32)
        poff = np.empty(nq + 1, dtype=np.uint64)
        dist = np.empty(nq, dtype=np.float64)
        self.ctx.check(self.ctx.lib.ss_dict_align(self.h, _ptr(q), _ptr(qo), nq, _ptr(seg), _ptr(path), cap, _ptr(poff), _ptr(dist)))
        return [path[int(poff[p]):int(poff[p + 1])].copy() for p in range(nq)], dist

    def locate(self, q_flat, q_frame_offsets, k=1):
        """ss_dict_locate: subsequence DTW (spec A12, DESIGN.md §3.1g), where inside a segment each query fits best -> (idx u32
        [nq, k], start u32 [nq, k], end u32 [nq, k], cost f64 [nq, k]); start / end are frames of the segment, end inclusive,
        cost is unnormalised. The k best (cost, index) hits, one per segment; unfilled slots (0xFFFFFFFF, 0xFFFFFFFF,
        0xFFFFFFFF, inf). The band does not apply."""
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        nq = qo.shape[0] - 1
        idx, start, end = (np.empty((nq, k), dtype=np.uint32) for _ in range(3))
        cost = np.empty((nq, k), dtype=np.float64)
        self.ctx.check(self.ctx.lib.ss_dict_locate(self.h, _ptr(q), _ptr(qo), nq, int(k), _ptr(idx), _ptr(start), _ptr(end), _ptr(cost)))
        return idx, start, end, cost

    def debug_tc_scan(self, q_flat, q_frame_offsets):
        """ss_dict_debug_tc_scan: raw tensor-core scan distance of every (query, segment) pair -> (scan f32 [nq, nseg],
        mean frame f64 [16], norm scale)."""
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        nq = qo.shape[0] - 1
        scan = np.empty((nq, len(self)), dtype=np.float32)
        mu = np.zeros(16, dtype=np.float64)
        scale = C.c_float(0.0)
        self.ctx.check(self.ctx.lib.ss_dict_debug_tc_scan(self.h, _ptr(q), _ptr(qo), nq, _ptr(scan), _ptr(mu), C.byref(scale)))
        return scan, mu, float(scale.value)

    def debug_h2_scan(self, q_flat, q_frame_offsets):
        """ss_dict_debug_h2_scan: raw packed-half scan distance of every pair -> (scan f32 [nq, nseg], mean frame, norm scale s, cost scale S)."""
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        nq = qo.shape[0] - 1
        scan = np.empty((nq, len(self)), dtype=np.float32)
        mu = np.zeros(16, dtype=np.float64)
        scale, s = C.c_float(0.0), C.c_float(0.0)
        self.ctx.check(self.ctx.lib.ss_dict_debug_h2_scan(self.h, _ptr(q), _ptr(qo), nq, _ptr(scan), _ptr(mu), C.byref(scale), C.byref(s)))
        return scan, mu, float(scale.value), float(s.value)

    def set_scan(self, first_stage):
        """ss_dict_set_scan: 0 = packed-half tensor-core scan first (default), 1 = fp32-DP tensor-core scan, 2 = fp32 CUDA-core scan"""
        self.ctx.check(self.ctx.lib.ss_dict_set_scan(self.h, int(first_stage)))

    def set_dtw_band(self, radius):
        """ss_dict_set_dtw_band: Sakoe-Chiba radius of SS_DTW matches and align() (0 = no band, the default). For a shard of a
        one-rank-per-process match (Comm.match), every rank must set the same radius."""
        self.ctx.check(self.ctx.lib.ss_dict_set_dtw_band(self.h, _band(radius)))

    @property
    def dtw_band(self):
        return int(self.ctx.lib.ss_dict_dtw_band(self.h))

    @property
    def last_scan_kind(self):
        return int(self.ctx.lib.ss_dict_last_scan_kind(self.h))

    @property
    def last_work(self):
        return int(self.ctx.lib.ss_dict_last_work(self.h))

    @property
    def last_uncertified(self):
        return int(self.ctx.lib.ss_dict_last_uncertified(self.h))

    @property
    def last_tc_fallback(self):
        return int(self.ctx.lib.ss_dict_last_tc_fallback(self.h))

    @property
    def last_exhaustive(self):
        return int(self.ctx.lib.ss_dict_last_exhaustive(self.h))


def _band(radius):
    r = int(radius)
    if not 0 <= r <= 0xFFFFFFFF:
        raise ValueError("dtw_band must be in 0..2**32-1 (got %d)" % r)
    return r


def shard_bounds(frame_offsets, nshards):
    """ss_shard_bounds: contiguous segment ranges balanced by frames -> nshards + 1 cut positions (host arithmetic only)."""
    off = np.ascontiguousarray(frame_offsets, dtype=np.uint64)
    cuts = np.zeros(int(nshards) + 1, dtype=np.uint64)
    L = _lib.load()
    rc = L.ss_shard_bounds(_ptr(off), off.shape[0] - 1, int(nshards), _ptr(cuts))
    if rc != 0:
        raise SoundsymError(rc, L.ss_last_error(None).decode())
    return [int(c) for c in cuts]


class Comm:
    """ss_comm: this rank's end of an NCCL communicator owned by the library (one rank per process). Rank 0 calls
    Comm.unique_id() and ships the bytes to the other ranks (any transport); every rank then constructs Comm(ctx, n, rank, id)."""

    def __init__(self, ctx, nranks, rank, id_bytes):
        self.ctx = ctx
        buf = (C.c_char * _lib.SS_COMM_ID_BYTES).from_buffer_copy(bytes(id_bytes))
        h = C.c_void_p()
        ctx.check(ctx.lib.ss_comm_create(ctx.h, int(nranks), int(rank), buf, C.byref(h)))
        self.h, self.nranks, self.rank = h, int(nranks), int(rank)

    @staticmethod
    def unique_id():
        buf = (C.c_char * _lib.SS_COMM_ID_BYTES)()
        L = _lib.load()
        rc = L.ss_comm_unique_id(buf)
        if rc != 0:
            raise SoundsymError(rc, L.ss_last_error(None).decode())
        return bytes(buf.raw)

    def close(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.lib.ss_comm_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def match(self, shard, q_flat, q_frame_offsets, mode=SS_DTW, k=1, targets=None):
        """ss_dict_match_sharded (collective: every rank calls it with the same queries and its own shard)
        -> the GLOBAL (idx u32 [nq, k], dist f64 [nq, k]) on every rank."""
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        nq = qo.shape[0] - 1
        idx = np.empty((nq, k), dtype=np.uint32)
        dist = np.empty((nq, k), dtype=np.float64)
        t = np.ascontiguousarray(targets, dtype=np.float64) if targets is not None else None
        self.ctx.check(self.ctx.lib.ss_dict_match_sharded(shard.h, self.h, _ptr(q), _ptr(qo), nq, int(mode), _ptr(t), int(k), _ptr(idx), _ptr(dist)))
        return idx, dist


class ShardedDictionary:
    """ss_sharded_dict: one dictionary partitioned across the GPUs of THIS process (one Context per GPU); match() has
    ss_dict_match's contract and returns the same bits as a single-GPU DeviceDictionary."""

    def __init__(self, ctxs, mfcc_flat, frame_offsets, ncoeffs=None):
        self.ctxs = list(ctxs)
        mfcc_flat = np.ascontiguousarray(mfcc_flat, dtype=np.float64)
        off = np.ascontiguousarray(frame_offsets, dtype=np.uint64)
        if ncoeffs is None:
            ncoeffs = mfcc_flat.shape[1]
        arr = (C.c_void_p * len(self.ctxs))(*[c.h for c in self.ctxs])
        h = C.c_void_p()
        lib = self.ctxs[0].lib
        self.ctxs[0].check(lib.ss_dict_create_sharded(arr, len(self.ctxs), _ptr(mfcc_flat), _ptr(off), off.shape[0] - 1, int(ncoeffs), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and self.ctxs[0].h:
            self.ctxs[0].lib.ss_sharded_dict_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __len__(self):
        return int(self.ctxs[0].lib.ss_sharded_dict_len(self.h))

    def set_dtw_band(self, radius):
        """ss_sharded_dict_set_dtw_band: the Sakoe-Chiba radius of every shard"""
        self.ctxs[0].check(self.ctxs[0].lib.ss_sharded_dict_set_dtw_band(self.h, _band(radius)))

    def match(self, q_flat, q_frame_offsets, mode=SS_DTW, k=1, targets=None):
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        nq = qo.shape[0] - 1
        idx = np.empty((nq, k), dtype=np.uint32)
        dist = np.empty((nq, k), dtype=np.float64)
        t = np.ascontiguousarray(targets, dtype=np.float64) if targets is not None else None
        lib = self.ctxs[0].lib
        self.ctxs[0].check(lib.ss_sharded_dict_match(self.h, _ptr(q), _ptr(qo), nq, int(mode), _ptr(t), int(k), _ptr(idx), _ptr(dist)))
        return idx, dist


class DeviceQueries:
    """ss_queries: a prepared query batch resident in HBM."""

    def __init__(self, ctx, q_flat, q_frame_offsets, ncoeffs=None):
        self.ctx = ctx
        q = np.ascontiguousarray(q_flat, dtype=np.float64)
        qo = np.ascontiguousarray(q_frame_offsets, dtype=np.uint64)
        if ncoeffs is None:
            ncoeffs = q.shape[1]
        self.nq = qo.shape[0] - 1
        h = C.c_void_p()
        ctx.check(ctx.lib.ss_queries_create(ctx.h, _ptr(q), _ptr(qo), self.nq, int(ncoeffs), C.byref(h)))
        self.h = h

    def close(self):
        if getattr(self, "h", None) and self.ctx.h:
            self.ctx.lib.ss_queries_destroy(self.h)
        self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


# ---------------------------------------------------------------------------------------------------------------
# the reference's types
# ---------------------------------------------------------------------------------------------------------------
_default_ctx = None


def default_context():
    global _default_ctx
    if _default_ctx is None:
        _default_ctx = Context(0)
    return _default_ctx


class Sound:
    """src/sound.rs:71-213. samples / mfccs are host f64 arrays; analyses run on the GPU."""

    def __init__(self, samples, sample_rate, mfccs, max_power, mean_mfccs, name=None, ctx=None):
        self.name = name
        self._samples = samples
        self._sample_rate = float(sample_rate)
        self._mfccs = mfccs
        self._max_power = max_power
        self._mean_mfccs = mean_mfccs
        self._ctx = ctx

    @classmethod
    def from_samples(cls, samples, sample_rate, mfccs=None, name=None, ctx=None):
        """Sound::from_samples (src/sound.rs:92-112). When mfccs are supplied they are kept (the reference recomputes
        and discards them, :94 — functionally invisible)."""
        ctx = ctx or default_context()
        samples = np.ascontiguousarray(samples, dtype=np.float64)
        m, mp, mean = ctx.analyze(samples, sample_rate, NCOEFFS)
        if mfccs is not None:
            m = np.ascontiguousarray(mfccs, dtype=np.float64).reshape(-1, NCOEFFS)
            with np.errstate(all="ignore"):
                mean = m.sum(axis=0) / m.shape[0] if m.shape[0] else np.full(NCOEFFS, np.nan)
        return cls(samples, sample_rate, m, mp, mean, name, ctx)

    @classmethod
    def from_path(cls, path, ctx=None):
        """Sound::from_path (src/sound.rs:116-126): integer PCM WAV, mono; sample conversion on the GPU."""
        import os
        ctx = ctx or default_context()
        pcm, sr, bits = _read_wav_pcm(path)
        if bits == 8:  # no integer ingest path for 8-bit: convert (src/sound.rs:118-120, denominator 127) then analyse
            samples = ctx.decode_pcm(pcm, 8)
            m, mp, mean = ctx.analyze(samples, sr, NCOEFFS)
        else:
            samples, m, mp, mean = ctx.analyze_pcm(pcm, bits, sr, NCOEFFS)
        return cls(samples, sr, m, mp, mean, os.path.splitext(os.path.basename(path))[0], ctx)

    def push_samples(self, new_samples):
        """Sound::push_samples (src/sound.rs:145-164), including its running-mean rule `(old*n0 + new*n1) * 0.5`."""
        initial = self.num_frames()
        self._samples = np.concatenate([self._samples, np.asarray(new_samples, dtype=np.float64)])
        tail = self._samples[initial * HOP:]
        m, mp, mean = self._ctx.analyze(tail, self._sample_rate, NCOEFFS)
        self._mfccs = np.concatenate([self._mfccs, m], axis=0)
        new_frames = self.num_frames() - initial
        with np.errstate(all="ignore"):
            self._mean_mfccs = (self._mean_mfccs * initial + mean * new_frames) * 0.5
        self._max_power = max(self._max_power, mp)

    def max_power(self):
        return self._max_power

    def samples(self):
        return self._samples

    def sample_rate(self):
        return self._sample_rate

    def mfccs(self):
        return self._mfccs.reshape(-1)

    def mfcc_arrays(self):
        return self._mfccs

    def mean_mfccs(self):
        return self._mean_mfccs

    def num_frames(self):
        return self._mfccs.shape[0]

    def write_file(self, path):
        """Sound::write_file (src/sound.rs:129-143): 32-bit int PCM, (i32::MAX as f64 * sample) as i32."""
        s = np.clip(np.trunc(self._samples * 2147483647.0), -2147483648.0, 2147483647.0).astype("<i4")
        with open(path, "wb") as f:
            f.write(b"RIFF" + struct.pack("<I", 36 + s.nbytes) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, int(self._sample_rate),
                    int(self._sample_rate) * 4, 4, 32) + b"data" + struct.pack("<I", s.nbytes))
            f.write(s.tobytes())


def _read_wav_pcm(path):
    """integer-PCM RIFF/WAVE reader (what hound::WavReader accepts at src/sound.rs:117): format tag 1, or 0xFFFE with the
    PCM sub-format; 8 / 16 / 24 / 32 bits (8-bit is unsigned offset-128, as hound converts it). Anything else raises
    ValueError, as hound returns Err."""
    with open(path, "rb") as f:
        data = f.read()
    if len(data) < 12 or data[:4] != b"RIFF" or data[8:12] != b"WAVE":
        raise ValueError("not a RIFF/WAVE file: %s" % path)
    pos, fmt, pcm = 12, None, None
    while pos + 8 <= len(data):
        cid, size = data[pos:pos + 4], struct.unpack("<I", data[pos + 4:pos + 8])[0]
        body = data[pos + 8:min(pos + 8 + size, len(data))]
        if cid == b"fmt ":
            if len(body) < 16:
                raise ValueError("truncated fmt chunk: %s" % path)
            tag, _, sr, _, _, bits = struct.unpack("<HHIIHH", body[:16])
            if tag == 0xFFFE:  # WAVE_FORMAT_EXTENSIBLE: the sub-format GUID's first two bytes carry the real tag
                if len(body) < 26:
                    raise ValueError("truncated extensible fmt chunk: %s" % path)
                tag = struct.unpack("<H", body[24:26])[0]
            if tag != 1:
                raise ValueError("unsupported WAV format tag %d (integer PCM only): %s" % (tag, path))
            if bits not in (8, 16, 24, 32):
                raise ValueError("unsupported bits per sample: %d" % bits)
            fmt = (sr, bits)
        elif cid == b"data" and pcm is None:
            if fmt is None:
                raise ValueError("data chunk before fmt chunk: %s" % path)
            bits = fmt[1]
            if bits == 8:
                pcm = np.frombuffer(body, dtype=np.uint8).astype(np.int32) - 128
            elif bits == 16:
                pcm = np.frombuffer(body[: len(body) // 2 * 2], dtype="<i2").astype(np.int32)
            elif bits == 24:
                b = np.frombuffer(body[: len(body) // 3 * 3], dtype=np.uint8).reshape(-1, 3).astype(np.int32)
                v = b[:, 0] | (b[:, 1] << 8) | (b[:, 2] << 16)
                pcm = np.where(v & 0x800000, v - (1 << 24), v).astype(np.int32)
            else:
                pcm = np.frombuffer(body[: len(body) // 4 * 4], dtype="<i4").astype(np.int32)
        pos += 8 + size + (size & 1)
    if fmt is None or pcm is None:
        raise ValueError("no fmt / data chunk: %s" % path)
    return pcm, float(fmt[0]), fmt[1]


class SoundDictionary:
    """src/sound.rs:288-371. `mode` selects the matcher: SS_COSINE_REF is the reference's, SS_DTW the extension, and
    SS_DTW_TARGET the extension's at_distance: the sounds whose SS_DTW distance is closest to each target (A13).
    `dtw_band`: Sakoe-Chiba radius of the SS_DTW distance and of align() (0 = no band; ss_dict_set_dtw_band)."""

    def __init__(self, ctx=None, mode=SS_COSINE_REF, dtw_band=0):
        self.sounds = []
        self.mode = mode
        self.dtw_band = _band(dtw_band)
        self._ctx = ctx or default_context()
        self._dev = None

    @classmethod
    def from_path(cls, path, ctx=None, mode=SS_COSINE_REF):
        """SoundDictionary::from_path (src/sound.rs:304-320): every *.wav of a directory (not recursive, other entries
        skipped) becomes one Sound, in directory order (sorted here: read_dir's order is platform-defined). The files
        are decoded on the host, then analysed together: one ss_sound_analyze_batch per distinct sample rate."""
        import os
        d = cls(ctx, mode)
        names = sorted(n for n in os.listdir(path) if os.path.splitext(n)[1] == ".wav" and os.path.isfile(os.path.join(path, n)))
        loaded = []
        for nme in names:
            pcm, sr, bits = _read_wav_pcm(os.path.join(path, nme))
            denom = float(0x7FFFFFFF >> (32 - bits))  # src/sound.rs:118-120
            loaded.append((os.path.splitext(nme)[0], sr, pcm.astype(np.float64) / denom))
        d.sounds = [None] * len(loaded)
        for sr in sorted(set(l[1] for l in loaded)):
            sel = [i for i, l in enumerate(loaded) if l[1] == sr]
            off = np.zeros(len(sel) + 1, dtype=np.uint64)
            off[1:] = np.cumsum([loaded[i][2].shape[0] for i in sel])
            flat = np.concatenate([loaded[i][2] for i in sel]) if sel else np.zeros(0)
            mfcc, foff, mp, mean = d._ctx.analyze_batch(flat, off, sr, NCOEFFS)
            for j, i in enumerate(sel):
                d.sounds[i] = Sound(loaded[i][2], sr, mfcc[int(foff[j]):int(foff[j + 1])], float(mp[j]), mean[j], loaded[i][0], d._ctx)
        return d

    @classmethod
    def from_segments(cls, sound, segments, ctx=None, mode=SS_COSINE_REF):
        d = cls(ctx or sound._ctx, mode)
        d.add_segments(sound, segments)
        return d

    def add_segments(self, sound, segments):
        """src/sound.rs:330-343: segment i takes seg_i samples and (seg_i / HOP) * NCOEFFS MFCC values, in order."""
        spos, fpos = 0, 0
        samples, mfccs = sound.samples(), sound.mfcc_arrays()
        segs = [int(s) for s in segments]
        # Sound::from_samples(samp, sr, Some(mfccs), None) runs analyze_max_power on every cut (src/sound.rs:95): all cuts
        # in ONE batched launch (ss_sound_analyze_batch with only the max-power output requested)
        ctx = sound._ctx or self._ctx
        bounds = np.zeros(len(segs) + 1, dtype=np.uint64)
        bounds[1:] = np.minimum(np.cumsum(segs), len(samples))
        powers = ctx.max_power_batch(samples[:int(bounds[-1])], bounds) if segs else np.zeros(0)
        for i, seg in enumerate(segs):
            nf = seg // HOP
            samp = samples[spos:spos + seg]
            m = mfccs[fpos:fpos + nf]
            spos += seg
            fpos += nf
            with np.errstate(all="ignore"):  # mean of the supplied MFCC rows as analyze_mean_mfccs
                mean = m.sum(axis=0) / m.shape[0] if m.shape[0] else np.full(NCOEFFS, np.nan)
            self.sounds.append(Sound(samp, sound.sample_rate(), m, float(powers[i]), mean, None, ctx))
        self._dev = None

    def _device(self):
        if self._dev is None:
            if not self.sounds:
                raise SoundsymError(_lib.SS_ERR_EMPTY_DICT, "match against an empty dictionary")
            lens = np.array([s.num_frames() for s in self.sounds], dtype=np.uint64)
            off = np.zeros(len(lens) + 1, dtype=np.uint64)
            off[1:] = np.cumsum(lens)
            flat = np.concatenate([s.mfcc_arrays() for s in self.sounds], axis=0) if int(off[-1]) else np.zeros((0, NCOEFFS))
            self._dev = DeviceDictionary(self._ctx, flat, off, NCOEFFS)
        if self._dev.dtw_band != self.dtw_band:  # a new device dictionary (add_segments drops it), or dtw_band was reassigned
            self._dev.set_dtw_band(self.dtw_band)
        return self._dev

    def match_indices(self, sounds, targets=None, k=1):
        """batched at_distance: one query per sound -> (idx [nq, k], dist [nq, k])."""
        lens = np.array([s.num_frames() for s in sounds], dtype=np.uint64)
        off = np.zeros(len(lens) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        flat = np.concatenate([s.mfcc_arrays() for s in sounds], axis=0) if int(off[-1]) else np.zeros((0, NCOEFFS))
        return self._device().match(flat, off, self.mode, k, targets)

    def align(self, sounds, indices):
        """the DTW warping path of every sound against the dictionary sound of the same position in `indices` (as
        match_indices returns them) -> (paths: list of uint32 [n, 2] arrays of (frame of the sound, frame of the dictionary
        sound), dist f64). Works in either mode: the path is the SS_DTW one whatever matcher chose the indices."""
        lens = np.array([s.num_frames() for s in sounds], dtype=np.uint64)
        off = np.zeros(len(lens) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        flat = np.concatenate([s.mfcc_arrays() for s in sounds], axis=0) if int(off[-1]) else np.zeros((0, NCOEFFS))
        return self._device().align(flat, off, indices)

    def locate(self, sounds, k=1):
        """where inside the dictionary sounds each sound occurs (subsequence DTW, ss_dict_locate) -> (idx, start, end, cost),
        each [n, k]: the k best dictionary sounds by (cost, index), and in each the frames start..end (inclusive) the sound
        fits best, at the unnormalised DTW cost. Frames map to samples as in add_segments: frame t of a sound begins at its
        sample t * HOP, so the located passage is samples [start * HOP, end * HOP + BIN) of dictionary sound idx. Works in
        either mode, and dtw_band does not apply."""
        lens = np.array([s.num_frames() for s in sounds], dtype=np.uint64)
        off = np.zeros(len(lens) + 1, dtype=np.uint64)
        off[1:] = np.cumsum(lens)
        flat = np.concatenate([s.mfcc_arrays() for s in sounds], axis=0) if int(off[-1]) else np.zeros((0, NCOEFFS))
        return self._device().locate(flat, off, k)

    def at_distance(self, distance, other):
        """src/sound.rs:351-370 (always Some)."""
        idx, _ = self.match_indices([other], [distance])
        return self.sounds[int(idx[0, 0])]

    def match_sound(self, other):
        """src/sound.rs:346-348. The reference's 1.0 is cosine's perfect similarity; in SS_DTW_TARGET mode the perfect
        distance is 0.0, so there match_sound is at_distance(0.0) (the nearest sound, as in SS_DTW)."""
        return self.at_distance(0.0 if self.mode == SS_DTW_TARGET else 1.0, other)


class SoundSequence:
    """src/sound.rs:373-484."""

    def __init__(self, sounds, ctx=None):
        self._sounds = list(sounds)
        self._ctx = ctx or (self._sounds[0]._ctx if self._sounds else default_context())
        if len(self._sounds) >= 2:
            self._distances = self._ctx.sequence_distances(np.stack([s.mean_mfccs() for s in self._sounds]))
        else:
            self._distances = np.zeros(0)

    def sounds(self):
        return self._sounds

    def distances(self):
        return self._distances

    def clone_from_dictionary(self, dictionary, warp=False):
        """src/sound.rs:451-472: nearest dictionary sound per segment (ONE batched match), zero-padded / truncated to
        the target segment's length on the GPU (ss_resynth). warp=True: each matched sound follows its target's timing along
        the DTW warping path of the pair (dictionary.align, with the dictionary's band, whichever matcher chose it; then
        ss_resynth_warped), and the output segments are analysed in one batch."""
        if not self._sounds:
            return SoundSequence([], self._ctx)
        idx, _ = dictionary.match_indices(self._sounds)
        idx = idx[:, 0]
        dlens = np.array([len(s.samples()) for s in dictionary.sounds], dtype=np.uint64)
        doff = np.zeros(len(dlens) + 1, dtype=np.uint64)
        doff[1:] = np.cumsum(dlens)
        dsamples = np.concatenate([s.samples() for s in dictionary.sounds]) if int(doff[-1]) else np.zeros(0)
        tlens = np.array([len(s.samples()) for s in self._sounds], dtype=np.uint64)
        if warp:
            return self._clone_warped(dictionary, idx, dsamples, doff, tlens)
        out = self._ctx.resynth(dsamples, doff, idx, tlens)
        sounds, pos = [], 0
        for t, s in enumerate(self._sounds):
            ln = int(tlens[t])
            m = dictionary.sounds[int(idx[t])]
            if ln == len(m.samples()):
                sounds.append(m)  # shares the Arc (src/sound.rs:463-464)
            else:
                sounds.append(Sound.from_samples(out[pos:pos + ln], s.sample_rate(), None, None, self._ctx))
            pos += ln
        seq = SoundSequence(sounds, self._ctx)
        seq._assembled = out
        return seq

    def _clone_warped(self, dictionary, idx, dsamples, doff, tlens):
        sr = self._sounds[0].sample_rate()
        if any(s.sample_rate() != sr for s in self._sounds):
            raise ValueError("warped resynthesis analyses its output in one batch: every segment needs the same sample rate")
        paths, _ = dictionary.align(self._sounds, idx)
        poff = np.zeros(len(paths) + 1, dtype=np.uint64)
        poff[1:] = np.cumsum([p.shape[0] for p in paths])
        cells = np.concatenate(paths) if int(poff[-1]) else np.zeros((0, 2), dtype=np.uint32)
        out = self._ctx.resynth_warped(dsamples, doff, idx, cells, poff, tlens)
        ooff = np.zeros(len(tlens) + 1, dtype=np.uint64)
        ooff[1:] = np.cumsum(tlens)
        mfcc, foff, mp, mean = self._ctx.analyze_batch(out, ooff, sr, NCOEFFS)
        sounds = [Sound(out[int(ooff[t]):int(ooff[t + 1])], sr, mfcc[int(foff[t]):int(foff[t + 1])], float(mp[t]), mean[t], None, self._ctx)
                  for t in range(len(tlens))]
        seq = SoundSequence(sounds, self._ctx)
        seq._assembled = out
        return seq

    @classmethod
    def from_timestamps(cls, sound, timestamps):
        """SoundSequence::from_timestamps (src/sound.rs:419-430): one new Sound per (start, end, label), cut at
        round(t * sample_rate) .. round(end * sample_rate) inclusive. The cuts are analysed together
        (ss_sound_analyze_batch) instead of one Sound::from_samples each."""
        sr = sound.sample_rate()
        src = sound.samples()
        cuts = []
        for t in timestamps:
            a, b = int(round(t[0] * sr)), int(round(t[1] * sr))
            if a < 0 or b + 1 > len(src) or a > b + 1:
                raise IndexError("timestamp (%r, %r) outside the sound" % (t[0], t[1]))  # the reference panics on the slice
            cuts.append(src[a:b + 1])
        off = np.zeros(len(cuts) + 1, dtype=np.uint64)
        off[1:] = np.cumsum([c.shape[0] for c in cuts])
        flat = np.concatenate(cuts) if cuts else np.zeros(0)
        ctx = sound._ctx or default_context()
        mfcc, foff, mp, mean = ctx.analyze_batch(flat, off, sr, NCOEFFS)
        sounds = [Sound(np.array(c), sr, mfcc[int(foff[j]):int(foff[j + 1])], float(mp[j]), mean[j], t[2], ctx)
                  for j, (c, t) in enumerate(zip(cuts, timestamps))]
        return cls(sounds, ctx)

    def morph_to(self, distances, dictionary):
        """src/sound.rs:440-449 (batched: one at_distance per (sound, distance) pair)."""
        n = min(len(self._sounds), len(distances))
        idx, _ = dictionary.match_indices(self._sounds[:n], list(distances[:n]))
        return SoundSequence([dictionary.sounds[int(i)] for i in idx[:, 0]], self._ctx)

    @classmethod
    def from_distances(cls, distances, start, dictionary):
        """src/sound.rs:405-417: a chain, step t matches the sound step t - 1 returned. SS_COSINE_REF runs it on the device
        in one call (ss_dict_walk), and so does SS_DTW_TARGET (ss_dict_walk_dtw; a step with no result raises IndexError
        there, as at_distance does); SS_DTW keeps the nq = 1 loop (its at_distance ignores the target)."""
        sounds = [start]
        distances = list(distances)
        if distances and dictionary.mode in (SS_COSINE_REF, SS_DTW_TARGET):
            dev = dictionary._device()
            walk = dev.walk if dictionary.mode == SS_COSINE_REF else dev.walk_dtw
            idx, _ = walk(start.mfcc_arrays(), distances)
            sounds += [dictionary.sounds[int(i)] for i in idx]  # (0xFFFFFFFF: IndexError at that step)
        else:
            for d in distances:
                sounds.append(dictionary.at_distance(d, sounds[-1]))
        return cls(sounds)

    def to_sound(self):
        """src/sound.rs:475-483."""
        if getattr(self, "_assembled", None) is not None:
            samples = self._assembled
        else:
            samples = np.concatenate([s.samples() for s in self._sounds]) if self._sounds else np.zeros(0)
        sr = self._sounds[0].sample_rate() if self._sounds else 44100.0
        return Sound.from_samples(samples, sr, None, None, self._ctx)


class Partitioner:
    """src/lib.rs:62-151. `model` = (means, covs, weights) of the 26-component GMM, or None before train()."""

    def __init__(self, sound, ctx=None):
        self.sound = sound
        self.depth = 5
        self.threshold = 4
        self.model = None
        self._ctx = ctx or sound._ctx or default_context()

    @classmethod
    def from_path(cls, path, ctx=None):
        """Partitioner::from_path (src/lib.rs:85-88)."""
        return cls(Sound.from_path(path, ctx), ctx)

    def set_depth(self, depth):
        self.depth = int(depth)
        return self

    def set_threshold(self, threshold):
        self.threshold = int(threshold)
        return self

    def train(self, model=None, seed=0):
        """Partitioner::train (src/lib.rs:101-107): 26 full-covariance Gaussians, 5 EM rounds, Regularized(0.1), on the
        GPU (ss_gmm_train). The reference seeds its means from thread_rng, so its model differs from run to run; here
        the draw is seeded. A ready model (means, covs, weights) may be supplied instead."""
        self.model = model if model is not None else self._ctx.gmm_train(self.sound.mfcc_arrays(), NCLUSTERS, 5, 0.1, seed)

    def partition_other(self, sound):
        """src/lib.rs:112-144: segment lengths in samples; error "Must first train model" without a model."""
        return self._ctx.partition(sound.mfcc_arrays(), self.model, self.depth, self.threshold)

    def partition(self):
        return self.partition_other(self.sound)


class Timestamp(tuple):
    """src/sound.rs:508: (start seconds, end seconds, optional label)."""

    def __new__(cls, start, end, label=None):
        return super().__new__(cls, (float(start), float(end), label))


def audacity_labels_to_timestamps(path):
    """src/sound.rs:511-531: one `start<TAB>end<TAB>label` line per stamp; a field that is missing or does not parse is
    0.0, a missing label is None."""
    def num(x):
        try:
            return float(x)
        except (TypeError, ValueError):
            return 0.0
    out = []
    with open(path, "r") as f:
        for line in f:
            if not line:
                continue
            parts = line.strip().split("\t")
            out.append(Timestamp(num(parts[0]) if len(parts) > 0 else 0.0, num(parts[1]) if len(parts) > 1 else 0.0,
                                 parts[2] if len(parts) > 2 else None))
    return out


def _write_wav_i32(path, samples, sample_rate):
    # hound WavSpec{channels 1, bits 32, Int}; `(sample * i32::MAX as f64) as i32` saturates and truncates toward zero
    v = np.asarray(samples, dtype=np.float64) * 2147483647.0
    v = np.where(np.isnan(v), 0.0, v)
    q = np.clip(np.trunc(v), -2147483648.0, 2147483647.0).astype("<i4")
    with open(path, "wb") as f:
        f.write(b"RIFF" + struct.pack("<I", 36 + q.nbytes) + b"WAVEfmt " + struct.pack("<IHHIIHH", 16, 1, 1, int(sample_rate), int(sample_rate) * 4,
                4, 32) + b"data" + struct.pack("<I", q.nbytes))
        f.write(q.tobytes())


def write_splits(sound, splits, out_path):
    """write_splits (src/lib.rs:155-178): consecutive cuts of `sound` written as `<out>/<idx:05>_<len>.wav`, 32-bit PCM."""
    import os
    pos, samples = 0, sound.samples()
    for idx, split in enumerate(splits):
        split = int(split)
        _write_wav_i32(os.path.join(out_path, "%05d_%d.wav" % (idx, split)), samples[pos:pos + split], sound.sample_rate())
        pos += split
