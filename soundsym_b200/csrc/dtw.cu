// dtw.cu — the DTW matcher (SURVEY.md §8a row 20; spec oracle/ASSUMPTIONS.h A8). No reference counterpart exists;
// it slots into SoundDictionary::at_distance's place (src/sound.rs:351-370) as match mode SS_DTW.
//
// Filter and refine:
//   1. k_dtw_scan     fp32, every (query, dictionary segment) pair. One THREAD per pair: the 32 lanes of a warp are 32
//                     queries of equal length, the dictionary segment is warp-uniform and is streamed through shared
//                     memory by TMA bulk copies (cp.async.bulk + mbarrier, 3-stage ring). A thread keeps one DP row
//                     (<= 32 columns = one "strip") in registers and walks RB query rows per pass so that each
//                     broadcast LDS of a dictionary frame feeds RB cells. Local cost = |a|^2 + |b|^2 - 2ab with the
//                     contraction on packed FFMA2 (fma.rn.f32x2); DP step = FMNMX3 + FADD. Every thread keeps its KP
//                     best candidates in registers.
//   2. k_dtw_merge    per query, merges the per-slice candidate lists.
//   3. k_dtw_rescore_warp  f64, direct (a-b)^2, unfused — the oracle's arithmetic — on the KP candidates only.
//   4. k_dtw_finalize sorts by (distance, index), writes the top-k, and certifies that no pair outside the candidate
//                     list could have entered it given the scan's error bound.
// SS_DTW_TARGET (DESIGN.md §3.1h) runs the same four steps with the scan's TARGET form: it keeps the pairs of smallest
// lower bound on e = |D - t| instead of smallest scan distance, under the dictionary's band, and 3. / 4. rank by exact e.
#include <algorithm>
#include <cmath>
#include <numeric>

#include <chrono>

#include "match.cuh"

namespace ss {

// ---------------------------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long ffma2(unsigned long long a, unsigned long long b, unsigned long long c) {
    unsigned long long d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ float min3f(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}
__device__ __forceinline__ float lo32(unsigned long long v) { return __uint_as_float((unsigned)v); }
__device__ __forceinline__ float hi32(unsigned long long v) { return __uint_as_float((unsigned)(v >> 32)); }

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, unsigned count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "WAIT_LOOP:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra DONE;\n"
        "bra WAIT_LOOP;\n"
        "DONE:\n"
        "}\n" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}
// 1-D TMA bulk copy global -> shared, completion counted in bytes on an mbarrier
__device__ __forceinline__ void bulk_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------------------------------------------------------
// layout builders
// ---------------------------------------------------------------------------------------------------------------
// dictionary stream: frame f -> 16 floats [b_0..b_{c-1}, 0.., |b|^2 at slot 13, 0, 0]
__global__ void k_dict_stream(const double* __restrict__ mfcc, size_t frames, int c, float* __restrict__ stream,
                              float* __restrict__ max_norm) {
    const size_t f = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    float nrm = 0.f;
    if (f < frames) {
        float v[kSlots];
#pragma unroll
        for (int k = 0; k < kSlots; k++) v[k] = 0.f;
        double acc = 0.0;
#pragma unroll
        for (int k = 0; k < SS_MAX_NCOEFFS; k++)
            if (k < c) {
                v[k] = (float)mfcc[f * c + k];
                acc += (double)v[k] * (double)v[k];
            }
        nrm = (float)acc;
        v[kNormSlot] = nrm;
        float4* dst = reinterpret_cast<float4*>(stream + f * kSlots);
        dst[0] = make_float4(v[0], v[1], v[2], v[3]);
        dst[1] = make_float4(v[4], v[5], v[6], v[7]);
        dst[2] = make_float4(v[8], v[9], v[10], v[11]);
        dst[3] = make_float4(v[12], v[13], v[14], v[15]);
    }
    // block max -> atomicMax on the (non-negative) float's bit pattern
    for (int o = 16; o; o >>= 1) nrm = fmaxf(nrm, __shfl_xor_sync(0xffffffffu, nrm, o));
    if ((threadIdx.x & 31) == 0 && nrm == nrm) atomicMax(reinterpret_cast<unsigned*>(max_norm), __float_as_uint(nrm));
}

// query lanes: row (group g, frame i), lane l -> 16 floats [-2 a_0..-2 a_{c-1}, 0.., 1.0 at slot 13, |a|^2 at slot 14, 0]
// stored as [row][4][32] float4 so that a warp's load of one float4 column is one 512-byte coalesced access.
__global__ void k_query_lanes(const double* __restrict__ mfcc, const uint64_t* __restrict__ off, int c,
                              const uint32_t* __restrict__ group_len, const uint32_t* __restrict__ group_rowbase,
                              const uint32_t* __restrict__ group_qid, uint32_t ngroups, float4* __restrict__ lanes,
                              float* __restrict__ max_norm) {
    const uint32_t g = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const uint32_t len = group_len[g];
    const uint32_t rows_padded = group_rowbase[g + 1] - group_rowbase[g];
    const uint32_t qid = group_qid[g * 32 + lane];
    float mx = 0.f;
    for (uint32_t i = threadIdx.x >> 5; i < rows_padded; i += blockDim.x >> 5) {
        float v[kSlots];
#pragma unroll
        for (int k = 0; k < kSlots; k++) v[k] = 0.f;
        if (qid != 0xFFFFFFFFu && i < len) {
            const double* src = mfcc + (off[qid] + i) * c;
            double acc = 0.0;
#pragma unroll
            for (int k = 0; k < SS_MAX_NCOEFFS; k++)
                if (k < c) {
                    const float a = (float)src[k];
                    v[k] = -2.f * a;
                    acc += (double)a * (double)a;
                }
            v[kNormSlot] = 1.f;
            v[kLaneNaSlot] = (float)acc;
            mx = fmaxf(mx, v[kLaneNaSlot]);
        }
        float4* dst = lanes + ((size_t)(group_rowbase[g] + i) * 4) * 32 + lane;
        dst[0] = make_float4(v[0], v[1], v[2], v[3]);
        dst[32] = make_float4(v[4], v[5], v[6], v[7]);
        dst[64] = make_float4(v[8], v[9], v[10], v[11]);
        dst[96] = make_float4(v[12], v[13], v[14], v[15]);
    }
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if (lane == 0 && mx == mx) atomicMax(reinterpret_cast<unsigned*>(max_norm), __float_as_uint(mx));
}

// ---------------------------------------------------------------------------------------------------------------
// the fp32 scan
// ---------------------------------------------------------------------------------------------------------------
struct ScanParams {
    const float4* qlane;
    const uint32_t* group_len;
    const uint32_t* group_rowbase;
    uint32_t ngroups;
    const float* stream;
    const int4* strips;
    const int4* tiles;
    const uint32_t* slice_tile;  // nslices + 1
    uint32_t nslices;
    unsigned long long* partial;  // [nslices][ngroups*32][KP]
    float* scratch;               // per CTA: scratch_rows x 128 floats (strip boundary columns of multi-strip segments)
    uint32_t scratch_rows;
};
// what the TARGET scans (SS_DTW_TARGET) read besides: the targets in the caller's query order (NULL: t = 0), the lanes' query
// ids, the batch's and the shard's largest frame norms (the per-cell error of E), the Sakoe-Chiba radius (0: no band)
struct ScanTarget {
    const double* targets;
    const uint32_t* group_qid;
    const float* max_na;
    const float* max_nb;
    uint32_t band;
};

// The TARGET scan's key of a pair (DESIGN.md §3.1h): a lower bound on e = |D - t| for a pair of ncells = Lq + Ld - 1 path cells
// at most whose scan distance is s, max(0, |s - t| - E), E = (g |s| + (1 + g) ec) / (1 - g) with g = gamma_{ncells+1} of fp32 and
// ec = kScanCellEps (max|a|^2 + max|b|^2) the error of one computed local cost. The f64 evaluation of E is covered by the factor
// 1.001, |s - t| and the subtraction of E round down, and so does the conversion to float. A NaN / inf scan distance stays what it
// is: such a pair is never a candidate, as in SS_DTW.
constexpr double kScanCellEps = 4e-6;
__device__ __forceinline__ float target_key(float s, double t, double ec, uint32_t ncells) {
    const double sd = (double)s;
    if (!(fabs(sd) < __longlong_as_double(0x7ff0000000000000ll))) return s;
    const double nu = (double)(ncells + 1) * 0x1p-24, g = nu / (1.0 - nu);
    const double e = 1.001 * (g * fabs(sd) + (1.0 + g) * ec) / (1.0 - g);
    const double lo = __dsub_rd(sd >= t ? __dsub_rd(sd, t) : __dsub_rd(t, sd), e);
    return lo > 0.0 ? __double2float_rd(lo) : 0.f;
}

constexpr int kTileFloats = kTileFrames * kSlots;
constexpr int kScanSmemBytes = kStages * kTileFloats * 4 + kStages * 8 + kStages * 4 + 4;

// TARGET: the SS_DTW_TARGET form. Each lane reads its query's target; a pair's key is target_key, not the scan distance, and
// under a band (p.band != 0) cells outside it are +inf by one 64-bit integer test per cell (A10's rule, warp-uniform: the
// lanes of a warp share Lq and the segment).
template <int RB, int KP, bool TARGET = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32, RB <= 2 ? 4 : 3) k_dtw_scan(const ScanParams p, const ScanTarget tg) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    float* stage_buf = reinterpret_cast<float*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + kStages * kTileFloats * 4);
    unsigned* cnt = reinterpret_cast<unsigned*>(full + kStages);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t qb = blockIdx.x / p.nslices, slice = blockIdx.x % p.nslices;
    const uint32_t g = qb * kWarpsPerCta + warp;
    const uint32_t nactive = min((uint32_t)kWarpsPerCta, p.ngroups - qb * kWarpsPerCta);
    const uint32_t t0 = p.slice_tile[slice], t1 = p.slice_tile[slice + 1];

    auto issue = [&](uint32_t t, int s) {
        const int4 td = __ldg(&p.tiles[t]);
        const unsigned bytes = (unsigned)td.y * kSlots * 4;
        mbar_expect_tx(&full[s], bytes);
        bulk_g2s(stage_buf + s * kTileFloats, p.stream + (size_t)(uint32_t)td.x * kSlots, bytes, &full[s]);
    };

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; s++) {
            mbar_init(&full[s], 1);
            cnt[s] = 0;
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    if (threadIdx.x == 0)
        for (int s = 0; s < kStages && t0 + s < t1; s++) issue(t0 + s, s);
    if (g >= p.ngroups) return;

    const uint32_t Lq = p.group_len[g];
    const uint32_t nbands = (Lq + RB - 1) / RB;
    const float4* arow = p.qlane + (size_t)p.group_rowbase[g] * 4 * 32 + lane;
    float* scr = p.scratch ? p.scratch + ((size_t)blockIdx.x * p.scratch_rows) * 128 + threadIdx.x : nullptr;
    const float INF = __int_as_float(0x7f800000);

    float kd[KP];
    uint32_t ki[KP];
#pragma unroll
    for (int s = 0; s < KP; s++) kd[s] = INF, ki[s] = 0xFFFFFFFFu;
    double tq = 0.0, ec = 0.0;
    uint32_t col_next = 0;  // TARGET: the first column of the segment's next strip
    if constexpr (TARGET) {
        const uint32_t qid = tg.group_qid[g * 32 + lane];
        tq = (tg.targets && qid != 0xFFFFFFFFu) ? tg.targets[qid] : 0.0;
        ec = kScanCellEps * ((double)tg.max_na[0] + (double)tg.max_nb[0]);
    }

    for (uint32_t t = t0; t < t1; ++t) {
        const uint32_t n = t - t0;
        const int s = (int)(n % kStages);
        const int4 td = __ldg(&p.tiles[t]);
        mbar_wait(&full[s], (n / kStages) & 1);
        const float* sb = stage_buf + s * kTileFloats;

        for (int u = 0; u < td.w; ++u) {
            const int4 sd = __ldg(&p.strips[td.z + u]);
            const int len = sd.z & 0xFFFF;
            const bool first = (sd.z >> 16) & 1, last = (sd.z >> 17) & 1;
            const float* bs = sb + ((uint32_t)sd.x - (uint32_t)td.x) * kSlots;
            // TARGET under a band: cell (i, col0 + j) is inside iff |i A - (col0 + j) B| <= bw (band_rows' test)
            long long bA = 0, bB = 0, bw = 0;
            uint32_t col0 = 0;
            bool banded = false;
            if constexpr (TARGET) {
                col0 = first ? 0 : col_next;
                col_next = col0 + (uint32_t)len;
                banded = tg.band != 0;
                bA = (long long)sd.w - 1, bB = (long long)Lq - 1;
                const long long lmax = max((long long)Lq, (long long)sd.w);
                bw = min((long long)tg.band, lmax) * max(bA, bB);
            }

            float dprev[kStrip];
#pragma unroll
            for (int j = 0; j < kStrip; j++) dprev[j] = INF;
            float leftv[RB];
            float carry = INF;  // D(i0-1, strip_start-1) for the next band of a non-first strip

            for (uint32_t b = 0; b < nbands; ++b) {
                const uint32_t i0 = b * RB;
                unsigned long long a[RB][8];
#pragma unroll
                for (int r = 0; r < RB; r++) {
                    const ulonglong2* src = reinterpret_cast<const ulonglong2*>(arow + (size_t)(i0 + r) * 4 * 32);
#pragma unroll
                    for (int q4 = 0; q4 < 4; q4++) {
                        const ulonglong2 v = __ldg(src + q4 * 32);
                        a[r][2 * q4] = v.x;
                        a[r][2 * q4 + 1] = v.y;
                    }
                }
                float diag0;
                if (first) {
#pragma unroll
                    for (int r = 0; r < RB; r++) leftv[r] = INF;
                    diag0 = b == 0 ? 0.f : INF;
                } else {
                    diag0 = b == 0 ? INF : carry;
#pragma unroll
                    for (int r = 0; r < RB; r++) leftv[r] = scr[(size_t)(i0 + r) * 128];
                    carry = leftv[RB - 1];
                }
#pragma unroll
                for (int j = 0; j < kStrip; j++) {
                    if (j < len) {
                        const ulonglong2 b0 = *reinterpret_cast<const ulonglong2*>(bs + j * kSlots);
                        const ulonglong2 b1 = *reinterpret_cast<const ulonglong2*>(bs + j * kSlots + 4);
                        const ulonglong2 b2 = *reinterpret_cast<const ulonglong2*>(bs + j * kSlots + 8);
                        const unsigned long long b3 = *reinterpret_cast<const unsigned long long*>(bs + j * kSlots + 12);
                        const float dold = dprev[j];
                        float upv = dold, diag = diag0;
#pragma unroll
                        for (int r = 0; r < RB; r++) {
                            unsigned long long acc = a[r][7];  // (|a|^2, 0)
                            acc = ffma2(a[r][0], b0.x, acc);
                            acc = ffma2(a[r][1], b0.y, acc);
                            acc = ffma2(a[r][2], b1.x, acc);
                            acc = ffma2(a[r][3], b1.y, acc);
                            acc = ffma2(a[r][4], b2.x, acc);
                            acc = ffma2(a[r][5], b2.y, acc);
                            acc = ffma2(a[r][6], b3, acc);  // (a_12 b_12, 1 * |b|^2)
                            const float c = lo32(acc) + hi32(acc);
                            const float m = min3f(leftv[r], upv, diag);
                            float cur = c + m;
                            if constexpr (TARGET) {
                                if (banded) {
                                    const long long x = (long long)(i0 + r) * bA - (long long)(col0 + j) * bB;
                                    if (x < -bw || x > bw) cur = INF;
                                }
                            }
                            diag = leftv[r];
                            leftv[r] = cur;
                            upv = cur;
                        }
                        diag0 = dold;
                        dprev[j] = upv;
                    }
                }
                if (!last) {
#pragma unroll
                    for (int r = 0; r < RB; r++) scr[(size_t)(i0 + r) * 128] = leftv[r];
                }
            }
            if (last) {
                const int rstar = (int)(Lq - 1 - (nbands - 1) * RB);
                float res = leftv[0];
#pragma unroll
                for (int r = 1; r < RB; r++)
                    if (r == rstar) res = leftv[r];
                float dist = res * (1.0f / (float)(Lq + (uint32_t)sd.w));
                if constexpr (TARGET) dist = target_key(dist, tq, ec, Lq + (uint32_t)sd.w - 1);
                if (dist < kd[KP - 1]) {
                    kd[KP - 1] = dist;
                    ki[KP - 1] = (uint32_t)sd.y;
#pragma unroll
                    for (int s2 = KP - 1; s2 > 0; s2--) {
                        if (kd[s2] < kd[s2 - 1]) {
                            const float td2 = kd[s2];
                            kd[s2] = kd[s2 - 1];
                            kd[s2 - 1] = td2;
                            const uint32_t ti = ki[s2];
                            ki[s2] = ki[s2 - 1];
                            ki[s2 - 1] = ti;
                        }
                    }
                }
            }
        }
        // release the stage: the last warp to finish this tile refills it with tile t + kStages
        __syncwarp();
        if (lane == 0) {
            __threadfence_block();
            const unsigned old = atomicAdd(&cnt[s], 1u);
            if (old == nactive - 1) {
                cnt[s] = 0;
                if (t + kStages < t1) {
                    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
                    issue(t + kStages, s);
                }
            }
        }
    }

    unsigned long long* out = p.partial + ((size_t)slice * p.ngroups * 32 + (size_t)g * 32 + lane) * KP;
#pragma unroll
    for (int s = 0; s < KP; s++)
        out[s] = ki[s] == 0xFFFFFFFFu ? kEmptyKey : (((unsigned long long)f2ord(kd[s]) << 32) | ki[s]);
}

// per query slot: merge nslices sorted lists (slices cover increasing index ranges, so a strict '<' keeps the lowest
// index among equal distances)
template <int KP>
__global__ void k_dtw_merge(const unsigned long long* __restrict__ partial, uint32_t nslices, uint32_t nslots,
                            uint32_t* __restrict__ cand_idx, float* __restrict__ cand_adist) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= nslots) return;
    unsigned long long best[KP];
#pragma unroll
    for (int s = 0; s < KP; s++) best[s] = kEmptyKey;
    for (uint32_t sl = 0; sl < nslices; sl++) {
        const unsigned long long* src = partial + ((size_t)sl * nslots + slot) * KP;
#pragma unroll
        for (int s = 0; s < KP; s++) {
            const unsigned long long key = src[s];
            if (key < best[KP - 1]) {
                best[KP - 1] = key;
#pragma unroll
                for (int s2 = KP - 1; s2 > 0; s2--)
                    if (best[s2] < best[s2 - 1]) {
                        const unsigned long long tmp = best[s2];
                        best[s2] = best[s2 - 1];
                        best[s2 - 1] = tmp;
                    }
            }
        }
    }
#pragma unroll
    for (int s = 0; s < KP; s++) {
        cand_idx[(size_t)slot * KP + s] = best[s] == kEmptyKey ? 0xFFFFFFFFu : (uint32_t)best[s];
        cand_adist[(size_t)slot * KP + s] = best[s] == kEmptyKey ? __int_as_float(0x7f800000) : key_dist(best[s]);
    }
}

}  // namespace ss

// exact f64 kernels live in exact.cu (compiled with --fmad=false)
namespace ss {
bool dtw_tc_applies(const ss_dict* d, const ss_queries* q);
int dtw_tc_match_dev(ss_dict* d, ss_queries* q, int k, bool timed, uint32_t* d_out_idx, double* d_out_dist);
bool dtw_h2_applies(const ss_dict* d, const ss_queries* q);
int dtw_h2_match_dev(ss_dict* d, ss_queries* q, int k, bool wide, bool second_chance, bool timed, uint32_t* d_out_idx, double* d_out_dist);
int dtw_exhaustive_match(ss_dict* d, ss_queries* q, int k, const std::vector<uint32_t>& subset, uint32_t* d_out_idx, double* d_out_dist,
                         bool target = false, const double* d_targets = nullptr);
}

namespace ss {

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
int dtw_dict_build(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    const size_t frames = d->total_frames;
    if (frames > 0xFFFFFFF0ull) return set_error(ctx, SS_ERR_INVALID, "dictionary shard too large (%zu frames)", frames);
    std::vector<StripDesc> strips;
    std::vector<TileDesc> tiles;
    strips.reserve(d->nseg + d->nseg / 8);
    d->h_tile_frames.clear();
    d->h_tile_segstart.clear();
    TileDesc cur{0, 0, 0, 0};
    bool cur_open = false;
    auto close_tile = [&]() {
        if (cur_open && cur.nstrips) {
            tiles.push_back(cur);
            d->h_tile_frames.push_back(cur.nframes);
        }
        cur_open = false;
    };
    for (size_t s = 0; s < d->nseg; s++) {
        const uint64_t b = d->h_off[s] - d->h_off[0], e = d->h_off[s + 1] - d->h_off[0];
        const uint32_t L = (uint32_t)(e - b);
        for (uint32_t o = 0; o < L; o += kStrip) {
            const uint32_t len = std::min<uint32_t>(kStrip, L - o);
            if (cur_open && cur.nframes + len > (uint32_t)kTileFrames) close_tile();
            if (!cur_open) {
                cur = TileDesc{(uint32_t)(b + o), 0, (uint32_t)strips.size(), 0};
                cur_open = true;
                d->h_tile_segstart.push_back(o == 0 ? 1 : 0);
            }
            StripDesc sd;
            sd.frame_begin = (uint32_t)(b + o);
            sd.seg = (uint32_t)s;
            sd.len_flags = len | (o == 0 ? 1u << 16 : 0u) | (o + len == L ? 1u << 17 : 0u);
            sd.seg_len = L;
            strips.push_back(sd);
            cur.nframes += len;
            cur.nstrips += 1;
        }
    }
    close_tile();
    d->nstrips = (uint32_t)strips.size();
    d->ntiles = (uint32_t)tiles.size();
    static_assert(sizeof(StripDesc) == sizeof(int4) && sizeof(TileDesc) == sizeof(int4), "descriptor size");
    SS_TRY(upload(ctx, d->d_strips, reinterpret_cast<const int4*>(strips.data()), strips.size()));
    SS_TRY(upload(ctx, d->d_tiles, reinterpret_cast<const int4*>(tiles.data()), tiles.size()));
    SS_CUDA(ctx, d->d_stream.reserve(std::max<size_t>(frames, 1) * kSlots));
    SS_CUDA(ctx, d->d_max_norm.reserve(1));
    SS_CUDA(ctx, cudaMemsetAsync(d->d_max_norm.p, 0, sizeof(float), ctx->stream));
    if (frames) {
        k_dict_stream<<<ceil_div((long long)frames, 256), 256, 0, ctx->stream>>>(d->d_mfcc.p, frames, d->c, d->d_stream.p,
                                                                                d->d_max_norm.p);
        SS_LAUNCHED(ctx);
    }
    // the descriptor vectors are read by the async copies above: finish before they go out of scope
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SS_OK;
}

int dtw_queries_build(ss_queries* q) {
    ss_ctx* ctx = q->ctx;
    if (q->lane_built) return SS_OK;
    // sort query ids by length, longest first (heavy CTAs are scheduled first); zero-length queries get no lane
    std::vector<uint32_t> order;
    order.reserve(q->nq);
    for (size_t i = 0; i < q->nq; i++)
        if (q->h_off[i + 1] > q->h_off[i]) order.push_back((uint32_t)i);
    auto len_of = [&](uint32_t i) { return (uint32_t)(q->h_off[i + 1] - q->h_off[i]); };
    std::stable_sort(order.begin(), order.end(), [&](uint32_t x, uint32_t y) { return len_of(x) > len_of(y); });
    std::vector<uint32_t> glen, gbase, gqid;
    uint64_t rows = 0;
    size_t pos = 0;
    while (pos < order.size()) {
        const uint32_t L = len_of(order[pos]);
        size_t end = pos;
        while (end < order.size() && len_of(order[end]) == L) end++;
        for (size_t b = pos; b < end; b += 32) {
            glen.push_back(L);
            gbase.push_back((uint32_t)rows);
            for (size_t l = 0; l < 32; l++) gqid.push_back(b + l < end ? order[b + l] : 0xFFFFFFFFu);
            rows += ((uint64_t)L + 3) / 4 * 4 + 4;  // padded so that any band of <= 4 rows stays in bounds
        }
        pos = end;
    }
    if (rows > 0xFFFFFFF0ull) return set_error(ctx, SS_ERR_INVALID, "query batch too large (%llu lane rows)", (unsigned long long)rows);
    gbase.push_back((uint32_t)rows);
    q->ngroups = (uint32_t)glen.size();
    q->total_rows = rows;
    q->h_group_len = glen;
    SS_TRY(upload(ctx, q->d_group_len, glen.data(), glen.size()));
    SS_TRY(upload(ctx, q->d_group_rowbase, gbase.data(), gbase.size()));
    SS_TRY(upload(ctx, q->d_group_qid, gqid.data(), gqid.size()));
    SS_CUDA(ctx, q->d_lane.reserve(std::max<uint64_t>(rows, 1) * 4 * 32));
    SS_CUDA(ctx, q->d_max_norm.reserve(1));
    SS_CUDA(ctx, cudaMemsetAsync(q->d_max_norm.p, 0, sizeof(float), ctx->stream));
    if (q->ngroups) {
        k_query_lanes<<<q->ngroups, 128, 0, ctx->stream>>>(q->d_mfcc.p, q->d_off.p, q->c, q->d_group_len.p,
                                                          q->d_group_rowbase.p, q->d_group_qid.p, q->ngroups, q->d_lane.p,
                                                          q->d_max_norm.p);
        SS_LAUNCHED(ctx);
    }
    // (the group tables are staged by cudaMemcpyAsync before it returns: no synchronisation needed for the host vectors)
    q->lane_built = true;
    return SS_OK;
}

constexpr int kScanRB = 4;     // query rows per pass of k_dtw_scan (DESIGN.md §3.1c)
constexpr int kScanWaves = 8;  // the fp32 scan's grid: about this many waves at 4 CTAs / SM

template <int KP, bool TARGET>
static int launch_scan_merge(ss_dict* d, const ScanParams& p, const ScanTarget& tg, uint32_t grid, uint32_t nslots, bool timed) {
    ss_ctx* ctx = d->ctx;
    if (timed) SS_CUDA(ctx, cudaEventRecord(d->ev_scan0, ctx->stream));
    SS_CUDA(ctx, cudaFuncSetAttribute(k_dtw_scan<kScanRB, KP, TARGET>, cudaFuncAttributeMaxDynamicSharedMemorySize, kScanSmemBytes));
    k_dtw_scan<kScanRB, KP, TARGET><<<grid, kWarpsPerCta * 32, kScanSmemBytes, ctx->stream>>>(p, tg);
    SS_LAUNCHED(ctx);
    if (timed) {
        SS_CUDA(ctx, cudaEventRecord(d->ev_scan1, ctx->stream));
        d->scan_timed = true;
    }
    k_dtw_merge<KP><<<ceil_div(nslots, 128), 128, 0, ctx->stream>>>(d->d_partial.p, p.nslices, nslots, d->d_cand_idx.p, d->d_cand_adist.p);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

// the fp32 CUDA-core scan of batch q, its f64 refine and certification (any sequence length). target: the SS_DTW_TARGET form,
// d_targets in q's order (NULL: t = 0)
static int dtw_fp32_match(ss_dict* d, ss_queries* q, int k, bool timed, uint32_t* d_out_idx, double* d_out_dist, bool target = false,
                          const double* d_targets = nullptr) {
    ss_ctx* ctx = d->ctx;
    SS_TRY(dtw_queries_build(q));
    const int kp = k <= 2 ? 4 : (k <= 6 ? 8 : 16);  // candidates kept per query by the scan
    const uint32_t nslots = q->ngroups * 32;

    // ---- slices: contiguous tile ranges starting at segment boundaries, balanced by frames ------------------------
    const uint32_t nqb = (q->ngroups + kWarpsPerCta - 1) / kWarpsPerCta;
    uint32_t nslices = 1;
    if (nqb && d->ntiles) {
        const uint32_t target_ctas = (uint32_t)ctx->sm_count * 4 * kScanWaves;
        nslices = std::max<uint32_t>(1, std::min<uint32_t>(d->ntiles, (target_ctas + nqb - 1) / nqb));
    }
    std::vector<uint32_t>& st = d->h_slice_tile;
    st.clear();
    st.push_back(0);
    if (d->ntiles) {
        const uint64_t per = (d->total_frames + nslices - 1) / nslices;
        uint64_t acc = 0;
        for (uint32_t t = 0; t < d->ntiles; t++) {
            if (t > 0 && d->h_tile_segstart[t] && st.size() < nslices && acc >= (uint64_t)st.size() * per) st.push_back(t);
            acc += d->h_tile_frames[t];
        }
    }
    st.push_back(d->ntiles);
    nslices = (uint32_t)st.size() - 1;
    SS_TRY(upload(ctx, d->d_slice_tile, st.data(), st.size()));

    SS_CUDA(ctx, d->d_partial.reserve(std::max<size_t>((size_t)nslices * nslots * kp, 1)));
    SS_CUDA(ctx, d->d_cand_idx.reserve(std::max<size_t>((size_t)nslots * kp, 1)));
    SS_CUDA(ctx, d->d_cand_adist.reserve(std::max<size_t>((size_t)nslots * kp, 1)));

    if (nqb) {
        const uint32_t grid = nqb * nslices;
        ScanParams p;
        p.qlane = q->d_lane.p;
        p.group_len = q->d_group_len.p;
        p.group_rowbase = q->d_group_rowbase.p;
        p.ngroups = q->ngroups;
        p.stream = d->d_stream.p;
        p.strips = d->d_strips.p;
        p.tiles = d->d_tiles.p;
        p.slice_tile = d->d_slice_tile.p;
        p.nslices = nslices;
        p.partial = d->d_partial.p;
        p.scratch = nullptr;
        p.scratch_rows = 0;
        if (d->max_len > (uint32_t)kStrip) {  // boundary columns of multi-strip segments
            p.scratch_rows = (q->max_len + 3) / 4 * 4 + 4;
            SS_CUDA(ctx, d->d_scratch.reserve((size_t)grid * p.scratch_rows * 128));
            p.scratch = d->d_scratch.p;
        }
        const ScanTarget tg = {d_targets, q->d_group_qid.p, q->d_max_norm.p, d->d_max_norm.p, d->dtw_band};
        if (!d->ev_scan0) {
            SS_CUDA(ctx, cudaEventCreate(&d->ev_scan0));
            SS_CUDA(ctx, cudaEventCreate(&d->ev_scan1));
        }
        if (kp == 4) SS_TRY((target ? launch_scan_merge<4, true> : launch_scan_merge<4, false>)(d, p, tg, grid, nslots, timed));
        else if (kp == 8) SS_TRY((target ? launch_scan_merge<8, true> : launch_scan_merge<8, false>)(d, p, tg, grid, nslots, timed));
        else SS_TRY((target ? launch_scan_merge<16, true> : launch_scan_merge<16, false>)(d, p, tg, grid, nslots, timed));
    }
    // fp32 scan: |error| of a normalised distance <= 4e-6 (max|a|^2 + max|b|^2)  (14 roundings of 2^-24 on terms <= 2(|a|^2+|b|^2);
    // the running sum along the path is not counted: DESIGN.md §3.1h). The TARGET keys carry their own bound.
    return dtw_rescore_finalize(d, q, k, kp, nslots, q->d_group_qid.p, 4e-6, q->d_max_norm.p, d->d_max_norm.p, nullptr, 0, q->d_uncert_flag.p,
                                d_out_idx, d_out_dist, target, d_targets);
}

// ---------------------------------------------------------------------------------------------------------------
// the stage cascade
// ---------------------------------------------------------------------------------------------------------------
// Each stage only runs for the queries the previous one could not certify; its bound decides which:
//   H2          packed-half tensor-core scan + second chance   dtw_h2.cu   bound: triangle inequality on the rounded frames
//   H2_WIDE     the same scan with 32 candidates per query      dtw_h2.cu
//   TC          fp32-DP tensor-core scan (<= 32 x <= 32 frames) dtw_tc.cu   bound: as H2
//   FP32        fp32 CUDA-core scan (any length)                k_dtw_scan  bound: 4e-6 (max|a|^2 + max|b|^2)
//   EXHAUSTIVE  f64 DTW against every segment                   exact.cu    exact by construction
// EXHAUSTIVE only triggers when more than KP segments are closer to each other than the scans can resolve (e.g. many
// near-identical dictionary entries); it guarantees that what ss_dict_match returns is THE f64 top-k.
//
// dtw_match_dev enqueues the first stage and returns without a host round trip: the whole step (layout kernel, scan, merge,
// refine) is in the stream before the GPU has started on it. Whether a later stage is needed is only known once the refine
// has run; dtw_match_finish waits for that (one event) and runs the later stages synchronously for the few queries
// concerned. Every reader of the results or of the last_* counters goes through dtw_match_finish first.

static const char* stage_name(DtwStage s) {
    static const char* const names[] = {"packed-half", "packed-half, 32 candidates", "fp32-DP tensor-core", "fp32 CUDA-core", "exhaustive f64"};
    return names[(int)s];
}

// The first stage: the ss_dict_set_scan preference, then what applies to the shapes
static DtwStage first_stage(const ss_dict* d, const ss_queries* q) {
    if ((d->scan_pref == 0 || d->scan_pref == 3) && dtw_h2_applies(d, q)) return DtwStage::H2;
    if (d->scan_pref != 2 && dtw_tc_applies(d, q)) return DtwStage::TC;
    return DtwStage::FP32;
}

// Whether later stage s applies to the uncertified queries (gathered into sub) after stage prev ran. H2_WIDE is only ever
// tried right after H2, and it replaces TC: it is for sequences of more than 32 frames, which TC does not take.
static bool later_stage_applies(const ss_dict* d, const ss_queries* sub, DtwStage prev, DtwStage s) {
    if (s == DtwStage::H2_WIDE) return dtw_h2_applies(d, sub) && (d->max_len > 32 || sub->max_len > 32);
    if (s == DtwStage::TC) return prev != DtwStage::H2_WIDE && dtw_tc_applies(d, sub);
    return true;
}

// runs one filter stage on batch q: scan, merge, f64 refine, certification (q->d_uncert_flag, d_counters[0]); only the
// first stage of a match records the scan-time events
static int run_stage(ss_dict* d, ss_queries* q, int k, DtwStage s, bool timed, uint32_t* d_out_idx, double* d_out_dist) {
    const bool second_chance = d->scan_pref != 3;
    switch (s) {
    case DtwStage::H2: return dtw_h2_match_dev(d, q, k, /*wide=*/false, second_chance, timed, d_out_idx, d_out_dist);
    case DtwStage::H2_WIDE: return dtw_h2_match_dev(d, q, k, /*wide=*/true, second_chance, timed, d_out_idx, d_out_dist);
    case DtwStage::TC: return dtw_tc_match_dev(d, q, k, timed, d_out_idx, d_out_dist);
    default: return dtw_fp32_match(d, q, k, timed, d_out_idx, d_out_dist);
    }
}

// Sequences of more than 32 frames have no cheap second filter (the fp32-DP tensor-core scan stops at 32 frames, the CUDA-core
// scan of ONE long query is a single warp's serial walk: 16 ms at config 5): below 2e8 cells the exhaustive stage is the
// fastest way to finish (f64, measured 9e10 cells / s: 2 ms); a dozen such queries first take the wide packed-half pass.
// Cells the banded strip kernel (exact.cu warp_dtw_exact_long with BAND) visits for a pair of la x lb frames (la, lb >= 1): per strip of
// 32 columns, the 32 x 32 step blocks from the one holding its first in-band row to the one in which lane 31 reaches its last.
static uint64_t band_strip_cells(int la, int lb, uint32_t r) {
    const int nsteps = la + 31;
    uint64_t blocks = 0;
    for (int s = 0; s < (lb + 31) / 32; s++) {
        int lo, hi, lo_last, hi_last;
        band_rows(32 * s, la, lb, r, &lo, &hi);
        band_rows(std::min(32 * s + 31, lb - 1), la, lb, r, &lo_last, &hi_last);
        blocks += (std::min(nsteps, hi_last + 32) - (lo & ~31) + 31) / 32;
    }
    return blocks * 32 * 32;
}

// ran_max_len: the longest query of the batch the last stage ran on; u: the uncertified queries of q.
// With a band, a pair costs what the banded strip kernel visits (band_strip_cells), but never more than its Lq Ld cells.
static bool exhaustive_is_cheaper(const ss_dict* d, uint32_t ran_max_len, const ss_queries* q, const std::vector<uint32_t>& u) {
    if (d->max_len <= 32 && ran_max_len <= 32) return false;
    const uint64_t limit = 200000000ull;
    uint64_t cells = 0;
    for (uint32_t i : u) {
        const uint64_t lq = q->h_off[i + 1] - q->h_off[i];
        if (!d->dtw_band || !lq) {
            cells += lq * d->total_frames;
            continue;
        }
        for (size_t s = 0; s < d->nseg && cells <= limit; s++) {
            const uint64_t ld = d->h_off[s + 1] - d->h_off[s];
            if (ld) cells += std::min<uint64_t>(lq * ld, band_strip_cells((int)lq, (int)ld, d->dtw_band));
        }
        if (cells > limit) return false;
    }
    return cells <= limit;
}

// the uncertified count of the stage that just ran travels to pinned host memory behind it; ev_done marks its arrival
static int post_counters(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    if (!d->h_counters) {
        if (!ctx->pinned_free.empty()) {  // (a block a destroyed dictionary of this ctx handed back)
            d->h_counters = static_cast<unsigned long long*>(ctx->pinned_free.back());
            ctx->pinned_free.pop_back();
        } else {
            SS_CUDA(ctx, cudaHostAlloc((void**)&d->h_counters, 4 * sizeof(unsigned long long), cudaHostAllocDefault));
        }
        SS_CUDA(ctx, cudaEventCreateWithFlags(&d->ev_done, cudaEventDisableTiming));
    }
    SS_CUDA(ctx, d->d_counters.reserve(4));
    SS_CUDA(ctx, cudaMemcpyAsync(d->h_counters, d->d_counters.p, 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaEventRecord(d->ev_done, ctx->stream));
    return SS_OK;
}

// The queries batch `ran` could not certify, as ids of the caller's batch: ids[i] for query i of `ran` (i itself when ids
// is null). Called once ev_done has been reached; synchronous when there are any.
static int read_uncertified(ss_dict* d, const ss_queries* ran, const std::vector<uint32_t>* ids, std::vector<uint32_t>* out) {
    ss_ctx* ctx = d->ctx;
    std::vector<uint32_t> u;
    if (d->h_counters[0]) {
        std::vector<uint8_t> flags(ran->nq);
        SS_CUDA(ctx, cudaMemcpyAsync(flags.data(), ran->d_uncert_flag.p, ran->nq, cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        for (size_t i = 0; i < ran->nq; i++)
            if (flags[i]) u.push_back(ids ? (*ids)[i] : (uint32_t)i);
    }
    out->swap(u);
    return SS_OK;
}

// target (SS_DTW_TARGET, DESIGN.md §3.1h): the cascade is FP32 -> EXHAUSTIVE, the scan's TARGET form first whatever ss_dict_set_scan
// chose (the tensor-core scans' bounds are one-sided or too wide); d_targets (q's order, NULL: t = 0) is read until dtw_match_finish.
int dtw_match_dev(ss_dict* d, ss_queries* q, int k, uint32_t* d_out_idx, double* d_out_dist, bool target, const double* d_targets) {
    ss_ctx* ctx = d->ctx;
    if (k < 1 || k > SS_MAX_TOPK) return set_error(ctx, SS_ERR_INVALID, "k must be in 1..%d (got %d)", SS_MAX_TOPK, k);
    SS_TRY(dtw_match_finish(d));  // the previous match shares this dictionary's workspaces
    SS_CUDA(ctx, q->d_uncert_flag.reserve(std::max<size_t>(q->nq, 1)));
    SS_CUDA(ctx, cudaMemsetAsync(q->d_uncert_flag.p, 0, std::max<size_t>(q->nq, 1), ctx->stream));
    const DtwStage first = target ? DtwStage::FP32 : first_stage(d, q);
    d->last_scan_kind = first == DtwStage::H2 ? 1 : (first == DtwStage::TC ? 2 : 3);
    d->last_work = d->total_frames * q->total_frames;
    d->last_tc_fallback = 0;
    d->last_exhaustive = 0;
    d->last_uncertified = q->nq;  // no row is final before dtw_match_finish
    if (target) SS_TRY(dtw_fp32_match(d, q, k, /*timed=*/true, d_out_idx, d_out_dist, true, d_targets));
    else SS_TRY(run_stage(d, q, k, first, /*timed=*/true, d_out_idx, d_out_dist));
    SS_TRY(post_counters(d));
    d->pending.active = true;
    d->pending.target = target;
    d->pending.d_targets = d_targets;
    d->pending.first = first;
    d->pending.q = q;
    d->pending.k = k;
    d->pending.d_out_idx = d_out_idx;
    d->pending.d_out_dist = d_out_dist;
    return SS_OK;
}

// ---- running a few queries through the later stages -----------------------------------------------------------------------
// The queries a stage could not certify are gathered (on the device) into a small batch of their own for the next stage;
// their rows are scattered back into the caller's result arrays. At config 4 without the second chance this is ~50 of the
// 10 000 queries: one group of 128 for the fp32-DP tensor-core scan (~0.6 ms) instead of a scan of the whole batch.
__global__ void k_gather_query_rows(const double* __restrict__ src, const uint64_t* __restrict__ src_off, const uint32_t* __restrict__ ids,
                                    const uint64_t* __restrict__ dst_off, int c, double* __restrict__ dst) {
    const uint32_t i = blockIdx.x;
    const double* from = src + src_off[ids[i]] * c;
    double* to = dst + dst_off[i] * c;
    const size_t n = (size_t)(dst_off[i + 1] - dst_off[i]) * c;
    for (size_t e = threadIdx.x; e < n; e += blockDim.x) to[e] = from[e];
}
__global__ void k_scatter_topk(const uint32_t* __restrict__ sub_idx, const double* __restrict__ sub_dist, const uint32_t* __restrict__ ids, uint32_t nsub,
                               int k, uint32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nsub * (uint32_t)k) return;
    const uint32_t i = t / (uint32_t)k, s = t % (uint32_t)k;
    out_idx[(size_t)ids[i] * k + s] = sub_idx[t];
    out_dist[(size_t)ids[i] * k + s] = sub_dist[t];
}

// queries `ids` of q -> the dictionary's sub-batch d->sub_q (refilled: no layout of its previous contents is kept), ids in
// d_sub_ids, room for its results in d_sub_idx / d_sub_dist
static int gather_queries(ss_dict* d, ss_queries* q, const std::vector<uint32_t>& ids, int k) {
    ss_ctx* ctx = d->ctx;
    if (!d->sub_q) {
        d->sub_q = new (std::nothrow) ss_queries();
        if (!d->sub_q) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
        d->sub_q->ctx = ctx;
        d->sub_q->c = d->c;
    }
    ss_queries* sub = d->sub_q;
    const size_t ns = ids.size();
    std::vector<uint64_t> off(ns + 1, 0);
    for (size_t i = 0; i < ns; i++) off[i + 1] = off[i] + (q->h_off[ids[i] + 1] - q->h_off[ids[i]]);
    SS_TRY(queries_prepare(sub, off.data(), ns));
    SS_TRY(upload(ctx, sub->d_off, sub->h_off.data(), ns + 1));
    SS_TRY(upload(ctx, d->d_sub_ids, ids.data(), ns));
    SS_CUDA(ctx, sub->d_mfcc.reserve(std::max<size_t>((size_t)sub->total_frames * sub->c, 1)));
    k_gather_query_rows<<<(unsigned)ns, 128, 0, ctx->stream>>>(q->d_mfcc.p, q->d_off.p, d->d_sub_ids.p, sub->d_off.p, q->c, sub->d_mfcc.p);
    SS_LAUNCHED(ctx);
    SS_TRY(dtw_tc_queries_group(sub));
    SS_CUDA(ctx, sub->d_uncert_flag.reserve(ns));
    SS_CUDA(ctx, cudaMemsetAsync(sub->d_uncert_flag.p, 0, ns, ctx->stream));
    SS_CUDA(ctx, d->d_sub_idx.reserve(ns * (size_t)k));
    SS_CUDA(ctx, d->d_sub_dist.reserve(ns * (size_t)k));
    return SS_OK;
}

// The later stages of the pending match. d->last_uncertified follows the number of queries whose rows are not final, so
// that it is right also when a stage fails.
static int run_later_stages(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    ss_queries* q = d->pending.q;
    const int k = d->pending.k;
    uint32_t* out_idx = d->pending.d_out_idx;
    double* out_dist = d->pending.d_out_dist;
    DtwStage s = d->pending.first;
    uint32_t ran_max_len = q->max_len;
    std::vector<uint32_t> u;  // the queries of q whose rows are not final
    TraceTimer tt(ctx);
    auto trace = [&](DtwStage st) {
        tt.lap(stage_name(st));
        if (dtw_trace()) fprintf(stderr, "[ss dtw trace]   -> %zu of %zu still uncertified\n", u.size(), q->nq);
    };
    SS_CUDA(ctx, cudaEventSynchronize(d->ev_done));
    SS_TRY(read_uncertified(d, q, nullptr, &u));
    trace(s);
    d->last_uncertified = u.size();
    if (s != DtwStage::FP32) d->last_tc_fallback = u.size();
    while (!u.empty()) {
        if (s == DtwStage::FP32 || exhaustive_is_cheaper(d, ran_max_len, q, u)) {
            d->last_exhaustive += u.size();
            SS_TRY(dtw_exhaustive_match(d, q, k, u, out_idx, out_dist, d->pending.target, d->pending.d_targets));
            u.clear();
            trace(DtwStage::EXHAUSTIVE);
            break;
        }
        SS_TRY(gather_queries(d, q, u, k));
        ss_queries* sub = d->sub_q;
        const DtwStage prev = s;
        do s = (DtwStage)((int)s + 1);
        while (!later_stage_applies(d, sub, prev, s));
        SS_TRY(run_stage(d, sub, k, s, /*timed=*/false, d->d_sub_idx.p, d->d_sub_dist.p));
        k_scatter_topk<<<ceil_div((long long)u.size() * k, 128), 128, 0, ctx->stream>>>(d->d_sub_idx.p, d->d_sub_dist.p, d->d_sub_ids.p,
                                                                                      (uint32_t)u.size(), k, out_idx, out_dist);
        SS_LAUNCHED(ctx);
        SS_TRY(post_counters(d));
        SS_CUDA(ctx, cudaEventSynchronize(d->ev_done));
        SS_TRY(read_uncertified(d, sub, &u, &u));
        ran_max_len = sub->max_len;
        trace(s);
        d->last_uncertified = u.size();
    }
    d->last_uncertified = 0;
    return SS_OK;
}

int dtw_match_finish(ss_dict* d) {
    if (!d->pending.active) return SS_OK;
    const int rc = run_later_stages(d);
    d->pending = ss_dict::Pending();  // (after a failure too: the next match can run, and last_uncertified is not 0)
    return rc;
}

}  // namespace ss
