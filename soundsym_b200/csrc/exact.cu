// exact.cu — f64 kernels whose arithmetic must equal the CPU path operation for operation. This translation unit is
// compiled with --fmad=false so that a*b+c stays a rounded multiply followed by a rounded add, as rustc emits it.
//
//   cosine-ref matcher   cosine_sim / norm / at_distance, src/sound.rs:23-38, 351-370 (+ rulinalg::utils::dot [RECALL A9])
//   DTW refine           the oracle's f64 recurrence (ASSUMPTIONS.h A8) on the candidates the fp32 scan kept
//   top-k merge          (distance, index) lexicographic merge of per-shard lists
//   DTW alignment        the refine's recurrence with the direction of every cell kept, then the backtrack (DESIGN.md §3.1e)
#include <cub/cub.cuh>

#include <algorithm>

#include "match.cuh"

namespace ss {

constexpr double kInf = __builtin_huge_val();

// ---------------------------------------------------------------------------------------------------------------
// norm(me) = fold(0, |memo, item| item*item + memo)   src/sound.rs:36-38 — one thread per segment, sequential
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_seg_norm(const double* __restrict__ v, const uint64_t* __restrict__ off, size_t nseg, int c,
                           double* __restrict__ out) {
    const size_t s = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= nseg) return;
    const double* p = v + off[s] * c;
    const size_t n = (size_t)(off[s + 1] - off[s]) * c;
    double memo = 0.0;
    for (size_t i = 0; i < n; i++) memo = p[i] * p[i] + memo;
    out[s] = memo;
}

// f64 lane layout for the cosine matcher: element e of query lane l of group g at [(rowbase*c + e) * 32 + l]
__global__ void k_query_lanes64(const double* __restrict__ mfcc, const uint64_t* __restrict__ off, int c,
                                const uint32_t* __restrict__ group_len, const uint32_t* __restrict__ group_rowbase,
                                const uint32_t* __restrict__ group_qid, double* __restrict__ lanes) {
    const uint32_t g = blockIdx.x;
    const int lane = threadIdx.x & 31;
    const uint32_t n = group_len[g] * (uint32_t)c;
    const uint32_t qid = group_qid[g * 32 + lane];
    double* dst = lanes + (size_t)group_rowbase[g] * c * 32 + lane;
    const double* src = qid != 0xFFFFFFFFu ? mfcc + off[qid] * c : nullptr;
    for (uint32_t e = threadIdx.x >> 5; e < n; e += blockDim.x >> 5) dst[(size_t)e * 32] = src ? src[e] : 0.0;
}

// one thread per (query, dictionary segment) pair: lanes are 32 equal-length queries, the dictionary segments are
// warp-uniform. Accumulation order is rulinalg's dot (A9): p_u += x[8c+u] * y[8c+u] chunk by chunk, then
// (p0+p4) + (p1+p5) + (p2+p6) + (p3+p7), then the scalar tail — per pair exactly as the CPU path; products and sums are
// rounded separately (--fmad=false), so one DMUL + one DADD per product on the FP64 pipe is the floor.
//
// The kernel walks the dictionary in (length, index) order (CosSeg table, built once per dictionary): a CTA stages
// kCosStage consecutive segments of that order in shared memory and consumes them G = 4 at a time — almost always four
// segments of the SAME length, so that all pairs of a thread run the same number of chunks and the chunk loop is
// branch-free straight-line code. A warp works on NQ query groups of one length at once (a "work item", table built per
// query batch): NQ = 2 wherever two groups of a length exist, NQ = 1 for the odd group of a length. With NQ = 2 a thread
// holds 2 queries x 4 segments = 64 partial sums: the 16 broadcast LDS.128 of a chunk feed 128 FP64 instructions instead
// of 64 (1.0 instead of 1.5 L1 wavefronts per product), and the query chunk is refilled IN PLACE — element pair v of the
// next chunk is loaded as soon as pair v of the current chunk has been consumed, a whole chunk (128 FP64 instructions)
// ahead of its use — so the 128 accumulator registers leave room for it without a second buffer. NQ = 1 keeps two
// register buffers, two chunks per iteration. Staging is asynchronous (cp.async into the other half of a double buffer
// while the current group is consumed, descriptors two groups ahead): one barrier per group and no exposed global
// latency. Slice `sl` takes groups sl, sl + nslices, ... — every slice sees the same mix of lengths. Because the walk is
// not in index order, the reference's "first minimum wins" (strict '<' in index order, src/sound.rs:361-366) is carried by
// an explicit (distance, index) comparison.
constexpr int kCosG = 4;        // segments in flight per thread
constexpr int kCosStage = 8;    // segments staged per barrier (a multiple of kCosG: consumed kCosG at a time)
constexpr int kCosWarps = 4;    // work items per CTA
// Measured at config 4 and NOT kept (45.0 ms for NQ = 1 everywhere, the state before the 2 x 4 tile):
//   two warps of a CTA on the same 32 queries, each on its own kCosG of a stage, so that the second warp's query loads
//   hit L1 (halves the 7.4 TB/s query stream from L2)                                                              49.9 ms
//   query chunks fetched two chunks ahead through three register buffers                                          46.9 ms
//   255 registers, 8 warps / SM (with two / three buffers)                                                 46.7 / 46.3 ms
//   four segments per barrier                                                                                     46.6 ms
// and with the 2 x 4 tile (39.5 ms):
//   one prefetch.global.L1 (CCTL.PF1) per chunk, lane l on line l of the two groups' chunk two / three chunks ahead     46.4 ms
// - neither the L2 -> SM traffic nor the load latency is what the NQ = 1 chunk loop waits for: the L1 data pipe is 66 % busy
// (a broadcast LDS.128 costs two wavefronts, a coalesced LDG.64 two), the FP64 pipe 44 %.
constexpr int kCosSegCap = 512; // doubles of shared memory per staged segment (longer segments are read from global memory)
constexpr uint32_t kCosNone = 0xFFFFFFFFu;

__device__ __forceinline__ void cos_cp_async8(double* smem_dst, const double* gsrc) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(d), "l"(gsrc) : "memory");
}
__device__ __forceinline__ void cos_cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }

// the 8 partial sums of all NQ x G pairs advance by one chunk: yv = the queries' 8 values, xs = chunk of segment 0 in shared memory
template <int NQ>
__device__ __forceinline__ void cos_chunk(double (&p)[NQ][kCosG][8], const double (&yv)[NQ][8], const double2* xs) {
#pragma unroll
    for (int u = 0; u < kCosG; u++) {
#pragma unroll
        for (int v = 0; v < 4; v++) {
            const double2 xx = xs[u * (kCosSegCap / 2) + v];
#pragma unroll
            for (int q = 0; q < NQ; q++) {
                p[q][u][2 * v] = p[q][u][2 * v] + xx.x * yv[q][2 * v];
                p[q][u][2 * v + 1] = p[q][u][2 * v + 1] + xx.y * yv[q][2 * v + 1];
            }
        }
    }
}

// rulinalg's combine of the 8 partial sums, then the scalar tail (elements 8 nch .. len - 1: yt = the queries' chunk nch,
// xs = that chunk of segment 0 in shared memory), per pair in the CPU path's order
template <int NQ>
__device__ __forceinline__ void cos_finish(const double (&p)[NQ][kCosG][8], double (&sum)[NQ][kCosG], const double (&yt)[NQ][8],
                                           const double2* xs, uint32_t ntail) {
#pragma unroll
    for (int q = 0; q < NQ; q++) {
#pragma unroll
        for (int u = 0; u < kCosG; u++) {
            sum[q][u] = 0.0 + (p[q][u][0] + p[q][u][4]);
            sum[q][u] = sum[q][u] + (p[q][u][1] + p[q][u][5]);
            sum[q][u] = sum[q][u] + (p[q][u][2] + p[q][u][6]);
            sum[q][u] = sum[q][u] + (p[q][u][3] + p[q][u][7]);
        }
    }
#pragma unroll
    for (int j = 0; j < 7; j++) {
        if ((uint32_t)j < ntail) {  // warp-uniform
#pragma unroll
            for (int u = 0; u < kCosG; u++) {
                const double xv = reinterpret_cast<const double*>(xs + u * (kCosSegCap / 2))[j];
#pragma unroll
                for (int q = 0; q < NQ; q++) sum[q][u] = sum[q][u] + xv * yt[q][j];
            }
        }
    }
}

struct CosShared {
    uint4 sdesc[3][kCosStage];  // {first frame lo, hi, frames, local segment index}
    double snorm[3][kCosStage];
};

// one CTA = kCosWarps work items (NQ query groups of one length each) x one slice of the dictionary's staged groups
template <int NQ>
__device__ __forceinline__ void cos_scan_body(double (*sseg)[kCosStage][kCosSegCap], CosShared& sh, const double* __restrict__ dmfcc,
                                              const uint4* __restrict__ cseg, const double* __restrict__ cnorm, uint32_t nseg, int c,
                                              uint32_t nslices, uint32_t slice, const double* __restrict__ qlanes,
                                              const uint32_t* __restrict__ group_len, const uint32_t* __restrict__ group_rowbase,
                                              const uint32_t* __restrict__ group_qid, uint32_t ngroups, const double* __restrict__ qnorm,
                                              const double* __restrict__ targets, double* __restrict__ part_dist,
                                              uint32_t* __restrict__ part_idx, const uint2* __restrict__ item) {
    const int lane = threadIdx.x & 31;
    const bool active = item != nullptr;  // warp-uniform
    uint32_t g[NQ], qid[NQ], best_idx[NQ];
    const double* y[NQ];
    double nq[NQ], target[NQ], best[NQ];
    {
        const uint2 it = active ? __ldg(item) : make_uint2(0, 0);
#pragma unroll
        for (int q = 0; q < NQ; q++) {
            g[q] = q == 0 ? it.x : it.y;
            qid[q] = active ? group_qid[g[q] * 32 + lane] : kCosNone;
            y[q] = active ? qlanes + (size_t)group_rowbase[g[q]] * c * 32 + lane : qlanes;
            nq[q] = qid[q] != kCosNone ? qnorm[qid[q]] : 1.0;
            target[q] = (qid[q] != kCosNone && targets) ? targets[qid[q]] : 1.0;
            best[q] = 2.0;  // fold((0, 2.0)), src/sound.rs:361
            best_idx[q] = kCosNone;
        }
    }
    const uint32_t kq = active ? group_len[g[0]] * (uint32_t)c : 0;  // the groups of an item have one length
    const uint32_t ngrp = (nseg + kCosStage - 1) / kCosStage;
    // strict '<' in index order (src/sound.rs:362): a smaller distance wins, an equal one only with a smaller index than a
    // winner already found; NaN never wins, 2.0 never beats the fold's seed
    auto consider = [&](int q, double dist, uint32_t idx) {
        if (dist < best[q] || (dist == best[q] && idx < best_idx[q] && best_idx[q] != kCosNone)) {
            best[q] = dist;
            best_idx[q] = idx;
        }
    };

    // descriptor of sorted position grp * kCosStage + t (thread t < kCosStage), absent beyond the table
    auto fetch = [&](uint32_t grp, uint4& dsc, double& nrm) {
        const uint64_t s = (uint64_t)grp * kCosStage + threadIdx.x;
        dsc = make_uint4(0, 0, 0, kCosNone);
        nrm = 1.0;
        if (threadIdx.x < kCosStage && s < nseg) {
            dsc = __ldg(&cseg[s]);
            nrm = __ldg(&cnorm[s]);
        }
    };
    auto stage = [&](int slot, int b) {
#pragma unroll
        for (int u = 0; u < kCosStage; u++) {
            const uint4 dsc = sh.sdesc[slot][u];
            const uint32_t kd = dsc.z * (uint32_t)c;
            if (dsc.w != kCosNone && kd <= (uint32_t)kCosSegCap) {
                const double* src = dmfcc + (((uint64_t)dsc.y << 32) | dsc.x) * c;
                for (uint32_t e = threadIdx.x; e < kd; e += 32 * kCosWarps) cos_cp_async8(&sseg[b][u][e], src + e);
            }
        }
    };
    {
        uint4 d0, d1;
        double n0, n1;
        fetch(slice, d0, n0);
        fetch(slice + nslices, d1, n1);
        if (threadIdx.x < kCosStage) {
            sh.sdesc[0][threadIdx.x] = d0, sh.snorm[0][threadIdx.x] = n0;
            sh.sdesc[1][threadIdx.x] = d1, sh.snorm[1][threadIdx.x] = n1;
        }
        __syncthreads();
        stage(0, 0);
    }
    int cur = 0, b = 0;  // descriptor slot and staging buffer of the current group
    for (uint32_t grp = slice; grp < ngrp; grp += nslices) {
        const int nxt = cur == 2 ? 0 : cur + 1, nxt2 = nxt == 2 ? 0 : nxt + 1;
        cos_cp_async_wait_all();
        __syncthreads();  // buffer b and descriptor slot nxt are complete; everyone is done with buffer b ^ 1 and slot nxt2
        stage(nxt, b ^ 1);
        uint4 d2;
        double n2;
        fetch(grp + 2 * nslices, d2, n2);
        if (active) {
#pragma unroll 1
          for (int u0 = 0; u0 < kCosStage; u0 += kCosG) {
            uint32_t kd[kCosG], sidx[kCosG], len[kCosG], nchunk[kCosG];
            const double* xg[kCosG];
            double p[NQ][kCosG][8];
            bool uniform = true, all_staged = true;
            uint32_t maxchunk = 0;
#pragma unroll
            for (int u = 0; u < kCosG; u++) {
                const uint4 dsc = sh.sdesc[cur][u0 + u];
                sidx[u] = dsc.w;
                kd[u] = dsc.w != kCosNone ? dsc.z * (uint32_t)c : 0;
                xg[u] = dmfcc + (((uint64_t)dsc.y << 32) | dsc.x) * c;
                len[u] = kd[u] < kq ? kd[u] : kq;
                nchunk[u] = len[u] / 8;
                maxchunk = nchunk[u] > maxchunk ? nchunk[u] : maxchunk;
                uniform = uniform && dsc.w != kCosNone && kd[u] == kd[0];
                all_staged = all_staged && kd[u] <= (uint32_t)kCosSegCap;
#pragma unroll
                for (int q = 0; q < NQ; q++) {
#pragma unroll
                    for (int v = 0; v < 8; v++) p[q][u][v] = 0.0;
                }
            }
            const double2* xs = reinterpret_cast<const double2*>(&sseg[b][u0][0]);
            if (uniform && all_staged) {
                // ---- four segments of one length: straight-line chunks -------------------------------------------------------
                // (query loads may run up to a chunk past the query's last element - the chunk that holds the tail: the lane
                // buffer is padded, values beyond the tail go unused)
                const uint32_t nch = nchunk[0], ntail = len[0] - nch * 8;
                double sum[NQ][kCosG];
                if constexpr (NQ == 1) {
                    // two register buffers, two chunks per iteration (no register copies)
                    const double* yp = y[0];
                    double ya[1][8], yb[1][8];
#pragma unroll
                    for (int v = 0; v < 8; v++) ya[0][v] = yp[v * 32];
                    uint32_t ch = 0;
                    for (; ch + 2 <= nch; ch += 2) {
#pragma unroll
                        for (int v = 0; v < 8; v++) yb[0][v] = yp[(8 + v) * 32];
                        cos_chunk<1>(p, ya, xs);
#pragma unroll
                        for (int v = 0; v < 8; v++) ya[0][v] = yp[(16 + v) * 32];
                        cos_chunk<1>(p, yb, xs + 4);
                        yp += 16 * 32;
                        xs += 8;
                    }
                    // the chunk after the last whole one holds the <= 7 tail elements: it is in registers by the time the sums
                    // are combined (a tail read from global memory element by element was 9 % of the kernel's stall samples);
                    // the four tails advance together, then the four divisions
                    if (ch < nch) {
#pragma unroll
                        for (int v = 0; v < 8; v++) yb[0][v] = yp[(8 + v) * 32];
                        cos_chunk<1>(p, ya, xs);
                        cos_finish<1>(p, sum, yb, xs + 4, ntail);
                    } else {
                        cos_finish<1>(p, sum, ya, xs, ntail);
                    }
                } else {
                    // one register buffer refilled in place: pair v of the next chunk is requested right after pair v of the
                    // current chunk has served all NQ x G pairs
                    const double* yp[NQ];
                    double yv[NQ][8];
#pragma unroll
                    for (int q = 0; q < NQ; q++) {
                        yp[q] = y[q];
#pragma unroll
                        for (int v = 0; v < 8; v++) yv[q][v] = yp[q][v * 32];
                    }
                    for (uint32_t ch = 0; ch < nch; ch++) {
#pragma unroll
                        for (int q = 0; q < NQ; q++) yp[q] += 8 * 32;
#pragma unroll
                        for (int v = 0; v < 4; v++) {
#pragma unroll
                            for (int u = 0; u < kCosG; u++) {
                                const double2 xx = xs[u * (kCosSegCap / 2) + v];
#pragma unroll
                                for (int q = 0; q < NQ; q++) {
                                    p[q][u][2 * v] = p[q][u][2 * v] + xx.x * yv[q][2 * v];
                                    p[q][u][2 * v + 1] = p[q][u][2 * v + 1] + xx.y * yv[q][2 * v + 1];
                                }
                            }
#pragma unroll
                            for (int q = 0; q < NQ; q++) {
                                yv[q][2 * v] = yp[q][(2 * v) * 32];
                                yv[q][2 * v + 1] = yp[q][(2 * v + 1) * 32];
                            }
                        }
                        xs += 4;
                    }
                    cos_finish<NQ>(p, sum, yv, xs, ntail);
                }
#pragma unroll
                for (int u = 0; u < kCosG; u++) {
#pragma unroll
                    for (int q = 0; q < NQ; q++)
                        consider(q, fabs(sum[q][u] / (sh.snorm[cur][u0 + u] * nq[q]) - target[q]), sidx[u]);  // src/sound.rs:30-32, 359
                    sidx[u] = kCosNone;  // done: the general epilogue below skips it
                }
            } else if (all_staged) {
                // ---- mixed lengths, all in shared memory: the queries' next chunk is fetched while the current one is consumed
                if constexpr (NQ == 1) {
                    double yv[NQ][8];
                    if (maxchunk) {
#pragma unroll
                        for (int q = 0; q < NQ; q++) {
#pragma unroll
                            for (int v = 0; v < 8; v++) yv[q][v] = y[q][v * 32];
                        }
                    }
                    for (uint32_t ch = 0; ch < maxchunk; ch++) {
                        double yn[NQ][8];
                        if (ch + 1 < maxchunk) {
#pragma unroll
                            for (int q = 0; q < NQ; q++) {
#pragma unroll
                                for (int v = 0; v < 8; v++) yn[q][v] = y[q][((size_t)(ch + 1) * 8 + v) * 32];
                            }
                        }
#pragma unroll
                        for (int u = 0; u < kCosG; u++) {
                            if (ch < nchunk[u]) {  // warp-uniform
#pragma unroll
                                for (int v = 0; v < 4; v++) {
                                    const double2 xx = xs[u * (kCosSegCap / 2) + ch * 4 + v];
#pragma unroll
                                    for (int q = 0; q < NQ; q++) {
                                        p[q][u][2 * v] = p[q][u][2 * v] + xx.x * yv[q][2 * v];
                                        p[q][u][2 * v + 1] = p[q][u][2 * v + 1] + xx.y * yv[q][2 * v + 1];
                                    }
                                }
                            }
                        }
#pragma unroll
                        for (int q = 0; q < NQ; q++) {
#pragma unroll
                            for (int v = 0; v < 8; v++) yv[q][v] = yn[q][v];
                        }
                    }
                } else {
                    // (in place, as above: the loads run at most one chunk past the last whole chunk of the query)
                    double yv[NQ][8];
#pragma unroll
                    for (int q = 0; q < NQ; q++) {
#pragma unroll
                        for (int v = 0; v < 8; v++) yv[q][v] = y[q][v * 32];
                    }
                    for (uint32_t ch = 0; ch < maxchunk; ch++) {
                        bool on[kCosG];
#pragma unroll
                        for (int u = 0; u < kCosG; u++) on[u] = ch < nchunk[u];  // warp-uniform
#pragma unroll
                        for (int v = 0; v < 4; v++) {
#pragma unroll
                            for (int u = 0; u < kCosG; u++) {
                                if (on[u]) {
                                    const double2 xx = xs[u * (kCosSegCap / 2) + ch * 4 + v];
#pragma unroll
                                    for (int q = 0; q < NQ; q++) {
                                        p[q][u][2 * v] = p[q][u][2 * v] + xx.x * yv[q][2 * v];
                                        p[q][u][2 * v + 1] = p[q][u][2 * v + 1] + xx.y * yv[q][2 * v + 1];
                                    }
                                }
                            }
#pragma unroll
                            for (int q = 0; q < NQ; q++) {
                                yv[q][2 * v] = y[q][((size_t)(ch + 1) * 8 + 2 * v) * 32];
                                yv[q][2 * v + 1] = y[q][((size_t)(ch + 1) * 8 + 2 * v + 1) * 32];
                            }
                        }
                    }
                }
            } else {
                // ---- some segment longer than the staging buffer: its frames come from global memory ----------------------
                for (uint32_t ch = 0; ch < maxchunk; ch++) {
                    double yv[NQ][8];
#pragma unroll
                    for (int q = 0; q < NQ; q++) {
#pragma unroll
                        for (int v = 0; v < 8; v++) yv[q][v] = y[q][((size_t)ch * 8 + v) * 32];
                    }
#pragma unroll
                    for (int u = 0; u < kCosG; u++) {
                        if (ch < nchunk[u]) {  // warp-uniform
                            if (kd[u] <= (uint32_t)kCosSegCap) {
#pragma unroll
                                for (int v = 0; v < 4; v++) {
                                    const double2 xx = xs[u * (kCosSegCap / 2) + ch * 4 + v];
#pragma unroll
                                    for (int q = 0; q < NQ; q++) {
                                        p[q][u][2 * v] = p[q][u][2 * v] + xx.x * yv[q][2 * v];
                                        p[q][u][2 * v + 1] = p[q][u][2 * v + 1] + xx.y * yv[q][2 * v + 1];
                                    }
                                }
                            } else {
#pragma unroll
                                for (int v = 0; v < 8; v++) {
                                    const double xv = __ldg(xg[u] + (size_t)ch * 8 + v);
#pragma unroll
                                    for (int q = 0; q < NQ; q++) p[q][u][v] = p[q][u][v] + xv * yv[q][v];
                                }
                            }
                        }
                    }
                }
            }
            // ---- combine, tail, similarity, argmin by (distance, index) ------------------------------------------------------
#pragma unroll
            for (int u = 0; u < kCosG; u++) {
                if (sidx[u] != kCosNone) {
                    double sum[NQ];
#pragma unroll
                    for (int q = 0; q < NQ; q++) {
                        sum[q] = 0.0;
                        sum[q] = sum[q] + (p[q][u][0] + p[q][u][4]);
                        sum[q] = sum[q] + (p[q][u][1] + p[q][u][5]);
                        sum[q] = sum[q] + (p[q][u][2] + p[q][u][6]);
                        sum[q] = sum[q] + (p[q][u][3] + p[q][u][7]);
                    }
                    for (uint32_t e = nchunk[u] * 8; e < len[u]; e++) {
                        const double xv = kd[u] <= (uint32_t)kCosSegCap ? sseg[b][u0 + u][e] : __ldg(xg[u] + e);
#pragma unroll
                        for (int q = 0; q < NQ; q++) sum[q] = sum[q] + xv * y[q][(size_t)e * 32];
                    }
#pragma unroll
                    for (int q = 0; q < NQ; q++) {
                        const double nrm = sh.snorm[cur][u0 + u] * nq[q];  // norm(me) * norm(you), src/sound.rs:30
                        const double sim = sum[q] / nrm;                   // src/sound.rs:32
                        consider(q, fabs(sim - target[q]), sidx[u]);       // src/sound.rs:359
                    }
                }
            }
          }
        }
        if (threadIdx.x < kCosStage) sh.sdesc[nxt2][threadIdx.x] = d2, sh.snorm[nxt2][threadIdx.x] = n2;
        cur = nxt;
        b ^= 1;
    }
    cos_cp_async_wait_all();
    if (!active) return;
#pragma unroll
    for (int q = 0; q < NQ; q++) {
        const size_t o = (size_t)slice * ngroups * 32 + (size_t)g[q] * 32 + lane;
        part_dist[o] = best[q];
        part_idx[o] = best_idx[q];
    }
}

// blocks [0, nqb2 * nslices) take the paired work items (two groups of one length per warp), the rest the single groups
// (half as long per CTA: they fill the tail); items = {g0, g1} x npairs, then {g, -} x nsingles
__global__ void __launch_bounds__(32 * kCosWarps, 2)
k_cosine_scan(const double* __restrict__ dmfcc, const uint4* __restrict__ cseg, const double* __restrict__ cnorm, uint32_t nseg, int c,
              uint32_t nslices, const double* __restrict__ qlanes, const uint32_t* __restrict__ group_len,
              const uint32_t* __restrict__ group_rowbase, const uint32_t* __restrict__ group_qid, uint32_t ngroups,
              const double* __restrict__ qnorm, const double* __restrict__ targets, double* __restrict__ part_dist,
              uint32_t* __restrict__ part_idx, const uint2* __restrict__ items, uint32_t npairs, uint32_t nsingles) {
    extern __shared__ __align__(16) double cos_sseg[];  // [2][kCosStage][kCosSegCap]: 32 KB per 4 staged segments
    double (*sseg)[kCosStage][kCosSegCap] = reinterpret_cast<double (*)[kCosStage][kCosSegCap]>(cos_sseg);
    __shared__ CosShared sh;
    const uint32_t warp = threadIdx.x >> 5;
    const uint32_t pair_blocks = (npairs + kCosWarps - 1) / kCosWarps * nslices;
    if (blockIdx.x < pair_blocks) {
        const uint32_t it = blockIdx.x / nslices * kCosWarps + warp;
        cos_scan_body<2>(sseg, sh, dmfcc, cseg, cnorm, nseg, c, nslices, blockIdx.x % nslices, qlanes, group_len, group_rowbase, group_qid,
                         ngroups, qnorm, targets, part_dist, part_idx, it < npairs ? items + it : nullptr);
    } else {
        const uint32_t r = blockIdx.x - pair_blocks;
        const uint32_t it = r / nslices * kCosWarps + warp;
        cos_scan_body<1>(sseg, sh, dmfcc, cseg, cnorm, nseg, c, nslices, r % nslices, qlanes, group_len, group_rowbase, group_qid,
                         ngroups, qnorm, targets, part_dist, part_idx, it < nsingles ? items + npairs + it : nullptr);
    }
}

__global__ void k_cosine_merge(const double* __restrict__ part_dist, const uint32_t* __restrict__ part_idx, uint32_t nslices,
                               uint32_t nslots, const uint32_t* __restrict__ group_qid, uint32_t index_base,
                               uint32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= nslots) return;
    const uint32_t qid = group_qid[slot];
    if (qid == 0xFFFFFFFFu) return;
    double best = 2.0;
    uint32_t idx = kCosNone;  // nothing < 2.0 -> index 0, as the reference's fold seed (src/sound.rs:361, 369)
    for (uint32_t sl = 0; sl < nslices; sl++) {
        const double d = part_dist[(size_t)sl * nslots + slot];
        const uint32_t i = part_idx[(size_t)sl * nslots + slot];
        // slices interleave the dictionary: equal distances go to the smaller index (first minimum wins, src/sound.rs:362)
        if (i != kCosNone && (d < best || (d == best && i < idx))) {
            best = d;
            idx = i;
        }
    }
    out_idx[qid] = (idx != kCosNone ? idx : 0) + index_base;
    out_dist[qid] = best;
}

__global__ void k_cos_gather_norm(const double* __restrict__ norm, const uint4* __restrict__ cseg, uint32_t n, double* __restrict__ out) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = norm[cseg[i].w];
}

// empty queries never reach a lane: their similarity is 0/0 = NaN against everything, so the fold keeps (0, 2.0)
__global__ void k_fill_result(uint32_t* __restrict__ idx, double* __restrict__ dist, size_t n, uint32_t idx_v, double dist_v) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) {
        idx[i] = idx_v;
        dist[i] = dist_v;
    }
}

int fill_result(ss_ctx* ctx, uint32_t* d_idx, double* d_dist, size_t n) {
    if (!n) return SS_OK;
    k_fill_result<<<ceil_div((long long)n, 256), 256, 0, ctx->stream>>>(d_idx, d_dist, n, 0xFFFFFFFFu, kInf);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

int cosine_dict_build(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    SS_CUDA(ctx, d->d_norm.reserve(std::max<size_t>(d->nseg, 1)));
    if (!d->nseg) return SS_OK;
    k_seg_norm<<<ceil_div((long long)d->nseg, 128), 128, 0, ctx->stream>>>(d->d_mfcc.p, d->d_off.p, d->nseg, d->c, d->d_norm.p);
    SS_LAUNCHED(ctx);
    // the scan's walk order: segments by (length, index), so that the four segments a CTA stages together have one length;
    // {first frame, frames, index} per position + the norms in the same order (ss_dict_create synchronises the stream
    // before it returns: the upload has left the local table by then)
    std::vector<uint64_t> key(d->nseg);
    for (size_t s = 0; s < d->nseg; s++) key[s] = ((d->h_off[s + 1] - d->h_off[s]) << 32) | (uint64_t)s;
    std::sort(key.begin(), key.end());
    d->h_cos_seg.resize(d->nseg);
    for (size_t i = 0; i < d->nseg; i++) {
        const uint32_t s = (uint32_t)key[i];
        const uint64_t f0 = d->h_off[s];
        d->h_cos_seg[i] = make_uint4((uint32_t)f0, (uint32_t)(f0 >> 32), (uint32_t)(d->h_off[s + 1] - f0), s);
    }
    SS_TRY(upload(ctx, d->d_cos_seg, d->h_cos_seg.data(), d->h_cos_seg.size()));
    SS_CUDA(ctx, d->d_cos_norm.reserve(d->nseg));
    k_cos_gather_norm<<<ceil_div((long long)d->nseg, 256), 256, 0, ctx->stream>>>(d->d_norm.p, d->d_cos_seg.p, (uint32_t)d->nseg, d->d_cos_norm.p);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

int cosine_queries_build(ss_queries* q) {
    ss_ctx* ctx = q->ctx;
    SS_TRY(dtw_queries_build(q));  // shares the length-sorted group tables
    if (q->cos_built) return SS_OK;
    SS_CUDA(ctx, q->d_norm.reserve(std::max<size_t>(q->nq, 1)));
    if (q->nq) {
        k_seg_norm<<<ceil_div((long long)q->nq, 128), 128, 0, ctx->stream>>>(q->d_mfcc.p, q->d_off.p, q->nq, q->c, q->d_norm.p);
        SS_LAUNCHED(ctx);
    }
    // (+ two chunks: the scan's register-buffered query loads run up to two chunks past the last group's rows)
    SS_CUDA(ctx, q->d_lane64.reserve(std::max<uint64_t>(q->total_rows, 1) * q->c * 32 + 16 * 32));
    if (q->ngroups) {
        k_query_lanes64<<<q->ngroups, 256, 0, ctx->stream>>>(q->d_mfcc.p, q->d_off.p, q->c, q->d_group_len.p,
                                                            q->d_group_rowbase.p, q->d_group_qid.p, q->d_lane64.p);
        SS_LAUNCHED(ctx);
    }
    // work items of the scan: two groups of one length per warp wherever a length has two, the odd group of a length alone
    {
        std::vector<uint2> pairs, singles;
        for (uint32_t g = 0; g < q->ngroups;) {
            if (g + 1 < q->ngroups && q->h_group_len[g + 1] == q->h_group_len[g]) {
                pairs.push_back(make_uint2(g, g + 1));
                g += 2;
            } else {
                singles.push_back(make_uint2(g, kCosNone));
                g += 1;
            }
        }
        q->cos_npairs = (uint32_t)pairs.size();
        q->cos_nsingles = (uint32_t)singles.size();
        pairs.insert(pairs.end(), singles.begin(), singles.end());
        if (!pairs.empty()) {
            SS_TRY(upload(ctx, q->d_cos_items, pairs.data(), pairs.size()));
            SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the table is local
        }
    }
    q->cos_built = true;
    return SS_OK;
}

int cosine_match_dev(ss_dict* d, ss_queries* q, const double* d_targets, uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    SS_TRY(cosine_queries_build(q));
    // work = sum over pairs of min(Kq, Kd) products (the sorted segment lengths and their prefix sums are built once per
    // dictionary: sorting 100 000 lengths on every call was 4 ms of a 4.05 ms nq = 1 match)
    {
        if (d->h_len_sorted.size() != d->nseg) {
            d->h_len_sorted.resize(d->nseg);
            for (size_t s = 0; s < d->nseg; s++) d->h_len_sorted[s] = d->h_off[s + 1] - d->h_off[s];
            std::sort(d->h_len_sorted.begin(), d->h_len_sorted.end());
            d->h_len_prefix.assign(d->nseg + 1, 0);
            for (size_t s = 0; s < d->nseg; s++) d->h_len_prefix[s + 1] = d->h_len_prefix[s] + d->h_len_sorted[s];
        }
        const std::vector<uint64_t>&dl = d->h_len_sorted, &pre = d->h_len_prefix;
        uint64_t work = 0;
        for (size_t i = 0; i < q->nq; i++) {
            const uint64_t lq = q->h_off[i + 1] - q->h_off[i];
            const size_t pos = std::upper_bound(dl.begin(), dl.end(), lq) - dl.begin();
            work += pre[pos] + (uint64_t)(dl.size() - pos) * lq;
        }
        d->last_work = work * (uint64_t)d->c;
    }
    if (q->nq) {
        k_fill_result<<<ceil_div((long long)q->nq, 256), 256, 0, ctx->stream>>>(d_out_idx, d_out_dist, q->nq, d->index_base, 2.0);
        SS_LAUNCHED(ctx);
    }
    const uint32_t nqb2 = (q->cos_npairs + kCosWarps - 1) / kCosWarps, nqb1 = (q->cos_nsingles + kCosWarps - 1) / kCosWarps;
    const uint32_t nqb = nqb2 + nqb1;  // CTAs per slice: paired work items first, single groups last
    if (!nqb || !d->nseg) return SS_OK;
    const uint32_t nslots = q->ngroups * 32;
    // slice sl takes the groups sl, sl + nslices, ... of that order: every slice sees the same mix of lengths. CTAs per SM over
    // the launch (two are resident), measured at config 4: 8 -> 41.0 ms, 16 -> 39.4, 32 -> 38.8; small batches keep 16 (the merge
    // walks a slot's slices one after the other)
    const uint32_t waves = nqb >= 8 ? 32 : 16;
    const uint32_t ngrp = (uint32_t)((d->nseg + kCosStage - 1) / kCosStage);
    const uint32_t nslices = std::max<uint32_t>(1, std::min<uint32_t>(ngrp, ((uint32_t)ctx->sm_count * waves + nqb - 1) / nqb));
    SS_CUDA(ctx, d->d_cand_exact.reserve((size_t)nslices * nslots));
    SS_CUDA(ctx, d->d_cand_idx.reserve((size_t)nslices * nslots));
    if (!d->ev_scan0) {
        SS_CUDA(ctx, cudaEventCreate(&d->ev_scan0));
        SS_CUDA(ctx, cudaEventCreate(&d->ev_scan1));
    }
    SS_CUDA(ctx, cudaEventRecord(d->ev_scan0, ctx->stream));
    const int cos_smem = (int)(sizeof(double) * 2 * kCosStage * kCosSegCap);
    SS_CUDA(ctx, cudaFuncSetAttribute(k_cosine_scan, cudaFuncAttributeMaxDynamicSharedMemorySize, cos_smem));
    k_cosine_scan<<<nqb * nslices, 32 * kCosWarps, cos_smem, ctx->stream>>>(d->d_mfcc.p, d->d_cos_seg.p, d->d_cos_norm.p, (uint32_t)d->nseg, d->c, nslices,
                                                         q->d_lane64.p, q->d_group_len.p, q->d_group_rowbase.p, q->d_group_qid.p,
                                                         q->ngroups, q->d_norm.p, d_targets, d->d_cand_exact.p, d->d_cand_idx.p, q->d_cos_items.p,
                                                         q->cos_npairs, q->cos_nsingles);
    SS_LAUNCHED(ctx);
    SS_CUDA(ctx, cudaEventRecord(d->ev_scan1, ctx->stream));
    d->scan_timed = true;
    k_cosine_merge<<<ceil_div(nslots, 128), 128, 0, ctx->stream>>>(d->d_cand_exact.p, d->d_cand_idx.p, nslices, nslots,
                                                                  q->d_group_qid.p, d->index_base, d_out_idx, d_out_dist);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// SoundSequence::from_distances (src/sound.rs:405-417) on the device: step t is at_distance(distances[t], previous), and
// from step 1 on the query IS a dictionary segment already in HBM, so the whole chain runs as one launch per step with
// no host decision in between. k_cosine_scan puts 32 queries on the lanes; with one query that lights one lane in 32, so
// this kernel turns the mapping around: DICTIONARY SEGMENTS on lanes, the one query broadcast from shared memory.
//
// kWalkLanes = 8 lanes per segment, lane u owning rulinalg's partial sum p_u (elements u, u + 8, ...): a group reads 64
// contiguous bytes of its segment per chunk. The combine is cos_finish's, through shuffles into lane 0 of the group:
// 0.0 + (p0 + p4), + (p1 + p5), + (p2 + p6), + (p3 + p7), then the <= 7 tail elements in order, then
// sum / (norm_d * norm_q) - the same operations in the same order as k_cosine_scan, so every (idx, dist) is the bits of
// ss_dict_match(nq = 1). A warp's four groups take four consecutive positions of the (length, index) walk order, so they
// almost always run the same number of chunks. Each CTA leaves its (distance, index) minimum in a partial; the last CTA
// to finish (atomic ticket) reduces the partials, writes step t's result and the local index the next step queries, and
// resets the ticket. No CTA ever waits for another.
constexpr int kWalkThreads = 256;                        // 32 segments in flight per CTA
constexpr int kWalkLanes = 8;                            // lanes per dictionary segment (rulinalg's 8 partial sums)
constexpr int kWalkGroups = kWalkThreads / kWalkLanes;
constexpr int kWalkCtasPerSm = 6;                        // all resident at 40 registers a thread: one wave
constexpr uint32_t kWalkQCap = 2048;                     // query doubles staged in shared memory (beyond: global memory)

// (distance, index) minimum with the fold's seed (2.0, none): a smaller distance wins, an equal one only with a smaller
// index than a winner already found - never against the seed, so a distance of exactly 2.0 never beats it (src/sound.rs:362);
// NaN never wins. Every candidate that replaces the seed is < 2.0, so partials merge with the same rule.
__device__ __forceinline__ void walk_min(double& bd, uint32_t& bi, double d, uint32_t i) {
    if (d < bd || (d == bd && i < bi && bi != kCosNone)) {
        bd = d;
        bi = i;
    }
}

__device__ __forceinline__ void walk_block_min(double& bd, uint32_t& bi) {
    __shared__ double sd[kWalkThreads / 32];
    __shared__ uint32_t si[kWalkThreads / 32];
#pragma unroll
    for (int o = 16; o; o >>= 1) walk_min(bd, bi, __shfl_xor_sync(0xffffffffu, bd, o), __shfl_xor_sync(0xffffffffu, bi, o));
    __syncthreads();  // (sd / si are reused by the last CTA's second reduction)
    if ((threadIdx.x & 31) == 0) sd[threadIdx.x >> 5] = bd, si[threadIdx.x >> 5] = bi;
    __syncthreads();
    if (threadIdx.x == 0)
        for (int w = 1; w < kWalkThreads / 32; w++) walk_min(bd, bi, sd[w], si[w]);
}

__global__ void __launch_bounds__(kWalkThreads)
k_cosine_walk_step(const double* __restrict__ dmfcc, const uint64_t* __restrict__ doff, const double* __restrict__ dnorm,
                   const uint4* __restrict__ cseg, const double* __restrict__ cnorm, uint32_t nseg, int c, uint32_t max_kd,
                   const double* __restrict__ start, const uint64_t* __restrict__ start_off, const double* __restrict__ start_norm,
                   const double* __restrict__ targets, uint32_t step, uint32_t index_base, double* __restrict__ part_dist,
                   uint32_t* __restrict__ part_idx, uint32_t* __restrict__ state /* [0] ticket, [1] query of the next step */,
                   uint32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    __shared__ double sq[kWalkQCap];
    __shared__ bool last;
    // the query: the start sound at step 0, else the segment the previous step returned (written by its last CTA)
    const double* qp;
    uint32_t kq;
    double nq;
    if (step == 0) {
        qp = start + start_off[0] * c;
        kq = (uint32_t)(start_off[1] - start_off[0]) * (uint32_t)c;
        nq = start_norm[0];
    } else {
        const uint32_t s = state[1];
        qp = dmfcc + doff[s] * c;
        kq = (uint32_t)(doff[s + 1] - doff[s]) * (uint32_t)c;
        nq = dnorm[s];
    }
    const double target = targets[step];
    const uint32_t nstage = min(min(kq, max_kd), kWalkQCap);  // no segment reads past max_kd
    for (uint32_t e = threadIdx.x; e < nstage; e += kWalkThreads) sq[e] = qp[e];
    __syncthreads();

    const uint32_t u = threadIdx.x % kWalkLanes;
    const uint32_t lane = threadIdx.x & 31;
    const uint32_t gmask = 0xFFu << (lane & ~(kWalkLanes - 1));  // this group's 8 lanes
    double bd = 2.0;              // fold((0, 2.0)), src/sound.rs:361
    uint32_t bi = kCosNone;
    for (uint32_t base = blockIdx.x * kWalkGroups; base < nseg; base += gridDim.x * kWalkGroups) {  // warp-uniform
        const uint32_t pos = base + threadIdx.x / kWalkLanes;
        if (pos >= nseg) break;  // (whole groups leave together: the shuffles below only span a group)
        const uint4 dsc = __ldg(&cseg[pos]);
        const double* x = dmfcc + (((uint64_t)dsc.y << 32) | dsc.x) * c;
        const uint32_t kd = dsc.z * (uint32_t)c;
        const uint32_t len = kd < kq ? kd : kq;
        const uint32_t nch = len / kWalkLanes;
        const uint32_t nch_s = min(nch, kWalkQCap / kWalkLanes);  // chunks whose query values are staged
        double p = 0.0;
        uint32_t ch = 0;
#pragma unroll 4
        for (; ch < nch_s; ch++) {
            const uint32_t e = ch * kWalkLanes + u;
            p = p + __ldg(x + e) * sq[e];
        }
        for (; ch < nch; ch++) {
            const uint32_t e = ch * kWalkLanes + u;
            p = p + __ldg(x + e) * qp[e];
        }
        // (p0 + p4), (p1 + p5), (p2 + p6), (p3 + p7) on lanes 0..3 of the group, then summed in that order on lane 0
        const double pair = p + __shfl_down_sync(gmask, p, 4, kWalkLanes);
        const double pr1 = __shfl_sync(gmask, pair, 1, kWalkLanes);
        const double pr2 = __shfl_sync(gmask, pair, 2, kWalkLanes);
        const double pr3 = __shfl_sync(gmask, pair, 3, kWalkLanes);
        if (u == 0) {
            double sum = 0.0 + pair;
            sum = sum + pr1;
            sum = sum + pr2;
            sum = sum + pr3;
            for (uint32_t e = nch * kWalkLanes; e < len; e++) sum = sum + __ldg(x + e) * (e < kWalkQCap ? sq[e] : qp[e]);
            const double sim = sum / (__ldg(&cnorm[pos]) * nq);  // src/sound.rs:30-32
            walk_min(bd, bi, fabs(sim - target), dsc.w);         // src/sound.rs:359-366
        }
    }
    walk_block_min(bd, bi);
    if (threadIdx.x == 0) {
        part_dist[blockIdx.x] = bd;
        part_idx[blockIdx.x] = bi;
        __threadfence();
        last = atomicAdd(&state[0], 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!last) return;
    // the last CTA: every other CTA's partial is visible (its fence came before its ticket)
    __threadfence();
    bd = 2.0;
    bi = kCosNone;
    for (uint32_t b = threadIdx.x; b < gridDim.x; b += kWalkThreads) walk_min(bd, bi, __ldcg(&part_dist[b]), __ldcg(&part_idx[b]));
    walk_block_min(bd, bi);
    if (threadIdx.x == 0) {
        const uint32_t s = bi != kCosNone ? bi : 0;  // nothing < 2.0: index 0, as the fold's seed (src/sound.rs:369)
        out_idx[step] = s + index_base;
        out_dist[step] = bd;
        state[1] = s;
        state[0] = 0;
    }
}

int cosine_walk_dev(ss_dict* d, const double* d_start, const uint64_t* d_start_off, const double* d_targets, size_t nsteps,
                    uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    if (!nsteps) return SS_OK;
    const uint32_t nseg = (uint32_t)d->nseg;
    const uint32_t grid = (uint32_t)std::min<long long>(ceil_div(nseg, kWalkGroups), (long long)ctx->sm_count * kWalkCtasPerSm);
    SS_CUDA(ctx, d->d_walk_part_dist.reserve(grid));
    SS_CUDA(ctx, d->d_walk_part_idx.reserve(grid));
    SS_CUDA(ctx, d->d_walk_state.reserve(2));
    SS_CUDA(ctx, d->d_walk_qnorm.reserve(1));
    SS_CUDA(ctx, cudaMemsetAsync(d->d_walk_state.p, 0, 2 * sizeof(uint32_t), ctx->stream));
    // the start query's norm by the same kernel as every query's and segment's (src/sound.rs:36-38)
    k_seg_norm<<<1, 32, 0, ctx->stream>>>(d_start, d_start_off, 1, d->c, d->d_walk_qnorm.p);
    SS_LAUNCHED(ctx);
    const uint32_t max_kd = d->max_len * (uint32_t)d->c;
    for (size_t t = 0; t < nsteps; t++) {
        k_cosine_walk_step<<<grid, kWalkThreads, 0, ctx->stream>>>(d->d_mfcc.p, d->d_off.p, d->d_norm.p, d->d_cos_seg.p, d->d_cos_norm.p, nseg, d->c,
                                                                   max_kd, d_start, d_start_off, d->d_walk_qnorm.p, d_targets, (uint32_t)t,
                                                                   d->index_base, d->d_walk_part_dist.p, d->d_walk_part_idx.p,
                                                                   d->d_walk_state.p, d_out_idx, d_out_dist);
        SS_LAUNCHED(ctx);
    }
    return SS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// DTW refine: exact f64 recurrence on the candidates. One thread per (query slot, candidate); the DP row lives in a
// global scratch laid out [column][pair] so that neighbouring threads touch neighbouring addresses.
// ---------------------------------------------------------------------------------------------------------------
// Lower bound on the EXACT distance of any pair whose scan distance is >= w (see k_dtw_finalize for the derivation):
//   bound_mode 0 (fp32 scan):  |scan - exact| <= eps (max|a|^2 + max|b|^2)
//   bound_mode 1 (fp16 products, fp32 DP):  exact >= w - 2 delta sqrt(w) - E32,  delta = 2^-11 (|a| + |b|)
//   bound_mode 2 (fp16 products AND packed-half DP, dtw_h2.cu): the scan is at most the rounded-frame DTW times (1 + 2^-11) per
//     rounding on the path (cost + running sum per cell, <= Lq + Ld cells, Ld <= 32) plus eta (fp16 subnormals; `eps` carries
//     it), and a path sum beyond the fp16 range reads +inf: w is capped at 60000 / (S (Lq + 32)). Then the same input-rounding
//     step as mode 1:  exact >= t - 2 delta sqrt(t),  t = (min(w, cap) - eta) (1 + 2^-11)^-(Lq + 34)
//   bound_mode 3 (dtw_h2.cu's strip kernel, sequences of any length): the candidate KEYS are per-pair lower bounds of the
//     rounded-frame distance already - (scan - eta)(1 + 2^-11)^-(Lq + Ld + 2), computed by the scan - so w needs no common
//     factor; only the cap remains (a path sum beyond the fp16 range reads +inf whatever the pair: its rounded-frame
//     distance is at least the bound of a pair of the longest segment, ld_max, at 60000 / S):  t = min(w, cap)
// The per-query part (two square roots, one exponential) is computed once (make_scan_bound); lower() is what runs per candidate.
struct ScanBound {
    int mode;
    double a, delta, cap, defl;  // a: the additive term of modes 0 / 1 (eps (na + nb) / E32), eta of mode 2
    __device__ __forceinline__ double lower(float scan) const {
        if (mode == 0) return (double)scan - a;
        const double w = scan > 0.f ? (double)scan : 0.0;  // (+inf stays +inf)
        if (mode == 3) {
            const double t = fmin(w, cap);
            return t - 2.0 * delta * sqrt(t);
        }
        if (mode == 2) {
            const double v = fmin(w, cap) - a;
            const double t = v > 0.0 ? v * defl : 0.0;
            return t - 2.0 * delta * sqrt(t);
        }
        return w - 2.0 * delta * sqrt(w) - a;
    }
};
__device__ __forceinline__ ScanBound make_scan_bound(double na, double nb, double eps, int bound_mode, int la = 0, double inv_s = 0.0, int ld_max = 32) {
    ScanBound b;
    b.mode = bound_mode;
    b.delta = 1.001 * (sqrt(na) + sqrt(nb)) / 2048.0 + 1e-6;
    b.cap = 0.0, b.defl = 1.0;
    if (bound_mode == 0) {
        b.a = eps * (na + nb);
    } else if (bound_mode == 3) {
        const double n = (double)(la + ld_max);
        b.a = 0.0;
        b.cap = fmax(60000.0 * inv_s / n - 1.001 * eps, 0.0) * exp(-(n + 2.0) * 4.8937e-4 /* = 7.06e-4 ln 2, as the scan */);
    } else if (bound_mode == 2) {
        b.a = eps;
        b.cap = 60000.0 * inv_s / (double)(la + 32);
        b.defl = exp(-(double)(la + 34) * 4.8816207e-4 /* > ln(1 + 2^-11) */);
    } else {
        // E32: fp32 accumulation of the 16 products in the tensor core (<= 16 ulp of na + nb + 2 sqrt(na nb), truncating)
        // plus <= Lq + Ld <= 64 roundings of the running sum along the path
        b.a = 2e-5 * (na + nb);
    }
    return b;
}
__device__ __forceinline__ double scan_lower_bound(float scan, double na, double nb, double eps, int bound_mode, int la = 0, double inv_s = 0.0,
                                                   int ld_max = 32) {
    return make_scan_bound(na, nb, eps, bound_mode, la, inv_s, ld_max).lower(scan);
}

// Pair t of a k_dtw_rescore_warp launch is candidate s_begin + t % s_count of slot t / s_count. Two launches per match:
//   (s_begin, s_count) = (0, k):       the k best candidates by scan distance, unconditionally;
//   (s_begin, s_count) = (k, kp - k):  the rest, but only those whose scan distance does not already PROVE (by the scan's
//                                      error bound) that they are farther than the k-th exact distance found in the first
//                                      launch - such a candidate cannot enter the top-k and is recorded as +inf.
struct RescoreBound {
    const float* cand_adist;   // scan distances of the candidates (nullptr: rescore unconditionally)
    const float* max_na;       // [0] max |a|^2 over the queries
    const float* max_nb;       // [0] max |b|^2 over the shard
    const float* slot_max_na;  // per slot max |a|^2 (nullable)
    double eps;
    int bound_mode, k;
    double inv_s;  // bound_mode 2 / 3: 1 / S
    int ld_max;    // bound_mode 3: the dictionary's longest segment
};
// ---------------------------------------------------------------------------------------------------------------
// The whole refine of one query slot by ONE warp (sequences of <= 32 frames on both sides): the k best candidates by scan
// distance unconditionally, the other kp - k only if the scan's error bound cannot rule them out against the k-th exact
// distance, then the (distance, index) sort, the top-k store and the certification - what k_dtw_rescore_warp (twice) and
// k_dtw_finalize do in three launches for longer sequences, with the same arithmetic per cell. Lane j owns dictionary column
// j; the pair's local costs go to shared memory first (39 f64 operations per cell on 32 busy lanes), then the recurrence runs
// as an anti-diagonal wavefront: at step t lane j computes cell (t - j, j) from its own previous value (up), its left
// neighbour's (one 64-bit shuffle) and the one it received a step earlier (diag).
// ---------------------------------------------------------------------------------------------------------------
// `sa` holds the query's frames (staged once per slot, coalesced); lane j keeps dictionary frame j in registers (its 13 loads
// are issued back to back: one memory latency per pair). cst = the pair's local costs, [row][lane].
// BAND: cells outside the band of radius `band` (>= 1) are +inf, one integer test per cell against the lane's row range.
template <bool BAND>
__device__ __forceinline__ double warp_dtw_exact(const double* __restrict__ sa, int la, const double* __restrict__ b, int lb, int c, double* cst,
                                                 int lane, uint32_t band) {
    double br[SS_MAX_NCOEFFS];
#pragma unroll
    for (int k = 0; k < SS_MAX_NCOEFFS; k++) br[k] = (k < c && lane < lb) ? b[(size_t)lane * c + k] : 0.0;
    int blo = 0, bhi = 0;
    if (BAND && la > 0 && lb > 0) band_rows(min(lane, lb - 1), la, lb, band, &blo, &bhi);
    __syncwarp();  // the previous pair's costs are no longer read
    for (int i = 0; i < la; i++) {
        double cost = 0.0;
#pragma unroll
        for (int k = 0; k < SS_MAX_NCOEFFS; k++)
            if (k < c) {
                const double dlt = sa[i * c + k] - br[k];
                cost = cost + dlt * dlt;
            }
        cst[i * 32 + lane] = cost;
    }
    __syncwarp();
    double cur = kInf, recv_prev = kInf, result = kInf;
    for (int step = 0; step < la + lb - 1; step++) {
        const double recv = __shfl_up_sync(0xffffffffu, cur, 1);  // left neighbour's last cell = D(i, j-1)
        const int i = step - lane;
        const bool active = lane < lb && i >= 0 && i < la;
        if (active) {
            const double up = cur;
            const double left = lane ? recv : kInf;
            const double diag = lane ? recv_prev : kInf;
            double m;
            if (i == 0 && lane == 0) m = 0.0;
            else m = fmin(fmin(up, left), diag);
            if (BAND && (i < blo || i > bhi)) cur = kInf;
            else cur = cst[i * 32 + lane] + m;
            if (i == la - 1 && lane == lb - 1) result = cur;
        }
        recv_prev = recv;
    }
    result = __shfl_sync(0xffffffffu, result, lb > 0 ? lb - 1 : 0);
    return (la && lb) ? result / (double)(la + lb) : kInf;
}

template <bool BAND>
__global__ void __launch_bounds__(128)
k_dtw_refine_warp(const double* __restrict__ dmfcc, const uint64_t* __restrict__ doff, const double* __restrict__ qmfcc,
                  const uint64_t* __restrict__ qoff, int c, const uint32_t* __restrict__ group_qid, const uint32_t* __restrict__ cand_idx,
                  const float* __restrict__ cand_adist, uint32_t nslots, int kp, int k, uint32_t index_base, const float* __restrict__ max_na,
                  const float* __restrict__ max_nb, double eps, const float* __restrict__ slot_max_na, int bound_mode, double inv_s,
                  uint8_t* __restrict__ uncert_flag, uint32_t* __restrict__ out_idx, double* __restrict__ out_dist,
                  unsigned long long* __restrict__ counters, uint32_t band) {
    __shared__ double scost[4][32 * 32];
    __shared__ double squery[4][32 * SS_MAX_NCOEFFS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t slot = blockIdx.x * 4 + warp;
    if (slot >= nslots) return;  // warp-uniform from here on
    const uint32_t qid = group_qid[slot];
    if (qid == 0xFFFFFFFFu) return;
    const uint32_t my_idx = lane < kp ? cand_idx[(size_t)slot * kp + lane] : 0xFFFFFFFFu;
    const float my_adist = lane < kp ? cand_adist[(size_t)slot * kp + lane] : __int_as_float(0x7f800000);
    const double na = slot_max_na ? (double)slot_max_na[slot] : (double)max_na[0];
    const double nb = (double)max_nb[0];
    const double* a = qmfcc + qoff[qid] * c;
    const int la = (int)(qoff[qid + 1] - qoff[qid]);
    for (int e = lane; e < la * c; e += 32) squery[warp][e] = a[e];  // the query's frames: one coalesced pass (la <= 32)
    __syncwarp();
    double my_exact = kInf, kth = 0.0;
    unsigned extra = 0;
    const ScanBound bound = make_scan_bound(na, nb, eps, bound_mode, la, inv_s);
    for (int s = 0; s < kp; s++) {
        const uint32_t idx = __shfl_sync(0xffffffffu, my_idx, s);
        if (idx == 0xFFFFFFFFu) {
            if (s < k) kth = kInf;  // an empty place among the first k: nothing can be ruled out
            continue;
        }
        if (s >= k) {
            const float adist = __shfl_sync(0xffffffffu, my_adist, s);
            if (bound.lower(adist) > kth) continue;  // provably outside the top-k
            extra++;
        }
        const double e = warp_dtw_exact<BAND>(squery[warp], la, dmfcc + doff[idx] * c, (int)(doff[idx + 1] - doff[idx]), c, scost[warp], lane, band);
        if (lane == s) my_exact = e;
        if (s < k) kth = fmax(kth, e < kInf ? e : kInf);
    }
    // (distance, index) insertion sort on lane 0; NaN / inf candidates are dropped
    double dv[kMaxKeep];
    uint32_t iv[kMaxKeep];
    int n = 0;
    for (int s = 0; s < kp; s++) {
        const double dd = __shfl_sync(0xffffffffu, my_exact, s);
        const uint32_t ii = __shfl_sync(0xffffffffu, my_idx, s);
        if (lane != 0 || ii == 0xFFFFFFFFu || !(dd < kInf)) continue;
        int pos = n;
        while (pos > 0 && (dd < dv[pos - 1] || (dd == dv[pos - 1] && ii < iv[pos - 1]))) {
            dv[pos] = dv[pos - 1];
            iv[pos] = iv[pos - 1];
            pos--;
        }
        dv[pos] = dd;
        iv[pos] = ii;
        n++;
    }
    const float worst = __shfl_sync(0xffffffffu, my_adist, kp - 1);
    if (lane == 0) {
        for (int s = 0; s < k; s++) {
            out_idx[(size_t)qid * k + s] = s < n ? iv[s] + index_base : 0xFFFFFFFFu;
            out_dist[(size_t)qid * k + s] = s < n ? dv[s] : kInf;
        }
        bool uncertified = false;  // see k_dtw_finalize
        // (bound_mode 2: a list that is not full does NOT mean every pair is in it - overflowed pairs read +inf and are never
        // inserted - so the bound is evaluated anyway, at its cap)
        if (bound_mode == 2 || worst < __int_as_float(0x7f800000)) {
            const double kth_exact = n >= k ? dv[k - 1] : kInf;
            uncertified = !(bound.lower(worst) > kth_exact);
            if (uncertified) atomicAdd(&counters[0], 1ull);
        }
        if (uncert_flag) uncert_flag[qid] = uncertified ? 1 : 0;
        if (extra) atomicAdd(&counters[1], (unsigned long long)extra);
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The same exact recurrence for sequences of ANY length, one warp per pair (a single thread needs
// ~80 ms for a pair of 383 x 383 frames, which was most of config 5's match). The dictionary segment is cut into strips of 32
// columns, lane j owning column 32 s + j of strip s with its frame in registers. Per strip the warp alternates
//   A. local costs of the next 32 query rows against the strip's 32 columns -> a shared-memory ring of 64 rows (the row's
//      frame is a broadcast load; all lanes busy; 39 f64 operations per cell, the oracle's order), and
//   B. 32 steps of the anti-diagonal wavefront (lane j computes cell (t - j, column j) at step t: up = its own previous
//      value, left / diag = its left neighbour's values one / two steps earlier, by shuffle),
// and the strip's last column travels to the next strip through `bnd` (global, one row of max query length per warp), IN
// PLACE: lane 31 writes row t - 31 at the step lane 0 reads row t.
// BAND: the strip's columns are inside the band for rows [rlo, rhi] at most (band_rows of its first and last column), so the
// step blocks run from the one holding row rlo to the one in which lane 31 reaches row rhi, and only rows <= rhi get costs.
// Cells outside the band inside those blocks are +inf by the per-cell test. Rows the strip never reaches are +inf for every
// column of it: they go to the boundary row as +inf, for the next strip's lane 0.
// ---------------------------------------------------------------------------------------------------------------
template <bool BAND>
__device__ __forceinline__ double warp_dtw_exact_long(const double* __restrict__ a, int la, const double* __restrict__ b, int lb, int c,
                                                      double* __restrict__ ring, double* bnd, int lane, uint32_t band) {
    if (!la || !lb) return kInf;
    double result = kInf;
    const int nstrips = (lb + 31) >> 5;
    const int nsteps = la + 31;
    for (int s = 0; s < nstrips; s++) {
        const int col = 32 * s + lane;
        const bool colv = col < lb, first = s == 0, last = s == nstrips - 1;
        double br[SS_MAX_NCOEFFS];
#pragma unroll
        for (int k = 0; k < SS_MAX_NCOEFFS; k++) br[k] = (k < c && colv) ? b[(size_t)col * c + k] : 0.0;
        double cur = kInf, recv_prev = kInf, bl_prev = kInf;
        int blo = 0, bhi = 0, rhi = 0, t0b = 0, t0e = nsteps;
        if (BAND) {
            band_rows(min(col, lb - 1), la, lb, band, &blo, &bhi);
            rhi = __shfl_sync(0xffffffffu, bhi, 31);
            t0b = __shfl_sync(0xffffffffu, blo, 0) & ~31;
            t0e = min(nsteps, rhi + 32);
        }
        __syncwarp();  // the previous strip's boundary writes and ring reads are complete
        if (BAND && lane == 0 && !first && t0b > 0) bl_prev = bnd[t0b - 1];  // D(t0b - 1, col0 - 1), the first step's diag
        int t0 = t0b;
        for (; t0 < t0e; t0 += 32) {
            // A: rows t0 .. t0 + 31 (ring slots of rows t0 - 64 .. t0 - 33, last read at step t0 - 2)
            const int rows = min(32, (BAND ? rhi + 1 : la) - t0);
            int r = 0;
            for (; r + 4 <= rows; r += 4) {  // four rows at a time: four independent accumulation chains
                const double* ar = a + (size_t)(t0 + r) * c;
                double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
#pragma unroll
                for (int k = 0; k < SS_MAX_NCOEFFS; k++)
                    if (k < c) {
                        const double d0 = ar[k] - br[k], d1 = ar[c + k] - br[k], d2 = ar[2 * c + k] - br[k], d3 = ar[3 * c + k] - br[k];
                        c0 = c0 + d0 * d0;
                        c1 = c1 + d1 * d1;
                        c2 = c2 + d2 * d2;
                        c3 = c3 + d3 * d3;
                    }
                double* dst = ring + ((t0 + r) & 63) * 32 + lane;  // (t0 + r is a multiple of 4: the four slots do not wrap)
                dst[0] = c0, dst[32] = c1, dst[64] = c2, dst[96] = c3;
            }
            for (; r < rows; r++) {
                const double* ar = a + (size_t)(t0 + r) * c;
                double cost = 0.0;
#pragma unroll
                for (int k = 0; k < SS_MAX_NCOEFFS; k++)
                    if (k < c) {
                        const double dlt = ar[k] - br[k];
                        cost = cost + dlt * dlt;
                    }
                ring[((t0 + r) & 63) * 32 + lane] = cost;
            }
            __syncwarp();
            // B: steps t0 .. t0 + 31
            const int steps = min(32, nsteps - t0);
            double left_in = (lane == 0 && !first && t0 < la) ? bnd[t0] : kInf;  // D(t, col0 - 1), fetched one step ahead
            for (int r = 0; r < steps; r++) {
                const int t = t0 + r;
                const double recv = __shfl_up_sync(0xffffffffu, cur, 1);  // left neighbour's last cell = D(i, col - 1)
                const double left_now = left_in;
                if (r + 1 < steps) left_in = (lane == 0 && !first && t + 1 < la) ? bnd[t + 1] : kInf;
                const int i = t - lane;
                const bool active = colv && i >= 0 && i < la;
                if (active) {
                    const double up = cur;
                    const double left = lane ? recv : left_now;
                    const double diag = lane ? recv_prev : bl_prev;
                    double m;
                    if (first && i == 0 && lane == 0) m = 0.0;
                    else m = fmin(fmin(up, left), diag);
                    if (BAND && (i < blo || i > bhi)) cur = kInf;
                    else cur = ring[(i & 63) * 32 + lane] + m;
                    if (last && i == la - 1 && col == lb - 1) result = cur;
                    if (!last && lane == 31) bnd[i] = cur;  // i = t - 31: behind every row lane 0 still has to read
                }
                bl_prev = left_now;
                recv_prev = recv;
            }
            __syncwarp();
        }
        if (BAND && !last)  // lane 31 stopped at row min(t0, nsteps) - 32
            for (int r = max(0, min(t0, nsteps) - 31) + lane; r < la; r += 32) bnd[r] = kInf;
    }
    result = __shfl_sync(0xffffffffu, result, (lb - 1) & 31);
    return result / (double)(la + lb);
}

// one WARP per (slot, candidate) pair (grid-stride over the pairs; bnd: one row of bnd_stride doubles per warp)
template <bool BAND>
__global__ void __launch_bounds__(64)
k_dtw_rescore_warp(const double* __restrict__ dmfcc, const uint64_t* __restrict__ doff, const double* __restrict__ qmfcc,
                   const uint64_t* __restrict__ qoff, int c, const uint32_t* __restrict__ group_qid, const uint32_t* __restrict__ cand_idx,
                   uint32_t nt, int kp, int s_begin, int s_count, RescoreBound rb, double* __restrict__ bnd, uint32_t bnd_stride,
                   double* __restrict__ exact, unsigned long long* __restrict__ counters, uint32_t band) {
    __shared__ double ring[2][64 * 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * 2 + warp, nw = gridDim.x * 2;
    for (uint32_t t = gw; t < nt; t += nw) {  // warp-uniform
        const uint32_t slot = t / (uint32_t)s_count;
        const uint32_t pair = slot * (uint32_t)kp + (uint32_t)s_begin + t % (uint32_t)s_count;
        const uint32_t qid = group_qid[slot];
        const uint32_t idx = cand_idx[pair];
        if (qid == 0xFFFFFFFFu || idx == 0xFFFFFFFFu) {
            if (lane == 0) exact[pair] = kInf;
            continue;
        }
        const int la = (int)(qoff[qid + 1] - qoff[qid]), lb = (int)(doff[idx + 1] - doff[idx]);
        if (rb.cand_adist) {
            double kth = 0.0;  // k-th smallest exact distance among the slot's first k candidates
            for (int s = 0; s < rb.k; s++) {
                double e = exact[(size_t)slot * kp + s];
                if (!(e < kInf)) e = kInf;  // empty slot / NaN: nothing can be ruled out
                kth = fmax(kth, e);
            }
            const double na = rb.slot_max_na ? (double)rb.slot_max_na[slot] : (double)rb.max_na[0];
            if (scan_lower_bound(rb.cand_adist[pair], na, (double)rb.max_nb[0], rb.eps, rb.bound_mode, la, rb.inv_s, rb.ld_max) > kth) {
                if (lane == 0) exact[pair] = kInf;  // provably outside the top-k
                continue;
            }
            if (lane == 0) atomicAdd(&counters[1], 1ull);
        }
        const double e =
            warp_dtw_exact_long<BAND>(qmfcc + qoff[qid] * c, la, dmfcc + doff[idx] * c, lb, c, ring[warp], bnd + (size_t)gw * bnd_stride, lane, band);
        if (lane == 0) exact[pair] = e;
    }
}

// ---------------------------------------------------------------------------------------------------------------
// Second chance for the queries the packed-half scan's merged candidate list could not certify (dtw_h2.cu, <= 32 x <= 32
// frames). The scan leaves one ascending list of kp keys per (slice, query), and a per-query threshold `thr` = the smallest
// "worst kept key" any CTA with a full list reported (later CTAs start from it). Every pair that is in NO slice list was
// dropped against a threshold >= thr, so its scan distance is >= W = dist(thr) - usually far above the merged list's kp-th
// entry, because one slice holds ~1/2000 of the dictionary. The union of the slice lists therefore contains every pair below
// W: one warp per uncertified query walks it, refines in f64 every entry the bound cannot rule out against the current k-th
// exact distance, and certifies against W. No host round trip, no second scan (the re-run of ~47 queries through the fp32-DP
// tensor-core scan was 1.5 of config 4's 39 ms, and a fixed ~0.5 ms of every shard's step at 8 GPUs).
// ---------------------------------------------------------------------------------------------------------------
constexpr int kSecondQueue = 192;  // entries a warp can queue for refinement; a query with more stays uncertified
template <bool BAND>
__global__ void __launch_bounds__(64)
k_dtw_second_chance(const double* __restrict__ dmfcc, const uint64_t* __restrict__ doff, const double* __restrict__ qmfcc,
                    const uint64_t* __restrict__ qoff, int c, const uint32_t* __restrict__ group_qid, const uint32_t* __restrict__ cand_idx,
                    const unsigned long long* __restrict__ partial, uint32_t nlists, const unsigned long long* __restrict__ thr, uint32_t nslots,
                    int kp, int k, uint32_t index_base, const float* __restrict__ max_na, const float* __restrict__ max_nb, double eps,
                    const float* __restrict__ slot_max_na, int bound_mode, double inv_s, uint8_t* __restrict__ uncert_flag,
                    uint32_t* __restrict__ out_idx, double* __restrict__ out_dist, unsigned long long* __restrict__ counters, uint32_t band) {
    __shared__ double scost[2][32 * 32];
    __shared__ double squery[2][32 * SS_MAX_NCOEFFS];
    __shared__ uint32_t squeue[2][kSecondQueue];
    __shared__ uint32_t scount[2];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t slot = blockIdx.x * 2 + warp;
    if (slot >= nslots) return;  // warp-uniform from here on
    const uint32_t qid = group_qid[slot];
    if (qid == 0xFFFFFFFFu || !uncert_flag[qid]) return;
    const double na = slot_max_na ? (double)slot_max_na[slot] : (double)max_na[0];
    const double nb = (double)max_nb[0];
    const double* a = qmfcc + qoff[qid] * c;
    const int la = (int)(qoff[qid + 1] - qoff[qid]);
    const ScanBound bound = make_scan_bound(na, nb, eps, bound_mode, la, inv_s);
    // current top-k (the k best of the merged list's kp candidates, exact)
    double dv[SS_MAX_TOPK];
    uint32_t iv[SS_MAX_TOPK];
    int n = 0;
    for (int s = 0; s < k; s++) {
        const uint32_t ii = out_idx[(size_t)qid * k + s];
        if (ii == 0xFFFFFFFFu) break;
        iv[n] = ii - index_base;
        dv[n] = out_dist[(size_t)qid * k + s];
        n++;
    }
    double kth = n >= k ? dv[k - 1] : kInf;
    const uint32_t my_cand = lane < kp ? cand_idx[(size_t)slot * kp + lane] : 0xFFFFFFFFu;  // already refined
    if (lane == 0) scount[warp] = 0;
    for (int e = lane; e < la * c; e += 32) squery[warp][e] = a[e];
    __syncwarp();
    // ---- walk the slice lists: queue every entry the bound cannot rule out and the first pass did not refine ----------------
    for (uint32_t l = lane; l < ((nlists + 31) & ~31u); l += 32) {
        for (int s = 0; s < kp; s++) {
            unsigned long long key = 0xFFFFFFFFFFFFFFFFull;
            if (l < nlists) key = __ldg(partial + ((size_t)l * nslots + slot) * kp + s);
            bool want = false;
            if (key != 0xFFFFFFFFFFFFFFFFull) {
                const uint32_t o = (uint32_t)(key >> 32);
                const float dist = __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
                want = !(bound.lower(dist) > kth);
            }
            if (!__any_sync(0xffffffffu, want)) break;  // lists ascend: nothing further down any of these 32 lists qualifies
            const uint32_t idx = (uint32_t)key;
            bool seen = false;
            for (int j = 0; j < kp; j++) seen |= __shfl_sync(0xffffffffu, my_cand, j) == idx;  // (all lanes take part)
            want = want && !seen;
            if (want) {
                const uint32_t pos = atomicAdd(&scount[warp], 1u);
                if (pos < (uint32_t)kSecondQueue) squeue[warp][pos] = idx;
            }
        }
    }
    __syncwarp();
    const uint32_t nqueued = scount[warp];
    if (nqueued > (uint32_t)kSecondQueue) return;  // stays uncertified: the host re-runs it
    // ---- refine the queue (exact f64, the oracle's arithmetic), keeping the (distance, index) top-k --------------------------
    for (uint32_t e = 0; e < nqueued; e++) {
        const uint32_t idx = squeue[warp][e];
        const double ex = warp_dtw_exact<BAND>(squery[warp], la, dmfcc + doff[idx] * c, (int)(doff[idx + 1] - doff[idx]), c, scost[warp], lane, band);
        if (!(ex < kInf)) continue;
        if (n == k && !(ex < dv[k - 1] || (ex == dv[k - 1] && idx < iv[k - 1]))) continue;
        int pos = n < k ? n : k - 1;
        while (pos > 0 && (ex < dv[pos - 1] || (ex == dv[pos - 1] && idx < iv[pos - 1]))) {
            dv[pos] = dv[pos - 1];
            iv[pos] = iv[pos - 1];
            pos--;
        }
        dv[pos] = ex;
        iv[pos] = idx;
        if (n < k) n++;
    }
    kth = n >= k ? dv[k - 1] : kInf;
    // ---- certify against W: every pair outside the union of the slice lists has scan distance >= W -------------------------
    const unsigned long long t = thr[slot];
    float w = __int_as_float(0x7f800000);  // no CTA kept a full list: every (finite) pair is in the union
    if (t != 0xFFFFFFFFFFFFFFFFull) {
        const uint32_t o = (uint32_t)(t >> 32);
        w = __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
    }
    const bool certified = bound.lower(w) > kth;
    if (lane == 0) {
        for (int s = 0; s < k; s++) {
            out_idx[(size_t)qid * k + s] = s < n ? iv[s] + index_base : 0xFFFFFFFFu;
            out_dist[(size_t)qid * k + s] = s < n ? dv[s] : kInf;
        }
        if (certified) {
            uncert_flag[qid] = 0;
            atomicAdd(&counters[0], ~0ull);  // -1
            atomicAdd(&counters[2], 1ull);
        }
    }
}

// The same for sequences of more than 32 frames (bound_mode 3), one CTA of 8 warps per uncertified query: a long pair takes a warp
// 0.1 - 0.5 ms, so the queue is refined by the CTA's warps in parallel (each with its own cost ring and boundary row), then
// thread 0 folds the results into the top-k and certifies.
constexpr int kSecondWarps = 8;
template <bool BAND>
__global__ void __launch_bounds__(kSecondWarps * 32)
k_dtw_second_chance_long(const double* __restrict__ dmfcc, const uint64_t* __restrict__ doff, const double* __restrict__ qmfcc,
                         const uint64_t* __restrict__ qoff, int c, const uint32_t* __restrict__ group_qid, const uint32_t* __restrict__ cand_idx,
                         const unsigned long long* __restrict__ partial, uint32_t nlists, const unsigned long long* __restrict__ thr,
                         uint32_t nslots, int kp, int k, uint32_t index_base, const float* __restrict__ max_na, const float* __restrict__ max_nb,
                         double eps, const float* __restrict__ slot_max_na, int bound_mode, double inv_s, int ld_max, double* __restrict__ bnd,
                         uint32_t bnd_stride, uint32_t bnd_rows_cap, uint8_t* __restrict__ uncert_flag, uint32_t* __restrict__ out_idx,
                         double* __restrict__ out_dist, unsigned long long* __restrict__ counters, uint32_t band) {
    extern __shared__ __align__(16) unsigned char second_smem[];
    double* rings = reinterpret_cast<double*>(second_smem);                 // [warps][64 * 32]
    double* sexact = rings + kSecondWarps * 64 * 32;                         // [kSecondQueue]
    uint32_t* squeue = reinterpret_cast<uint32_t*>(sexact + kSecondQueue);   // [kSecondQueue]
    __shared__ uint32_t scount;
    __shared__ unsigned long long srow;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t slot = blockIdx.x;
    const uint32_t qid = group_qid[slot];
    if (qid == 0xFFFFFFFFu || !uncert_flag[qid]) return;  // CTA-uniform
    if (threadIdx.x == 0) {
        scount = 0;
        srow = atomicAdd(&counters[3], (unsigned long long)kSecondWarps);
    }
    __syncthreads();
    if (srow + kSecondWarps > bnd_rows_cap) return;  // no boundary rows left: stays uncertified
    double* my_bnd = bnd + (size_t)(srow + warp) * bnd_stride;
    const double na = slot_max_na ? (double)slot_max_na[slot] : (double)max_na[0];
    const double nb = (double)max_nb[0];
    const double* a = qmfcc + qoff[qid] * c;
    const int la = (int)(qoff[qid + 1] - qoff[qid]);
    const ScanBound bound = make_scan_bound(na, nb, eps, bound_mode, la, inv_s, ld_max);
    double kth = out_idx[(size_t)qid * k + k - 1] != 0xFFFFFFFFu ? out_dist[(size_t)qid * k + k - 1] : kInf;
    const uint32_t my_cand = lane < kp ? cand_idx[(size_t)slot * kp + lane] : 0xFFFFFFFFu;  // already refined
    // ---- walk the slice lists (32 lists per warp and round) ------------------------------------------------------------------
    const uint32_t lround = kSecondWarps * 32;
    for (uint32_t l0 = 0; l0 < nlists; l0 += lround) {
        const uint32_t l = l0 + warp * 32 + lane;
        for (int s = 0; s < kp; s++) {
            unsigned long long key = 0xFFFFFFFFFFFFFFFFull;
            if (l < nlists) key = __ldg(partial + ((size_t)l * nslots + slot) * kp + s);
            bool want = false;
            if (key != 0xFFFFFFFFFFFFFFFFull) {
                const uint32_t o = (uint32_t)(key >> 32);
                const float dist = __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
                want = !(bound.lower(dist) > kth);
            }
            if (!__any_sync(0xffffffffu, want)) break;  // lists ascend
            const uint32_t idx = (uint32_t)key;
            bool seen = false;
            for (int j = 0; j < kp; j++) seen |= __shfl_sync(0xffffffffu, my_cand, j) == idx;
            want = want && !seen;
            if (want) {
                const uint32_t pos = atomicAdd(&scount, 1u);
                if (pos < (uint32_t)kSecondQueue) squeue[pos] = idx;
            }
        }
    }
    __syncthreads();
    const uint32_t nqueued = scount;
    if (nqueued > (uint32_t)kSecondQueue) return;  // stays uncertified: the host re-runs it
    for (uint32_t e = warp; e < nqueued; e += kSecondWarps) {
        const uint32_t idx = squeue[e];
        const double ex = warp_dtw_exact_long<BAND>(a, la, dmfcc + doff[idx] * c, (int)(doff[idx + 1] - doff[idx]), c, rings + warp * 64 * 32, my_bnd,
                                                    lane, band);
        if (lane == 0) sexact[e] = ex;
    }
    __syncthreads();
    if (threadIdx.x != 0) return;
    double dv[SS_MAX_TOPK];
    uint32_t iv[SS_MAX_TOPK];
    int n = 0;
    for (int s = 0; s < k; s++) {
        const uint32_t ii = out_idx[(size_t)qid * k + s];
        if (ii == 0xFFFFFFFFu) break;
        iv[n] = ii - index_base;
        dv[n] = out_dist[(size_t)qid * k + s];
        n++;
    }
    for (uint32_t e = 0; e < nqueued; e++) {
        const uint32_t idx = squeue[e];
        const double ex = sexact[e];
        if (!(ex < kInf)) continue;
        if (n == k && !(ex < dv[k - 1] || (ex == dv[k - 1] && idx < iv[k - 1]))) continue;
        int pos = n < k ? n : k - 1;
        while (pos > 0 && (ex < dv[pos - 1] || (ex == dv[pos - 1] && idx < iv[pos - 1]))) {
            dv[pos] = dv[pos - 1];
            iv[pos] = iv[pos - 1];
            pos--;
        }
        dv[pos] = ex;
        iv[pos] = idx;
        if (n < k) n++;
    }
    kth = n >= k ? dv[k - 1] : kInf;
    const unsigned long long t = thr[slot];
    float w = __int_as_float(0x7f800000);
    if (t != 0xFFFFFFFFFFFFFFFFull) {
        const uint32_t o = (uint32_t)(t >> 32);
        w = __uint_as_float((o & 0x80000000u) ? (o & 0x7FFFFFFFu) : ~o);
    }
    for (int s = 0; s < k; s++) {
        out_idx[(size_t)qid * k + s] = s < n ? iv[s] + index_base : 0xFFFFFFFFu;
        out_dist[(size_t)qid * k + s] = s < n ? dv[s] : kInf;
    }
    if (bound.lower(w) > kth) {
        uncert_flag[qid] = 0;
        atomicAdd(&counters[0], ~0ull);  // -1
        atomicAdd(&counters[2], 1ull);
    }
}

int dtw_second_chance(ss_dict* d, ss_queries* q, int k, int kp, uint32_t nslots, const uint32_t* d_slot_qid, const unsigned long long* d_partial,
                      uint32_t nlists, const unsigned long long* d_thr, double eps, const float* d_max_na, const float* d_max_nb,
                      const float* d_slot_max_na, int bound_mode, uint8_t* d_uncert_flag, uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    if (!nslots) return SS_OK;
    if (d->max_len > 32 || q->max_len > 32) {
        const uint32_t stride = (std::max<uint32_t>(q->max_len, 1) + 15) & ~15u;
        const uint32_t rows_cap = (uint32_t)std::max<uint64_t>(kSecondWarps, std::min<uint64_t>((uint64_t)nslots * kSecondWarps, (4ull << 20) / stride));
        SS_CUDA(ctx, d->d_second_bnd.reserve((size_t)rows_cap * stride));  // <= 32 MB of boundary rows
        const size_t smem = (size_t)kSecondWarps * 64 * 32 * sizeof(double) + kSecondQueue * (sizeof(double) + sizeof(uint32_t));
        const auto kern = d->dtw_band ? k_dtw_second_chance_long<true> : k_dtw_second_chance_long<false>;
        SS_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        kern<<<nslots, kSecondWarps * 32, smem, ctx->stream>>>(
            d->d_mfcc.p, d->d_off.p, q->d_mfcc.p, q->d_off.p, d->c, d_slot_qid, d->d_cand_idx.p, d_partial, nlists, d_thr, nslots, kp, std::min(k, kp),
            d->index_base, d_max_na, d_max_nb, eps, d_slot_max_na, bound_mode, d->h2_bound_inv_s, (int)d->max_len, d->d_second_bnd.p, stride, rows_cap,
            d_uncert_flag, d_out_idx, d_out_dist, d->d_counters.p, d->dtw_band);
    } else {
        (d->dtw_band ? k_dtw_second_chance<true> : k_dtw_second_chance<false>)<<<ceil_div(nslots, 2), 64, 0, ctx->stream>>>(
            d->d_mfcc.p, d->d_off.p, q->d_mfcc.p, q->d_off.p, d->c, d_slot_qid, d->d_cand_idx.p, d_partial, nlists, d_thr, nslots, kp, std::min(k, kp),
            d->index_base, d_max_na, d_max_nb, eps, d_slot_max_na, bound_mode, d->h2_bound_inv_s, d_uncert_flag, d_out_idx, d_out_dist, d->d_counters.p,
            d->dtw_band);
    }
    SS_LAUNCHED(ctx);
    return SS_OK;
}

__global__ void k_dtw_finalize(const uint32_t* __restrict__ cand_idx, const float* __restrict__ cand_adist,
                               const double* __restrict__ exact, const uint32_t* __restrict__ group_qid, uint32_t nslots, int kp,
                               int k, uint32_t index_base, const float* __restrict__ max_na, const float* __restrict__ max_nb, double eps,
                               const float* __restrict__ slot_max_na, int bound_mode, double inv_s, int ld_max,
                               const uint64_t* __restrict__ qoff, uint8_t* __restrict__ uncert_flag,
                               uint32_t* __restrict__ out_idx, double* __restrict__ out_dist, unsigned long long* __restrict__ counters) {
    const uint32_t slot = blockIdx.x * blockDim.x + threadIdx.x;
    if (slot >= nslots) return;
    const uint32_t qid = group_qid[slot];
    if (qid == 0xFFFFFFFFu) return;
    double dv[kMaxKeep];
    uint32_t iv[kMaxKeep];
    int n = 0;
    for (int s = 0; s < kp; s++) {  // insertion sort by (distance, index); NaN / inf candidates are dropped
        const double dd = exact[(size_t)slot * kp + s];
        const uint32_t ii = cand_idx[(size_t)slot * kp + s];
        if (ii == 0xFFFFFFFFu || !(dd < kInf)) continue;
        int pos = n;
        while (pos > 0 && (dd < dv[pos - 1] || (dd == dv[pos - 1] && ii < iv[pos - 1]))) {
            dv[pos] = dv[pos - 1];
            iv[pos] = iv[pos - 1];
            pos--;
        }
        dv[pos] = dd;
        iv[pos] = ii;
        n++;
    }
    for (int s = 0; s < k; s++) {
        out_idx[(size_t)qid * k + s] = s < n ? iv[s] + index_base : 0xFFFFFFFFu;
        out_dist[(size_t)qid * k + s] = s < n ? dv[s] : kInf;
    }
    // certification: every pair X outside the candidate list has scan distance >= the list's worst entry w, and
    //   bound_mode 0 (fp32 scan):  |scan - exact| <= E = eps (max|a|^2 + max|b|^2)            => exact(X) >= w - E
    //   bound_mode 1 (fp16 scan):  the scan is the DTW of the fp16-ROUNDED frames (products of fp16 values are exact in
    //     fp32), and for every cell sqrt(c) >= sqrt(c~) - delta with delta = |a - a~| + |b - b~| <= 2^-11 (|a| + |b|)
    //     (triangle inequality). Summing along the exact optimum and using Cauchy-Schwarz over its <= Lq+Ld cells:
    //                              exact(X) >= w - 2 delta sqrt(w) - E32,   E32 = fp32 accumulation slack
    // If that lower bound exceeds the exact k-th distance found among the candidates, the reported top-k is THE f64 top-k.
    const float worst = cand_adist[(size_t)slot * kp + kp - 1];
    bool uncertified = false;
    // (bound_mode 2 / 3: a list that is not full does NOT mean every pair is in it - an overflowed pair reads +inf)
    if (bound_mode >= 2 || worst < __int_as_float(0x7f800000)) {
        const double kth = n >= k ? dv[k - 1] : kInf;
        const double na = slot_max_na ? (double)slot_max_na[slot] : (double)max_na[0];
        const double nb = (double)max_nb[0];
        double lower;
        lower = scan_lower_bound(worst, na, nb, eps, bound_mode, (int)(qoff[qid + 1] - qoff[qid]), inv_s, ld_max);
        uncertified = !(lower > kth);
        if (uncertified) atomicAdd(&counters[0], 1ull);
    }
    if (uncert_flag) uncert_flag[qid] = uncertified ? 1 : 0;
}

int dtw_rescore_finalize(ss_dict* d, ss_queries* q, int k, int kp, uint32_t nslots, const uint32_t* d_slot_qid, double eps,
                         const float* d_max_na, const float* d_max_nb, const float* d_slot_max_na, int bound_mode, uint8_t* d_uncert_flag,
                         uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    // queries without a frame never reach a slot: their rows keep (inf, 0xFFFFFFFF). Only launched when such queries exist.
    if (q->nq && q->nonempty < q->nq) {
        k_fill_result<<<ceil_div((long long)q->nq * k, 256), 256, 0, ctx->stream>>>(d_out_idx, d_out_dist, q->nq * (size_t)k,
                                                                                   0xFFFFFFFFu, kInf);
        SS_LAUNCHED(ctx);
    }
    SS_CUDA(ctx, d->d_counters.reserve(4));
    SS_CUDA(ctx, cudaMemsetAsync(d->d_counters.p, 0, 4 * sizeof(unsigned long long), ctx->stream));
    if (!nslots || !d->ntiles) return SS_OK;
    if (d->max_len <= 32 && q->max_len <= 32) {  // one warp per query slot does the whole refine
        (d->dtw_band ? k_dtw_refine_warp<true> : k_dtw_refine_warp<false>)<<<ceil_div(nslots, 4), 128, 0, ctx->stream>>>(
            d->d_mfcc.p, d->d_off.p, q->d_mfcc.p, q->d_off.p, d->c, d_slot_qid, d->d_cand_idx.p, d->d_cand_adist.p, nslots, kp, std::min(k, kp),
            d->index_base, d_max_na, d_max_nb, eps, d_slot_max_na, bound_mode, d->h2_bound_inv_s, d_uncert_flag, d_out_idx, d_out_dist,
            d->d_counters.p, d->dtw_band);
        SS_LAUNCHED(ctx);
        return SS_OK;
    }
    SS_CUDA(ctx, d->d_cand_exact.reserve(nslots * (uint32_t)kp));
    // one warp per pair: the k best of every slot, then the others unless the scan's bound rules them out, then the sort
    const uint32_t stride = (std::max<uint32_t>(q->max_len, 1) + 15) & ~15u;
    const uint32_t max_ctas = (uint32_t)ctx->sm_count * 6;  // 33 KB of shared memory each
    SS_CUDA(ctx, d->d_rescore_rows.reserve((size_t)max_ctas * 2 * stride));
    for (int phase = 0; phase < 2; phase++) {
        const int s_begin = phase ? std::min(k, kp) : 0, s_count = phase ? kp - std::min(k, kp) : std::min(k, kp);
        if (s_count <= 0) continue;
        RescoreBound rb = {phase ? d->d_cand_adist.p : nullptr, d_max_na, d_max_nb, d_slot_max_na, eps, bound_mode, std::min(k, kp), d->h2_bound_inv_s,
                           (int)d->max_len};
        const uint32_t nt = nslots * (uint32_t)s_count;
        (d->dtw_band ? k_dtw_rescore_warp<true> : k_dtw_rescore_warp<false>)<<<std::min<uint32_t>(max_ctas, ceil_div(nt, 2)), 64, 0, ctx->stream>>>(
            d->d_mfcc.p, d->d_off.p, q->d_mfcc.p, q->d_off.p, d->c, d_slot_qid, d->d_cand_idx.p, nt, kp, s_begin, s_count, rb, d->d_rescore_rows.p,
            stride, d->d_cand_exact.p, d->d_counters.p, d->dtw_band);
        SS_LAUNCHED(ctx);
    }
    k_dtw_finalize<<<ceil_div(nslots, 128), 128, 0, ctx->stream>>>(d->d_cand_idx.p, d->d_cand_adist.p, d->d_cand_exact.p, d_slot_qid, nslots, kp, k,
                                                                  d->index_base, d_max_na, d_max_nb, eps, d_slot_max_na, bound_mode, d->h2_bound_inv_s,
                                                                  (int)d->max_len, q->d_off.p, d_uncert_flag, d_out_idx, d_out_dist, d->d_counters.p);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// exhaustive f64 DTW: (uncertified query u, every dictionary segment). One warp per pair (warp_dtw_exact_long); then one block
// per query selects its top-k by (distance, index).
// ---------------------------------------------------------------------------------------------------------------
template <bool BAND>
__global__ void __launch_bounds__(64)
k_dtw_pairs_exact_warp(const double* __restrict__ dmfcc, const uint64_t* __restrict__ doff, const double* __restrict__ qmfcc,
                       const uint64_t* __restrict__ qoff, int c, const uint32_t* __restrict__ qids, uint32_t nu, uint32_t nseg,
                       double* __restrict__ bnd, uint32_t bnd_stride, double* __restrict__ exact, uint32_t band) {
    __shared__ double ring[2][64 * 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t gw = blockIdx.x * 2 + warp, nw = gridDim.x * 2;
    const uint64_t npairs = (uint64_t)nu * nseg;
    for (uint64_t t = gw; t < npairs; t += nw) {  // warp-uniform; consecutive warps take consecutive segments of one query
        const uint32_t u = (uint32_t)(t / nseg), sidx = (uint32_t)(t % nseg);
        const uint32_t qid = qids[u];
        const int la = (int)(qoff[qid + 1] - qoff[qid]), lb = (int)(doff[sidx + 1] - doff[sidx]);
        const double e =
            warp_dtw_exact_long<BAND>(qmfcc + qoff[qid] * c, la, dmfcc + doff[sidx] * c, lb, c, ring[warp], bnd + (size_t)gw * bnd_stride, lane, band);
        if (lane == 0) exact[(size_t)u * nseg + sidx] = e;
    }
}

__global__ void __launch_bounds__(256)
k_dtw_select_exact(const double* __restrict__ exact, uint32_t nseg, int k, const uint32_t* __restrict__ qids, uint32_t index_base,
                   uint32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    __shared__ double sd[256 * SS_MAX_TOPK];
    __shared__ uint32_t si[256 * SS_MAX_TOPK];
    const uint32_t u = blockIdx.x, t = threadIdx.x;
    double dv[SS_MAX_TOPK];
    uint32_t iv[SS_MAX_TOPK];
    int n = 0;
    auto push = [&](double dd, uint32_t ii) {
        if (!(dd < kInf)) return;
        if (n == k && !(dd < dv[k - 1] || (dd == dv[k - 1] && ii < iv[k - 1]))) return;
        int pos = n < k ? n : k - 1;
        while (pos > 0 && (dd < dv[pos - 1] || (dd == dv[pos - 1] && ii < iv[pos - 1]))) {
            dv[pos] = dv[pos - 1];
            iv[pos] = iv[pos - 1];
            pos--;
        }
        dv[pos] = dd;
        iv[pos] = ii;
        if (n < k) n++;
    };
    for (uint32_t s = t; s < nseg; s += 256) push(exact[(size_t)u * nseg + s], s);
    for (int s = 0; s < k; s++) {
        sd[t * SS_MAX_TOPK + s] = s < n ? dv[s] : kInf;
        si[t * SS_MAX_TOPK + s] = s < n ? iv[s] : 0xFFFFFFFFu;
    }
    __syncthreads();
    if (t == 0) {
        n = 0;
        for (int w = 0; w < 256; w++)
            for (int s = 0; s < k; s++)
                if (si[w * SS_MAX_TOPK + s] != 0xFFFFFFFFu) push(sd[w * SS_MAX_TOPK + s], si[w * SS_MAX_TOPK + s]);
        const uint32_t qid = qids[u];
        for (int s = 0; s < k; s++) {
            out_idx[(size_t)qid * k + s] = s < n ? iv[s] + index_base : 0xFFFFFFFFu;
            out_dist[(size_t)qid * k + s] = s < n ? dv[s] : kInf;
        }
    }
}

int dtw_exhaustive_match(ss_dict* d, ss_queries* q, int k, const std::vector<uint32_t>& subset, uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    const uint32_t nseg = (uint32_t)d->nseg;
    const uint64_t budget = 32ull << 20;  // doubles of the distance table (256 MB)
    const uint32_t ubatch = (uint32_t)std::max<uint64_t>(1, std::min<uint64_t>(subset.size(), budget / std::max<uint32_t>(nseg, 1)));
    SS_CUDA(ctx, d->d_exh_qid.reserve(subset.size()));
    SS_CUDA(ctx, cudaMemcpyAsync(d->d_exh_qid.p, subset.data(), subset.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    SS_CUDA(ctx, d->d_exh_dist.reserve((size_t)ubatch * nseg));
    const uint32_t stride = (std::max<uint32_t>(q->max_len, 1) + 15) & ~15u;
    const uint32_t max_ctas = (uint32_t)ctx->sm_count * 6;
    SS_CUDA(ctx, d->d_rescore_rows.reserve((size_t)max_ctas * 2 * stride));
    for (size_t u0 = 0; u0 < subset.size(); u0 += ubatch) {
        const uint32_t nu = (uint32_t)std::min<size_t>(ubatch, subset.size() - u0);
        const uint64_t npairs = (uint64_t)nu * nseg;
        if (npairs) {
            (d->dtw_band ? k_dtw_pairs_exact_warp<true> : k_dtw_pairs_exact_warp<false>)<<<(unsigned)std::min<uint64_t>(max_ctas, (npairs + 1) / 2), 64, 0,
                                                                                            ctx->stream>>>(
                d->d_mfcc.p, d->d_off.p, q->d_mfcc.p, q->d_off.p, d->c, d->d_exh_qid.p + u0, nu, nseg, d->d_rescore_rows.p, stride, d->d_exh_dist.p,
                d->dtw_band);
            SS_LAUNCHED(ctx);
        }
        k_dtw_select_exact<<<nu, 256, 0, ctx->stream>>>(d->d_exh_dist.p, nseg, k, d->d_exh_qid.p + u0, d->index_base, d_out_idx, d_out_dist);
        SS_LAUNCHED(ctx);
    }
    SS_CUDA(ctx, cudaMemsetAsync(d->d_counters.p, 0, sizeof(unsigned long long), ctx->stream));  // everything is exact now
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // `subset` is read by the async copy above
    return SS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// merge of per-shard top-k lists, list-major [nlists][nq][k] -> [nq][k]; (distance, index) lexicographic
// ---------------------------------------------------------------------------------------------------------------
__global__ void k_topk_merge(const uint32_t* __restrict__ idx, const double* __restrict__ dist, int nlists, size_t nq, int k,
                             uint32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    const size_t qi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    double dv[SS_MAX_TOPK];
    uint32_t iv[SS_MAX_TOPK];
    int n = 0;
    for (int l = 0; l < nlists; l++)
        for (int s = 0; s < k; s++) {
            const double dd = dist[((size_t)l * nq + qi) * k + s];
            const uint32_t ii = idx[((size_t)l * nq + qi) * k + s];
            if (ii == 0xFFFFFFFFu || dd != dd) continue;
            if (n == k && !(dd < dv[k - 1] || (dd == dv[k - 1] && ii < iv[k - 1]))) continue;
            int pos = n < k ? n : k - 1;
            while (pos > 0 && (dd < dv[pos - 1] || (dd == dv[pos - 1] && ii < iv[pos - 1]))) {
                dv[pos] = dv[pos - 1];
                iv[pos] = iv[pos - 1];
                pos--;
            }
            dv[pos] = dd;
            iv[pos] = ii;
            if (n < k) n++;
        }
    for (int s = 0; s < k; s++) {
        out_idx[qi * k + s] = s < n ? iv[s] : 0xFFFFFFFFu;
        out_dist[qi * k + s] = s < n ? dv[s] : kInf;
    }
}

int topk_merge_dev(ss_ctx* ctx, const uint32_t* d_idx, const double* d_dist, int nlists, size_t nq, int k, uint32_t* d_out_idx,
                   double* d_out_dist) {
    if (k < 1 || k > SS_MAX_TOPK || nlists < 1) return set_error(ctx, SS_ERR_INVALID, "topk_merge: bad k / nlists");
    if (!nq) return SS_OK;
    k_topk_merge<<<ceil_div((long long)nq, 128), 128, 0, ctx->stream>>>(d_idx, d_dist, nlists, nq, k, d_out_idx, d_out_dist);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

// ---------------------------------------------------------------------------------------------------------------
// DTW alignment (ss_dict_align, spec in DESIGN.md §3.1e): the warping path of query p against dictionary segment seg_idx[p].
// The recurrences below are warp_dtw_exact / warp_dtw_exact_long with one addition: every cell also records which of its
// three neighbours the min chose, as 2 bits (0 diag, 1 up, 2 left; ties in that order), compared against the very value
// fmin(fmin(up, left), diag) returned. D's bits are the refine's, so the path is the oracle's path cell for cell.
//   <= 32 x <= 32 (k_dtw_align_warp): lane j owns column j, whose 32 rows of directions fit in one u64 register; the
//     backtrack is <= 63 steps of one shuffle of the current column's word.
//   longer (k_dtw_align_long, waves of pairs): per strip, lane j packs 32 rows of its column into a u64 and stores it to the
//     pair's direction block [strip][row / 32][lane], coalesced, once the whole warp has finished those rows. The backtrack
//     loads one 32 x 32 tile (one coalesced u64 per lane) whenever the path enters it, then shuffles within it.
// Paths are found from the end: cell s from the end goes to stage[last - s] of the pair's staging slot (last = its end),
// so a path lands in forward order without knowing its length first. A scan of the lengths then gives the offsets and
// k_dtw_align_compact packs the paths. Nothing is read back to the host.
// ---------------------------------------------------------------------------------------------------------------
constexpr uint32_t kAlignNone = 0xFFFFFFFFu;
constexpr uint64_t kAlignDirBudget = 256ull << 20;  // direction blocks + boundary rows of one wave of long pairs

struct AlignArgs {
    const double* dmfcc;
    const uint64_t* doff;
    uint32_t nseg, index_base;
    const double* qmfcc;
    const uint64_t* qoff;
    uint32_t nq;
    int c;
    const uint32_t* seg_idx;
    uint32_t wpad;  // max(longest segment, 1) - 1: pair p stages its path in [qoff[p] + p wpad, + Lq + wpad)
    uint2* stage;
    uint64_t* len;
    double* out_dist;
};

// the pair's two sides; false (the pair's empty result written) when there is nothing to align
__device__ __forceinline__ bool align_pair(const AlignArgs& A, uint32_t p, int lane, int* la, int* lb, uint32_t* s) {
    const uint32_t idx = A.seg_idx[p];
    *s = idx - A.index_base;
    const bool known = idx != kAlignNone && *s < A.nseg;
    *la = (int)(A.qoff[p + 1] - A.qoff[p]);
    *lb = known ? (int)(A.doff[*s + 1] - A.doff[*s]) : 0;
    if (known && *la && *lb) return true;
    if (lane == 0) {
        A.len[p] = 0;
        A.out_dist[p] = (idx == kAlignNone || known) ? kInf : __longlong_as_double(0x7ff8000000000000ll);  // out of range: NaN
    }
    return false;
}

__device__ __forceinline__ uint64_t align_dir(double up, double left, double diag, double m) {
    return diag == m ? 0ull : (up == m ? 1ull : 2ull);
}

// warp_dtw_exact (same loads, same operations in the same order) + the directions of lane `lane`'s column in *dirs
template <bool BAND>
__device__ __forceinline__ double warp_dtw_align(const double* __restrict__ sa, int la, const double* __restrict__ b, int lb, int c, double* cst,
                                                 int lane, uint64_t* dirs, uint32_t band) {
    double br[SS_MAX_NCOEFFS];
#pragma unroll
    for (int k = 0; k < SS_MAX_NCOEFFS; k++) br[k] = (k < c && lane < lb) ? b[(size_t)lane * c + k] : 0.0;
    int blo = 0, bhi = 0;
    if (BAND) band_rows(min(lane, lb - 1), la, lb, band, &blo, &bhi);
    for (int i = 0; i < la; i++) {
        double cost = 0.0;
#pragma unroll
        for (int k = 0; k < SS_MAX_NCOEFFS; k++)
            if (k < c) {
                const double dlt = sa[i * c + k] - br[k];
                cost = cost + dlt * dlt;
            }
        cst[i * 32 + lane] = cost;
    }
    __syncwarp();
    double cur = kInf, recv_prev = kInf, result = kInf;
    uint64_t w = 0;
    for (int step = 0; step < la + lb - 1; step++) {
        const double recv = __shfl_up_sync(0xffffffffu, cur, 1);
        const int i = step - lane;
        const bool active = lane < lb && i >= 0 && i < la;
        if (active) {
            const double up = cur;
            const double left = lane ? recv : kInf;
            const double diag = lane ? recv_prev : kInf;
            double m;
            if (i == 0 && lane == 0) m = 0.0;
            else m = fmin(fmin(up, left), diag);
            w |= align_dir(up, left, diag, m) << (2 * i);
            if (BAND && (i < blo || i > bhi)) cur = kInf;
            else cur = cst[i * 32 + lane] + m;
            if (i == la - 1 && lane == lb - 1) result = cur;
        }
        recv_prev = recv;
    }
    *dirs = w;
    result = __shfl_sync(0xffffffffu, result, lb - 1);
    return result / (double)(la + lb);
}

// one warp per pair, both sides <= 32 frames (the other pairs are k_dtw_align_long's)
template <bool BAND>
__global__ void __launch_bounds__(128) k_dtw_align_warp(AlignArgs A, uint32_t band) {
    __shared__ double scost[4][32 * 32];
    __shared__ double squery[4][32 * SS_MAX_NCOEFFS];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t p = blockIdx.x * 4 + warp;
    if (p >= A.nq) return;  // warp-uniform from here on
    int la, lb;
    uint32_t s;
    if (!align_pair(A, p, lane, &la, &lb, &s) || la > 32 || lb > 32) return;
    const int c = A.c;
    const double* a = A.qmfcc + A.qoff[p] * c;
    for (int e = lane; e < la * c; e += 32) squery[warp][e] = a[e];
    __syncwarp();
    uint64_t dirs;
    const double dist = warp_dtw_align<BAND>(squery[warp], la, A.dmfcc + A.doff[s] * c, lb, c, scost[warp], lane, &dirs, band);
    if (!(dist < kInf)) {  // NaN or inf: no path
        if (lane == 0) A.len[p] = 0, A.out_dist[p] = kInf;
        return;
    }
    // backtrack: lane (n & 31) keeps cell n from the end (n < 32 in keep0, else keep1)
    int i = la - 1, j = lb - 1, n = 0;
    uint2 keep0 = make_uint2(0, 0), keep1 = keep0;
    for (;;) {
        if (lane == (n & 31)) (n < 32 ? keep0 : keep1) = make_uint2((uint32_t)i, (uint32_t)j);
        n++;
        if (i == 0 && j == 0) break;
        const uint64_t w = __shfl_sync(0xffffffffu, dirs, j);
        const uint32_t dir = i == 0 ? 2u : j == 0 ? 1u : (uint32_t)(w >> (2 * i)) & 3u;
        i -= dir != 2u;
        j -= dir != 1u;
    }
    uint2* last = A.stage + A.qoff[p] + (uint64_t)p * A.wpad + (uint64_t)la + A.wpad - 1;
    if (lane < n) *(last - lane) = keep0;
    if (lane + 32 < n) *(last - 32 - lane) = keep1;
    if (lane == 0) A.len[p] = (uint64_t)n, A.out_dist[p] = dist;
}

// warp_dtw_exact_long (same loads, same operations in the same order) + the direction block `dir`, [strip][row / 32][lane].
// BAND: the same strip range; the words of row blocks outside it are not written, and no path cell reads them.
template <bool BAND>
__device__ __forceinline__ double warp_dtw_align_long(const double* __restrict__ a, int la, const double* __restrict__ b, int lb, int c,
                                                      double* __restrict__ ring, double* bnd, uint64_t* __restrict__ dir, int lane, uint32_t band) {
    double result = kInf;
    const int nstrips = (lb + 31) >> 5, nrb = (la + 31) >> 5;
    const int nsteps = la + 31;
    for (int s = 0; s < nstrips; s++) {
        const int col = 32 * s + lane;
        const bool colv = col < lb, first = s == 0, last = s == nstrips - 1;
        double br[SS_MAX_NCOEFFS];
#pragma unroll
        for (int k = 0; k < SS_MAX_NCOEFFS; k++) br[k] = (k < c && colv) ? b[(size_t)col * c + k] : 0.0;
        double cur = kInf, recv_prev = kInf, bl_prev = kInf;
        // at step t0 + r lane j is on row t0 + r - j: row block t0 / 32 - 1 (wprev) or t0 / 32 (wcur)
        uint64_t wprev = 0, wcur = 0;
        uint64_t* sdir = dir + (size_t)s * nrb * 32 + lane;
        int blo = 0, bhi = 0, rhi = 0, t0b = 0, t0e = nsteps;
        if (BAND) {
            band_rows(min(col, lb - 1), la, lb, band, &blo, &bhi);
            rhi = __shfl_sync(0xffffffffu, bhi, 31);
            t0b = __shfl_sync(0xffffffffu, blo, 0) & ~31;
            t0e = min(nsteps, rhi + 32);
        }
        __syncwarp();
        if (BAND && lane == 0 && !first && t0b > 0) bl_prev = bnd[t0b - 1];
        int t0 = t0b;
        for (; t0 < t0e; t0 += 32) {
            const int rows = min(32, (BAND ? rhi + 1 : la) - t0);
            int r = 0;
            for (; r + 4 <= rows; r += 4) {
                const double* ar = a + (size_t)(t0 + r) * c;
                double c0 = 0.0, c1 = 0.0, c2 = 0.0, c3 = 0.0;
#pragma unroll
                for (int k = 0; k < SS_MAX_NCOEFFS; k++)
                    if (k < c) {
                        const double d0 = ar[k] - br[k], d1 = ar[c + k] - br[k], d2 = ar[2 * c + k] - br[k], d3 = ar[3 * c + k] - br[k];
                        c0 = c0 + d0 * d0;
                        c1 = c1 + d1 * d1;
                        c2 = c2 + d2 * d2;
                        c3 = c3 + d3 * d3;
                    }
                double* dst = ring + ((t0 + r) & 63) * 32 + lane;
                dst[0] = c0, dst[32] = c1, dst[64] = c2, dst[96] = c3;
            }
            for (; r < rows; r++) {
                const double* ar = a + (size_t)(t0 + r) * c;
                double cost = 0.0;
#pragma unroll
                for (int k = 0; k < SS_MAX_NCOEFFS; k++)
                    if (k < c) {
                        const double dlt = ar[k] - br[k];
                        cost = cost + dlt * dlt;
                    }
                ring[((t0 + r) & 63) * 32 + lane] = cost;
            }
            __syncwarp();
            const int steps = min(32, nsteps - t0);
            double left_in = (lane == 0 && !first && t0 < la) ? bnd[t0] : kInf;
            for (int r = 0; r < steps; r++) {
                const int t = t0 + r;
                const double recv = __shfl_up_sync(0xffffffffu, cur, 1);
                const double left_now = left_in;
                if (r + 1 < steps) left_in = (lane == 0 && !first && t + 1 < la) ? bnd[t + 1] : kInf;
                const int i = t - lane;
                const bool active = colv && i >= 0 && i < la;
                if (active) {
                    const double up = cur;
                    const double left = lane ? recv : left_now;
                    const double diag = lane ? recv_prev : bl_prev;
                    double m;
                    if (first && i == 0 && lane == 0) m = 0.0;
                    else m = fmin(fmin(up, left), diag);
                    const uint64_t bits = align_dir(up, left, diag, m) << (2 * (i & 31));
                    if (i < t0) wprev |= bits;
                    else wcur |= bits;
                    if (BAND && (i < blo || i > bhi)) cur = kInf;
                    else cur = ring[(i & 63) * 32 + lane] + m;
                    if (last && i == la - 1 && col == lb - 1) result = cur;
                    if (!last && lane == 31) bnd[i] = cur;
                }
                bl_prev = left_now;
                recv_prev = recv;
            }
            __syncwarp();
            if (t0 >= 32) sdir[(size_t)((t0 >> 5) - 1) * 32] = wprev;  // every lane is past that row block
            wprev = wcur;
            wcur = 0;
        }
        const int rb_last = ((BAND ? t0 : nsteps) - 1) >> 5;
        if (rb_last < nrb) sdir[(size_t)rb_last * 32] = wprev;
        if (BAND && !last)
            for (int r = max(0, min(t0, nsteps) - 31) + lane; r < la; r += 32) bnd[r] = kInf;
    }
    result = __shfl_sync(0xffffffffu, result, (lb - 1) & 31);
    return result / (double)(la + lb);
}

// one warp per pair of the wave [p0, p0 + np) that has a side longer than 32 frames; the pair's direction block and
// boundary row are its own (dir_stride u64 words, bnd_stride doubles)
template <bool BAND>
__global__ void __launch_bounds__(64) k_dtw_align_long(AlignArgs A, uint32_t p0, uint32_t np, uint64_t* __restrict__ dir, uint64_t dir_stride,
                                                       double* __restrict__ bnd, uint32_t bnd_stride, uint32_t band) {
    __shared__ double ring[2][64 * 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t t = blockIdx.x * 2 + warp;
    if (t >= np) return;
    const uint32_t p = p0 + t;
    int la, lb;
    uint32_t s;
    if (!align_pair(A, p, -1, &la, &lb, &s) || (la <= 32 && lb <= 32)) return;  // (lane -1: k_dtw_align_warp wrote those)
    const int c = A.c;
    uint64_t* my_dir = dir + (size_t)t * dir_stride;
    const double dist = warp_dtw_align_long<BAND>(A.qmfcc + A.qoff[p] * c, la, A.dmfcc + A.doff[s] * c, lb, c, ring[warp],
                                                  bnd + (size_t)t * bnd_stride, my_dir, lane, band);
    if (!(dist < kInf)) {
        if (lane == 0) A.len[p] = 0, A.out_dist[p] = kInf;
        return;
    }
    const int nrb = (la + 31) >> 5;
    uint2* last = A.stage + A.qoff[p] + (uint64_t)p * A.wpad + (uint64_t)la + A.wpad - 1;
    int i = la - 1, j = lb - 1, ts = -1, trb = -1;
    uint32_t n = 0;
    uint64_t w = 0;
    uint2 keep = make_uint2(0, 0);
    for (;;) {
        if (lane == (int)(n & 31)) keep = make_uint2((uint32_t)i, (uint32_t)j);
        n++;
        if ((n & 31) == 0) *(last - (n - 32) - lane) = keep;  // lane l holds cell n - 32 + l from the end
        if (i == 0 && j == 0) break;
        if ((j >> 5) != ts || (i >> 5) != trb) {  // the path enters another 32 x 32 tile (warp-uniform)
            ts = j >> 5;
            trb = i >> 5;
            w = my_dir[((size_t)ts * nrb + trb) * 32 + lane];  // this lane's own store
        }
        const uint64_t wc = __shfl_sync(0xffffffffu, w, j & 31);
        const uint32_t d = i == 0 ? 2u : j == 0 ? 1u : (uint32_t)(wc >> (2 * (i & 31))) & 3u;
        i -= d != 2u;
        j -= d != 1u;
    }
    const uint32_t rem = n & 31;
    if ((uint32_t)lane < rem) *(last - (n - rem) - lane) = keep;
    if (lane == 0) A.len[p] = (uint64_t)n, A.out_dist[p] = dist;
}

// one warp per pair: its path from the end of its staging slot to out_path[out_off[p] ..), as (i, j) uint32 pairs
__global__ void __launch_bounds__(256) k_dtw_align_compact(const uint2* __restrict__ stage, const uint64_t* __restrict__ qoff, uint32_t nq,
                                                           uint32_t wpad, const uint64_t* __restrict__ out_off, uint32_t* __restrict__ out) {
    const int lane = threadIdx.x & 31;
    const uint32_t p = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (p >= nq) return;
    const uint64_t o = out_off[p], n = out_off[p + 1] - o;
    const uint2* src = stage + qoff[p] + (uint64_t)p * wpad + (qoff[p + 1] - qoff[p]) + wpad - n;
    for (uint64_t e = lane; e < n; e += 32) {
        const uint2 v = src[e];
        out[2 * (o + e)] = v.x;
        out[2 * (o + e) + 1] = v.y;
    }
}

int dtw_align_dev(ss_dict* d, const double* d_qmfcc, const uint64_t* d_qoff, const uint64_t* h_qoff, size_t nq, const uint32_t* d_seg_idx,
                  uint32_t* d_out_path, uint64_t* d_out_off, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    SS_CUDA(ctx, cudaMemsetAsync(d_out_off, 0, sizeof(uint64_t), ctx->stream));
    if (!nq) return SS_OK;
    const uint32_t ld_max = std::max<uint32_t>(d->max_len, 1), wpad = ld_max - 1;
    uint32_t lq_max = 0;
    for (size_t p = 0; p < nq; p++) lq_max = std::max<uint32_t>(lq_max, (uint32_t)(h_qoff[p + 1] - h_qoff[p]));
    SS_CUDA(ctx, d->d_align_stage.reserve(h_qoff[nq] + nq * (size_t)wpad)  /* (offsets start at 0) */);
    SS_CUDA(ctx, d->d_align_len.reserve(nq));
    AlignArgs A{d->d_mfcc.p, d->d_off.p, (uint32_t)d->nseg, d->index_base, d_qmfcc, d_qoff, (uint32_t)nq, d->c, d_seg_idx, wpad,
                d->d_align_stage.p, d->d_align_len.p, d_out_dist};
    // waves of long pairs, sized from host-known bounds only: (the wave's longest query) x (the longest segment)
    struct Wave {
        uint32_t p0, np, lq;
    };
    std::vector<Wave> waves;
    if (lq_max > 32 || ld_max > 32) {
        const uint64_t nsb = (ld_max + 31) / 32;
        auto bytes_of = [&](uint64_t lq) { return (lq + 31) / 32 * nsb * 32 * sizeof(uint64_t) + lq * sizeof(double); };
        for (size_t p0 = 0; p0 < nq;) {
            uint32_t lq = 0;
            size_t p1 = p0;
            for (; p1 < nq; p1++) {
                const uint32_t m = std::max<uint32_t>(lq, (uint32_t)(h_qoff[p1 + 1] - h_qoff[p1]));
                if (p1 > p0 && (p1 - p0 + 1) * bytes_of(m) > kAlignDirBudget) break;  // (one pair alone may exceed the budget)
                lq = m;
            }
            if (lq > 32 || (lq > 0 && ld_max > 32)) waves.push_back({(uint32_t)p0, (uint32_t)(p1 - p0), lq});
            p0 = p1;
        }
        size_t dir_words = 0, bnd_rows = 0;
        for (const Wave& w : waves) {
            dir_words = std::max<size_t>(dir_words, (size_t)w.np * ((w.lq + 31) / 32) * nsb * 32);
            bnd_rows = std::max<size_t>(bnd_rows, (size_t)w.np * w.lq);
        }
        if (!waves.empty()) {
            SS_CUDA(ctx, d->d_align_dir.reserve(dir_words));
            SS_CUDA(ctx, d->d_align_bnd.reserve(bnd_rows));
        }
    }
    size_t cub_bytes = 0;
    SS_CUDA(ctx, cub::DeviceScan::InclusiveSum(nullptr, cub_bytes, d->d_align_len.p, d_out_off + 1, (int)nq, ctx->stream));
    SS_CUDA(ctx, d->d_align_cub.reserve(cub_bytes));

    (d->dtw_band ? k_dtw_align_warp<true> : k_dtw_align_warp<false>)<<<ceil_div((long long)nq, 4), 128, 0, ctx->stream>>>(A, d->dtw_band);
    SS_LAUNCHED(ctx);
    for (const Wave& w : waves) {
        const uint64_t dir_stride = (uint64_t)((w.lq + 31) / 32) * ((ld_max + 31) / 32) * 32;
        (d->dtw_band ? k_dtw_align_long<true> : k_dtw_align_long<false>)<<<ceil_div(w.np, 2), 64, 0, ctx->stream>>>(A, w.p0, w.np, d->d_align_dir.p,
                                                                                                                 dir_stride, d->d_align_bnd.p, w.lq,
                                                                                                                 d->dtw_band);
        SS_LAUNCHED(ctx);
    }
    SS_CUDA(ctx, cub::DeviceScan::InclusiveSum(d->d_align_cub.p, cub_bytes, d->d_align_len.p, d_out_off + 1, (int)nq, ctx->stream));
    ctx->launches++;
    k_dtw_align_compact<<<ceil_div((long long)nq, 8), 256, 0, ctx->stream>>>(d->d_align_stage.p, d_qoff, (uint32_t)nq, wpad, d_out_off, d_out_path);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

}  // namespace ss
