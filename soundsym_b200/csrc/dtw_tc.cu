// dtw_tc.cu — tensor-core variant of the DTW scan (filter stage only; merge / f64 refine / certification are shared
// with dtw.cu + exact.cu). Used when every dictionary segment and every query has <= 32 frames; otherwise dtw.cu's fp32
// scan runs.
//
// Idea: the local-cost matrix is a K = 13 contraction, c(i,j) = |a_i|^2 + |b_j|^2 - 2 a_i.b_j. One tcgen05.mma per
// (dictionary tile, query row i) computes, for the CTA's 128 queries at once, the costs of row i against the 128 columns
// of the tile (4 slots x 32 columns):
//     D[m, n] = sum_k A_i[m, k] * B[n, k],   A_i[m, :] = [-2 a^(m)_i (13), s, s, rd(|a_i|^2 / s)]   (fp16, K-major, no swizzle)
//                                            B[n, :]   = [ b_n (13), (|b_n|^2/s)_hi, (|b_n|^2/s)_lo, s ]
// with fp32 accumulation in TMEM (M = 128 lanes = the 128 queries, N = 128 columns, K = 16 = one MMA). The WHOLE local cost
// comes out of the tensor core: |b|^2 as a hi + lo pair, |a|^2 in the one spare K slot ROUNDED DOWN to fp16, so the scan's
// cost is <= the cost of the fp16-rounded frames (by at most 2^-10 |a|^2) and the scan distance stays a LOWER bound of
// their DTW - which is all the certification in k_dtw_finalize needs (a slightly blunter filter, the same proof). TMEM lane
// m is read back by the threads that own query m (tcgen05.ld 32x32b), which run the DP recurrence for one slot each with
// the row state in registers: FMNMX3 + FADD per cell instead of the fp32 scan's 7 FFMA2 + 2 FADD + FMNMX3.
// Both sides are centred on the dictionary's mean frame before the fp16 conversion (the cost is translation invariant).
//
// Warp roles (640 threads, 1 CTA / SM): warps 0-15 = DP (warp w owns TMEM lane quadrant w % 4 and slot w / 4); warp 16 =
// TMEM allocator, and its lane 0 issues the TMA bulk copies (A block once, B tiles through a 4-stage ring) and the MMAs;
// warps 17-19 are idle and only make the producer's warpgroup a donor of registers (setmaxnreg: DP 112, producer 32).
// A pipeline step is TWO query rows (two MMAs, one commit) into one of two 256-column TMEM buffers, so the DP warps pay
// one mbarrier round trip per two rows and advance a two-row band in place (cell (i,j) reads d[j] = row i-1 and feeds
// cell (i+1,j), which overwrites d[j]): two independent dependency chains per thread and no register copies.
// A slot holds one segment of 17..32 frames, or two of <= 16 frames (the second at column 16) whose bands the thread
// advances together - the step's fixed cost is then paid once for both; the two tile kinds are separate instantiations.
// Queries are grouped 128 at a time in length order; a group's queries may differ in length by a row or two (shorter ones
// are zero-padded and every lane captures its result at its own last row).
#include <cuda_fp16.h>

#include <algorithm>
#include <atomic>

#include "match.cuh"
#include "tc_common.cuh"

namespace ss {

int dtw_rescore_finalize(ss_dict* d, ss_queries* q, int k, int kp, uint32_t nslots, const uint32_t* d_slot_qid, double eps,
                         const float* d_max_na, const float* d_max_nb, const float* d_slot_max_na, int bound_mode, uint8_t* d_uncert_flag,
                         uint32_t* d_out_idx, double* d_out_dist);

// ---------------------------------------------------------------------------------------------------------------
// layout builders
// ---------------------------------------------------------------------------------------------------------------
// per-coefficient mean of the dictionary frames -> mu, in two deterministic stages (fixed summation order)
__global__ void k_tc_mean_partial(const double* __restrict__ mfcc, size_t frames, int c, double* __restrict__ partial) {
    __shared__ double s[256];
    const int col = threadIdx.x % 16, rl = threadIdx.x / 16;
    double acc = 0.0;
    if (col < c)
        for (size_t r = (size_t)blockIdx.x * 16 + rl; r < frames; r += (size_t)gridDim.x * 16) acc += mfcc[r * c + col];
    s[threadIdx.x] = acc;
    __syncthreads();
    if (rl == 0) {
        for (int j = 1; j < 16; j++) acc += s[j * 16 + col];
        partial[(size_t)blockIdx.x * 16 + col] = acc;
    }
}
__global__ void k_tc_mean_final(const double* __restrict__ partial, int nblocks, size_t frames, int c, double* __restrict__ mu) {
    const int col = threadIdx.x;
    if (col >= c) return;
    double acc = 0.0;
    for (int b = 0; b < nblocks; b++) acc += partial[(size_t)b * 16 + col];
    mu[col] = frames ? acc / (double)frames : 0.0;
}
// max over frames of |fp16(b - mu)|^2 (to pick the power-of-two scale of the norm columns) and max |fp16(b - mu)|
__global__ void k_tc_dict_maxnorm(const double* __restrict__ mfcc, size_t frames, int c, const double* __restrict__ mu,
                                  float* __restrict__ out /* [0] max norm, [1] max abs */) {
    const size_t f = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    float nrm = 0.f, mx = 0.f;
    if (f < frames) {
        for (int k = 0; k < c; k++) {
            const float v = __half2float(__float2half_rn((float)(mfcc[f * c + k] - mu[k])));
            nrm += v * v;
            mx = fmaxf(mx, fabsf(v));
        }
    }
    for (int o = 16; o; o >>= 1) {
        nrm = fmaxf(nrm, __shfl_xor_sync(0xffffffffu, nrm, o));
        mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    }
    if ((threadIdx.x & 31) == 0) {
        if (nrm == nrm) atomicMax(reinterpret_cast<unsigned*>(out), __float_as_uint(nrm));
        if (mx == mx) atomicMax(reinterpret_cast<unsigned*>(out + 1), __float_as_uint(mx));
    }
}
// one thread per (tile, column n): writes row n of the tile's B operand
__global__ void k_tc_dict_tiles(const double* __restrict__ mfcc, const uint64_t* __restrict__ off, int c, const double* __restrict__ mu,
                                const int4* __restrict__ desc, uint32_t ntiles, float scale, unsigned char* __restrict__ tiles) {
    const uint32_t t = blockIdx.x, n = threadIdx.x;  // blockDim = kTcN
    if (t >= ntiles) return;
    const int W = 32;  // slot width
    const int slot = (int)n / W;
    int j = (int)n % W;
    const int4 sl = desc[(size_t)t * 4 + slot];  // {segment A, length A, segment B, length B}; B >= 0: a pair of short segments
    int seg = sl.x, len = sl.y;
    if (sl.z >= 0 && j >= kTcPairCol) seg = sl.z, len = sl.w, j -= kTcPairCol;  // B's columns start at column 16 of the slot
    __half row[kTcK];
#pragma unroll
    for (int k = 0; k < kTcK; k++) row[k] = __float2half_rn(0.f);
    if (seg >= 0 && j < len) {
        const double* src = mfcc + (off[seg] + j) * c;
        float nrm = 0.f;
        for (int k = 0; k < c; k++) {
            const __half h = __float2half_rn((float)(src[k] - mu[k]));
            row[k] = h;
            const float v = __half2float(h);
            nrm += v * v;
        }
        const float sn = nrm * (1.0f / scale);  // s is a power of two: exact
        const __half hi = __float2half_rn(sn);
        row[13] = hi;
        row[14] = __float2half_rn(sn - __half2float(hi));
        row[15] = __float2half_rn(scale);  // multiplies the query side's rd(|a|^2 / s)
    }
    unsigned char* base = tiles + (size_t)t * kTcBTileBytes;
#pragma unroll
    for (int k = 0; k < kTcK; k++) *reinterpret_cast<__half*>(base + tc_tile_offset<kTcN>((int)n, k)) = row[k];
}
// ---------------------------------------------------------------------------------------------------------------
// the scan
// ---------------------------------------------------------------------------------------------------------------
struct TcParams {
    const unsigned char* a_blocks;
    const uint64_t* group_off;
    const uint32_t* group_len;   // longest | shortest << 16 query length of each group of 128
    const uint32_t* slot_len;    // per query slot: its own length (0 = padding lane)
    uint32_t ngroups;
    const unsigned char* tiles;
    const int4* desc;
    const uint32_t* slice_tile;  // all slices + 1
    uint32_t nslices;            // slices of THIS launch, starting at slice_begin
    uint32_t slice_begin;
    unsigned long long* partial;  // [nslices][ngroups * 128][KP]
    uint32_t max_len;
    float* dbg;                   // DBG instantiation only: [ngroups * 128][dbg_nseg] raw scan distances (ss_dict_debug_tc_scan)
    uint32_t dbg_nseg;
};

// TMEM -> registers: W (8 / 16 / 32) consecutive columns of this thread's lane
template <int W>
__device__ __forceinline__ void tc_ld(uint32_t taddr, float* v);
template <>
__device__ __forceinline__ void tc_ld<8>(uint32_t taddr, float* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = __uint_as_float(r[i]);
}
template <>
__device__ __forceinline__ void tc_ld<16>(uint32_t taddr, float* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
}
template <>
__device__ __forceinline__ void tc_ld<32>(uint32_t taddr, float* v) { tc_ld32(taddr, v); }
// the 4*NG columns of one row, with the narrowest loads that cover them
template <int NG>
__device__ __forceinline__ void tc_ld_row(uint32_t taddr, float (&v)[4 * NG]) {
    if constexpr (NG == 2 || NG == 4 || NG == 8) {
        tc_ld<4 * NG>(taddr, v);
    } else if constexpr (NG == 6) {
        tc_ld<16>(taddr, v);
        tc_ld<8>(taddr + 16, v + 16);
    } else {  // 1, 3, 5, 7: load the next even group count into a scratch of that width
        float t[4 * (NG + 1)];
        tc_ld_row<NG + 1>(taddr, t);
#pragma unroll
        for (int j = 0; j < 4 * NG; j++) v[j] = t[j];
    }
}

// TWO rows (i, i+1) of one segment slot in column-major order, row state updated in place: cell (i, j) reads d[j]
// (row i-1) and feeds cell (i+1, j), which overwrites d[j]. Two independent dependency chains per thread (ILP 2), no
// register copies, no guards: per cell FMNMX3 + FADD. The column count 4*NG is a compile-time constant. The band also
// hands back row i's values of the last 4-column group (c0l; row i+1's are d[4 NG - 4 ..]): the column len - 1 lies in
// that group, and the caller picks D(i, len-1) / D(i+1, len-1) from them only in the steps where a query can end.
struct TcCarry {  // what a band carries from column j-1 to column j: D(i, j-1), D(i-1, j-1), D(i+1, j-1)
    float left0, diag0, left1;
};
// columns [J0, J1) of the band; tm0 / tm1 hold the costs of those columns only
template <int NG, int J0, int J1, int W>
__device__ __forceinline__ void tc_dp_band_cols(const float (&tm0)[W], const float (&tm1)[W], float (&d)[4 * NG], TcCarry& c, float (&c0l)[4]) {
#pragma unroll
    for (int j = J0; j < J1; j++) {
        const float up0 = d[j];
        const float c0 = tm0[j - J0] + tc_min3(c.left0, up0, c.diag0);
        const float c1 = tm1[j - J0] + tc_min3(c.left1, c0, c.left0);  // up = D(i, j), diag = D(i, j-1)
        c.diag0 = up0;
        c.left0 = c0;
        c.left1 = c1;
        d[j] = c1;
        if (j >= 4 * (NG - 1)) c0l[j - 4 * (NG - 1)] = c0;
    }
}
// a single trailing row (odd group length), in place
template <int NG>
__device__ __forceinline__ void tc_dp_row_ng(const float (&tm)[4 * NG], float (&d)[4 * NG], float dinit) {
    const float INF = __int_as_float(0x7f800000);
    float left = INF, diag = dinit;
#pragma unroll
    for (int j = 0; j < 4 * NG; j++) {
        const float up = d[j];
        const float cur = tm[j] + tc_min3(left, up, diag);
        diag = up;
        left = cur;
        d[j] = cur;
    }
}
__device__ __forceinline__ float tc_pick4(const float* v, int r) { return r == 0 ? v[0] : (r == 1 ? v[1] : (r == 2 ? v[2] : v[3])); }

// one pipeline step for one thread: wait for the step's MMAs, pull this slot's columns of both rows into registers, hand
// the TMEM buffer back, advance the band
template <int NG>
__device__ __forceinline__ void tc_step2(TcCursor& cur, float (&d)[4 * NG], float dinit, float (&c0l)[4]) {
    const float INF = __int_as_float(0x7f800000);
    cur.wait();
    TcCarry c = {INF, dinit, INF};  // dinit = 0 on the first row of the pair (the virtual D(-1,-1)), +inf after
    if constexpr (kTcChunked && NG > 4) {
        // 112-register budget: the step's costs come in two column chunks (16 + the rest), each two rows; the compiler
        // starts the second chunk's loads while the first is being consumed
        const uint32_t taddr = cur.taddr;
        {
            float a0[16], a1[16];
            tc_ld<16>(taddr, a0);
            tc_ld<16>(taddr + kTcN, a1);
            tc_wait_ld();
            tc_dp_band_cols<NG, 0, 16, 16>(a0, a1, d, c, c0l);
        }
        constexpr int W2 = NG <= 6 ? 8 : 16;  // the remaining 4 NG - 16 columns, loaded as x8 or x16
        float b0[W2], b1[W2];
        tc_ld<W2>(taddr + 16, b0);
        tc_ld<W2>(taddr + kTcN + 16, b1);
        tc_wait_ld();
        cur.release();
        tc_dp_band_cols<NG, 16, 4 * NG, W2>(b0, b1, d, c, c0l);
    } else {
        float tm0[4 * NG], tm1[4 * NG];
        tc_ld_row<NG>(cur.taddr, tm0);
        tc_ld_row<NG>(cur.taddr + kTcN, tm1);
        tc_wait_ld();
        cur.release();
        tc_dp_band_cols<NG, 0, 4 * NG, 4 * NG>(tm0, tm1, d, c, c0l);
    }
}

// one dictionary tile for one thread (= one query x one segment slot), column-group count NG fixed at compile time so
// that the whole step loop is straight-line code over exactly 4*NG row-state registers. Returns D(Lm-1, len-1).
// L = longest, lmin = shortest query of the CTA's group, Lm = this lane's own.
template <int NG>
__device__ __forceinline__ float tc_tile(uint32_t L, uint32_t lmin, uint32_t Lm, int len, TcCursor& cur) {
    const float INF = __int_as_float(0x7f800000);
    float d[4 * NG];
#pragma unroll
    for (int j = 0; j < 4 * NG; j++) d[j] = INF;
    float res = INF, dinit = 0.f;
    const uint32_t nfull = L >> 1;           // steps that carry two rows
    const uint32_t ncap = min((lmin - 1) >> 1, nfull);   // steps before any query of the group can end
    const int r = (len - 1) & 3;             // where column len - 1 sits in the last 4-column group
    uint32_t st = 0;
    // no query of the group ends in steps [0, ncap). They run two per iteration on buffer 0 then buffer 1, from cursors
    // rebuilt out of loop invariants - barrier and TMEM addresses are then constants of the loop and only the parity flips
    // (once per pair) - after one plain step if the tile happens to start on buffer 1.
    if (st < ncap && cur.buf) {
        float c0l[4];
        tc_step2<NG>(cur, d, dinit, c0l);
        dinit = INF;
        st++;
    }
    if (st + 2 <= ncap) {
        const uint32_t full0 = cur.full, taddr0 = cur.taddr;
        uint32_t par = cur.par;
#pragma unroll 1
        for (; st + 2 <= ncap; st += 2) {
            float c0l[4];
            TcCursor c0 = {0u, par, full0, taddr0, cur.full_sum, cur.taddr_sum};
            tc_step2<NG>(c0, d, dinit, c0l);
            TcCursor c1 = {1u, par, full0 + 8u, taddr0 + (uint32_t)kTcBufCols, cur.full_sum, cur.taddr_sum};
            tc_step2<NG>(c1, d, INF, c0l);
            dinit = INF;
            par ^= 1u;
        }
        cur.par = par;
    }
    if (st < ncap) {
        float c0l[4];
        tc_step2<NG>(cur, d, dinit, c0l);
        dinit = INF;
        st++;
    }
#pragma unroll 1
    for (; st < nfull; st++) {  // only the last step or two of a tile
        float c0l[4];
        tc_step2<NG>(cur, d, dinit, c0l);
        dinit = INF;
        const float e0 = tc_pick4(c0l, r), e1 = tc_pick4(&d[4 * (NG - 1)], r);
        res = (2 * st + 1 == Lm) ? e0 : ((2 * st + 2 == Lm) ? e1 : res);  // this lane's query ends in this band?
    }
    if (L & 1) {  // odd group length: the last step carries one row
        cur.wait();
        float tm0[4 * NG];
        tc_ld_row<NG>(cur.taddr, tm0);
        tc_wait_ld();
        cur.release();
        tc_dp_row_ng<NG>(tm0, d, dinit);
        res = (L == Lm) ? tc_pick4(&d[4 * (NG - 1)], r) : res;
    }
    return res;
}

// ---- two short segments (<= 16 frames each) in one slot: columns [0, 4 NG) and [16, 16 + 4 NG) ---------------------------
// A step for short segments is mostly hand-off overhead (about 30 of its 42..102 instructions); sharing it between two
// segments halves that. The two bands are independent: each has its own row state, carry and capture. Both run with the
// larger of the two column-group counts, so a band's column len - 1 can sit in any group: the capture steps select it by
// index (CAP), column by column.
template <int N>
__device__ __forceinline__ float tc_pick_n(const float (&v)[N], int idx) {
    float r = v[0];
#pragma unroll
    for (int j = 1; j < N; j++) r = idx == j ? v[j] : r;
    return r;
}
template <int NG, bool CAP>
__device__ __forceinline__ void tc_dp_band_pair(const float (&tm0)[4 * NG], const float (&tm1)[4 * NG], float (&d)[4 * NG], float dinit, int len,
                                                float& e0) {
    const float INF = __int_as_float(0x7f800000);
    float left0 = INF, diag0 = dinit, left1 = INF;
#pragma unroll
    for (int j = 0; j < 4 * NG; j++) {
        const float up0 = d[j];
        const float c0 = tm0[j] + tc_min3(left0, up0, diag0);
        const float c1 = tm1[j] + tc_min3(left1, c0, left0);
        diag0 = up0;
        left0 = c0;
        left1 = c1;
        d[j] = c1;
        if (CAP) e0 = j == len - 1 ? c0 : e0;  // D(i, len-1); the second row's value stays in d[len-1]
    }
}
template <int NG, bool CAP>
__device__ __forceinline__ void tc_step2_pair(TcCursor& cur, float (&dA)[4 * NG], float (&dB)[4 * NG], float dinit, int lenA, int lenB, float& e0A,
                                              float& e0B) {
    cur.wait();
    const uint32_t taddr = cur.taddr;
    {
        float a0[4 * NG], a1[4 * NG];
        tc_ld_row<NG>(taddr, a0);
        tc_ld_row<NG>(taddr + kTcN, a1);
        tc_wait_ld();
        tc_dp_band_pair<NG, CAP>(a0, a1, dA, dinit, lenA, e0A);
    }
    float b0[4 * NG], b1[4 * NG];
    tc_ld_row<NG>(taddr + kTcPairCol, b0);
    tc_ld_row<NG>(taddr + kTcN + kTcPairCol, b1);
    tc_wait_ld();
    cur.release();
    tc_dp_band_pair<NG, CAP>(b0, b1, dB, dinit, lenB, e0B);
}
// returns D(Lm-1, lenA-1) and D(Lm-1, lenB-1); lenB = 0 when the slot's second place is empty
template <int NG>
__device__ __forceinline__ void tc_tile_pair(uint32_t L, uint32_t lmin, uint32_t Lm, int lenA, int lenB, TcCursor& cur, float& resA, float& resB) {
    const float INF = __int_as_float(0x7f800000);
    float dA[4 * NG], dB[4 * NG];
#pragma unroll
    for (int j = 0; j < 4 * NG; j++) dA[j] = INF, dB[j] = INF;
    resA = INF, resB = INF;
    float dinit = 0.f;
    const uint32_t nfull = L >> 1;
    const uint32_t ncap = min((lmin - 1) >> 1, nfull);
    uint32_t st = 0;
    // steps [0, ncap): no query of the group ends; two per iteration on buffers 0, 1 with loop-invariant addresses (tc_tile)
    if (st < ncap && cur.buf) {
        float e0A, e0B;
        tc_step2_pair<NG, false>(cur, dA, dB, dinit, lenA, lenB, e0A, e0B);
        dinit = INF;
        st++;
    }
    if (st + 2 <= ncap) {
        const uint32_t full0 = cur.full, taddr0 = cur.taddr;
        uint32_t par = cur.par;
#pragma unroll 1
        for (; st + 2 <= ncap; st += 2) {
            float e0A, e0B;
            TcCursor c0 = {0u, par, full0, taddr0, cur.full_sum, cur.taddr_sum};
            tc_step2_pair<NG, false>(c0, dA, dB, dinit, lenA, lenB, e0A, e0B);
            TcCursor c1 = {1u, par, full0 + 8u, taddr0 + (uint32_t)kTcBufCols, cur.full_sum, cur.taddr_sum};
            tc_step2_pair<NG, false>(c1, dA, dB, INF, lenA, lenB, e0A, e0B);
            dinit = INF;
            par ^= 1u;
        }
        cur.par = par;
    }
    if (st < ncap) {
        float e0A, e0B;
        tc_step2_pair<NG, false>(cur, dA, dB, dinit, lenA, lenB, e0A, e0B);
        dinit = INF;
        st++;
    }
#pragma unroll 1
    for (; st < nfull; st++) {  // only the last step or two of a tile
        float e0A = INF, e0B = INF;
        tc_step2_pair<NG, true>(cur, dA, dB, dinit, lenA, lenB, e0A, e0B);
        dinit = INF;
        const bool end0 = 2 * st + 1 == Lm, end1 = 2 * st + 2 == Lm;  // this lane's query ends in this band?
        resA = end0 ? e0A : (end1 ? tc_pick_n<4 * NG>(dA, lenA - 1) : resA);
        resB = end0 ? e0B : (end1 ? tc_pick_n<4 * NG>(dB, lenB - 1) : resB);
    }
    if (L & 1) {  // odd group length: the last step carries one row
        cur.wait();
        float a0[4 * NG], b0[4 * NG];
        tc_ld_row<NG>(cur.taddr, a0);
        tc_ld_row<NG>(cur.taddr + kTcPairCol, b0);
        tc_wait_ld();
        cur.release();
        tc_dp_row_ng<NG>(a0, dA, dinit);
        tc_dp_row_ng<NG>(b0, dB, dinit);
        resA = (L == Lm) ? tc_pick_n<4 * NG>(dA, lenA - 1) : resA;
        resB = (L == Lm) ? tc_pick_n<4 * NG>(dB, lenB - 1) : resB;
    }
}

// PAIRED selects the tile kind the launch covers (the dictionary's tiles are sorted: single-segment slots first, paired
// slots after; each kind gets its own instantiation so that neither pays for the other's registers and code).
// DBG additionally writes every pair's scan distance to p.dbg (the measurement hook behind ss_dict_debug_tc_scan; the
// product launches never instantiate it).
template <int KP, bool PAIRED, bool DBG = false>
__global__ void __launch_bounds__(kTcThreads, 1) k_dtw_scan_tc(const TcParams p) {
    extern __shared__ unsigned char smem_raw[];
    // [A tiles: max_len x 4 KB][B ring: 4 x 4 KB][barriers][candidate lists], 128-byte aligned
    unsigned char* smem = smem_raw + ((128u - (s32(smem_raw) & 127u)) & 127u);
    unsigned char* sA = smem;
    unsigned char* sB = smem + (size_t)p.max_len * kTcATileBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sB + kTcStages * kTcBTileBytes);
    uint64_t* a_full = bars;
    uint64_t* b_full = bars + 1;
    uint64_t* b_empty = b_full + kTcStages;
    uint64_t* t_full = bars + 10;
    uint64_t* t_empty = bars + 12;  // = t_full + 16 bytes (TcCursor::release)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 14);
    unsigned long long* topk = reinterpret_cast<unsigned long long*>(bars + 32);  // [KP][512]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x / p.nslices, slice = p.slice_begin + blockIdx.x % p.nslices;
    // the other tile kind's launch may start filling SMs as this one's CTAs retire (programmatic dependent launch; the two
    // write disjoint candidate lists and neither reads the other's output)
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    const uint32_t glen = p.group_len[g];
    const uint32_t L = glen & 0xFFFFu, lmin = glen >> 16;  // longest (= rows of the A block) and shortest query of the group
    const uint32_t t0 = p.slice_tile[slice], t1 = p.slice_tile[slice + 1];
    const uint32_t ntiles = t1 - t0;

    if (threadIdx.x == 0) {
        mb_init(a_full, 1);
        for (int s = 0; s < kTcStages; s++) mb_init(&b_full[s], 1), mb_init(&b_empty[s], 1);
        for (int s = 0; s < 2; s++) mb_init(&t_full[s], 1), mb_init(&t_empty[s], kTcDpWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == kTcDpWarps) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(tmem_slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // register re-distribution between warpgroups (setmaxnreg): the producer's warpgroup (one working lane, three idle
    // warps) hands registers to the three DP warpgroups, whose band loop keeps 32 + 64 values live per thread
    if (warp >= kTcDpWarps) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kTcRegsProd));
    if (warp > kTcDpWarps) {
        // idle warps of the producer's warpgroup
    } else if (warp == kTcDpWarps) {
        if (lane == 0 && ntiles) {
            // ---- producer: TMA + MMA issue (32-bit shared addresses and running counters: it lives in kTcRegsProd registers)
            const uint32_t bars_s = s32(bars), sA_s = s32(sA), sB_s = s32(sB);
            const uint32_t a_full_s = bars_s, b_full_s = bars_s + 8, b_empty_s = bars_s + 8 + 8 * kTcStages, t_full_s = bars_s + 80,
                           t_empty_s = bars_s + 96;
            mbs_expect_tx(a_full_s, L * kTcATileBytes);
            tmas_g2s(sA_s, p.a_blocks + p.group_off[g], L * kTcATileBytes, a_full_s);
            const unsigned char* tile_src = p.tiles + (size_t)t0 * kTcBTileBytes;
            for (uint32_t n = 0; n < ntiles && n < (uint32_t)kTcStages; n++) {
                mbs_expect_tx(b_full_s + 8 * n, kTcBTileBytes);
                tmas_g2s(sB_s + n * kTcBTileBytes, tile_src + (size_t)n * kTcBTileBytes, kTcBTileBytes, b_full_s + 8 * n);
            }
            tile_src += (size_t)kTcStages * kTcBTileBytes;  // the next tile to fetch
            mbs_wait_sleep(a_full_s, 0);
            const uint32_t idesc = (1u << 4) | ((uint32_t)(kTcN >> 3) << 17) | ((uint32_t)(kTcM >> 4) << 24);  // f16 x f16 -> f32, K-major
            const uint64_t adesc0 = tc_smem_desc_s<kTcM>(sA_s);
            uint32_t cnt = 0, stage = 0, sphase = 0;
            for (uint32_t n = 0; n < ntiles; n++) {
                mbs_wait_sleep(b_full_s + 8 * stage, sphase);
                const uint64_t bdesc = tc_smem_desc_s<kTcN>(sB_s + stage * kTcBTileBytes);
                uint64_t adesc = adesc0;  // advances by one A tile (4 KB = 256 descriptor units) per row
                for (uint32_t row = 0; row < L; row += 2, cnt++) {
                    const uint32_t buf = cnt & 1;
                    if (cnt >= 2) mbs_wait_sleep(t_empty_s + 8 * buf, ((cnt >> 1) - 1) & 1);
                    tc_fence_after();
                    const uint32_t tm = tmem_base + buf * kTcBufCols;
                    tc_mma_f16(tm, adesc, bdesc, idesc);
                    if (row + 1 < L) tc_mma_f16(tm + kTcN, adesc + (kTcATileBytes >> 4), bdesc, idesc);
                    tcs_commit(t_full_s + 8 * buf);
                    adesc += 2 * (kTcATileBytes >> 4);
                }
                tcs_commit(b_empty_s + 8 * stage);
                if (n + kTcStages < ntiles) {  // refill this stage once its MMAs have completed
                    mbs_wait_sleep(b_empty_s + 8 * stage, sphase);
                    mbs_expect_tx(b_full_s + 8 * stage, kTcBTileBytes);
                    tmas_g2s(sB_s + stage * kTcBTileBytes, tile_src, kTcBTileBytes, b_full_s + 8 * stage);
                    tile_src += kTcBTileBytes;
                }
                if (++stage == (uint32_t)kTcStages) stage = 0, sphase ^= 1;
            }
        }
    } else {
        // ---- DP warps ---------------------------------------------------------------------------------------------------
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kTcRegsDp));
        const int q = warp & 3, slot = warp >> 2;
        const int m = q * 32 + lane;
        unsigned long long* list = topk + threadIdx.x;  // [KP][512] keys, this thread's column
#pragma unroll
        for (int s = 0; s < KP; s++) list[s * kTcDpThreads] = 0xFFFFFFFFFFFFFFFFull;
        unsigned long long worst = 0xFFFFFFFFFFFFFFFFull;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + slot * 32;
        const uint32_t Lm = p.slot_len[g * kTcM + m];  // this lane's own query length
        TcCursor cur;
        cur.init(s32(t_full), lane_addr);
        for (uint32_t n = 0; n < ntiles; n++) {
            const int4 sl = __ldg(p.desc + (size_t)(t0 + n) * 4 + slot);  // {segment A, length A, segment B, length B} of this slot
            if constexpr (PAIRED) {  // two short segments per slot (an empty place has length 0)
                const int ngp = (max(sl.y, sl.w) + 3) >> 2;
                float resA, resB;
                switch (ngp) {
                    case 0:
                    case 1: tc_tile_pair<1>(L, lmin, Lm, sl.y, sl.w, cur, resA, resB); break;
                    case 2: tc_tile_pair<2>(L, lmin, Lm, sl.y, sl.w, cur, resA, resB); break;
                    case 3: tc_tile_pair<3>(L, lmin, Lm, sl.y, sl.w, cur, resA, resB); break;
                    default: tc_tile_pair<4>(L, lmin, Lm, sl.y, sl.w, cur, resA, resB); break;
                }
                if (Lm) {
                    if (sl.y > 0) tc_insert<KP>(list, worst, __fdividef(resA, (float)(Lm + (uint32_t)sl.y)), (uint32_t)sl.x);
                    if (sl.w > 0) tc_insert<KP>(list, worst, __fdividef(resB, (float)(Lm + (uint32_t)sl.w)), (uint32_t)sl.z);
                    if constexpr (DBG) {
                        float* row = p.dbg + (size_t)(g * kTcM + m) * p.dbg_nseg;
                        if (sl.y > 0) row[sl.x] = __fdividef(resA, (float)(Lm + (uint32_t)sl.y));
                        if (sl.w > 0) row[sl.z] = __fdividef(resB, (float)(Lm + (uint32_t)sl.w));
                    }
                }
            } else {
                const int seg = sl.x, len = sl.y;
                const int ng = (len + 3) >> 2;  // 4-column groups of the DP row (tile-uniform up to +-1: segments are sorted by length)
                float res;
                switch (ng) {  // one dispatch per tile
                    case 1: res = tc_tile<1>(L, lmin, Lm, len, cur); break;
                    case 2: res = tc_tile<2>(L, lmin, Lm, len, cur); break;
                    case 3: res = tc_tile<3>(L, lmin, Lm, len, cur); break;
                    case 4: res = tc_tile<4>(L, lmin, Lm, len, cur); break;
                    case 5: res = tc_tile<5>(L, lmin, Lm, len, cur); break;
                    case 6: res = tc_tile<6>(L, lmin, Lm, len, cur); break;
                    case 7: res = tc_tile<7>(L, lmin, Lm, len, cur); break;
                    default: res = tc_tile<8>(L, lmin, Lm, len, cur); break;
                }
                // result: D(Lm-1, len-1) / (Lm + len)
                if (seg >= 0 && Lm) tc_insert<KP>(list, worst, __fdividef(res, (float)(Lm + (uint32_t)len)), (uint32_t)seg);
                if constexpr (DBG)
                    if (seg >= 0 && Lm) p.dbg[(size_t)(g * kTcM + m) * p.dbg_nseg + seg] = __fdividef(res, (float)(Lm + (uint32_t)len));
            }
        }
        // the four slots' lists of query m (threads m, m + 128, m + 256, m + 384) are merged by the slot-0 thread: one list per
        // (slice, query) leaves the CTA
        asm volatile("bar.sync 1, %0;" ::"n"(kTcDpThreads) : "memory");
        if (slot == 0) {
            for (int o = 1; o < kTcSlots; o++) {
                const unsigned long long* other = list + o * kTcM;
                for (int s = 0; s < KP; s++) {  // ascending: stop at the first key that does not make the cut
                    const unsigned long long key = other[s * kTcDpThreads];
                    if (key >= worst) break;
                    tc_insert_key<KP>(list, worst, key);
                }
            }
            unsigned long long* out = p.partial + ((size_t)slice * p.ngroups * kTcM + (size_t)g * kTcM + m) * KP;
#pragma unroll
            for (int s = 0; s < KP; s++) out[s] = list[s * kTcDpThreads];
        }
    }
    // a dependent launch may finish its own work before the launch ahead of it has: it must not be seen as complete (the
    // merge kernel is ordered after THIS grid) until that one is, so every CTA waits for it on the way out. By then all of
    // the earlier grid's CTAs are at least resident, so nothing is held up; a no-op for a normal launch.
    if constexpr (PAIRED) asm volatile("griddepcontrol.wait;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (warp == kTcDpWarps) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// Statistics both tensor-core scans centre and scale their fp16 operands with (any segment length): the dictionary's mean
// frame, max |fp16(b - mu)|^2 and max |fp16(b - mu)|, the power-of-two norm scale s; tc_serial identifies this build.
static int tc_dict_stats(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    d->tc_stats_ready = false;
    if (d->total_frames == 0) return SS_OK;
    SS_CUDA(ctx, d->d_mu.reserve(16));
    SS_CUDA(ctx, cudaMemsetAsync(d->d_mu.p, 0, 16 * sizeof(double), ctx->stream));
    {
        const int nb = (int)std::min<size_t>(std::max<size_t>(d->total_frames / 256, 1), 512);
        SS_CUDA(ctx, d->d_rescore_rows.reserve((size_t)nb * 16));  // scratch
        k_tc_mean_partial<<<nb, 256, 0, ctx->stream>>>(d->d_mfcc.p, d->total_frames, d->c, d->d_rescore_rows.p);
        SS_LAUNCHED(ctx);
        k_tc_mean_final<<<1, 32, 0, ctx->stream>>>(d->d_rescore_rows.p, nb, d->total_frames, d->c, d->d_mu.p);
        SS_LAUNCHED(ctx);
    }
    DevBuf<float>& d_mx = d->d_tc_max_norm;
    SS_CUDA(ctx, d_mx.reserve(2));
    SS_CUDA(ctx, cudaMemsetAsync(d_mx.p, 0, 2 * sizeof(float), ctx->stream));
    k_tc_dict_maxnorm<<<ceil_div((long long)d->total_frames, 256), 256, 0, ctx->stream>>>(d->d_mfcc.p, d->total_frames, d->c, d->d_mu.p, d_mx.p);
    SS_LAUNCHED(ctx);
    float mx[2] = {0, 0};
    SS_CUDA(ctx, cudaMemcpyAsync(mx, d_mx.p, sizeof(mx), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (!(mx[1] < 3.0e4f) || !(mx[0] < 1.0e9f)) return SS_OK;  // values outside a safe fp16 range: keep the fp32 scan
    float scale = 1.f;
    while (mx[0] / scale > 16384.f) scale *= 2.f;  // |b|^2 / s must fit fp16 comfortably; s <= 2^16 is exact in fp16
    if (scale > 32768.f) return SS_OK;
    d->tc_nb_scale = scale;
    d->tc_max_nb = mx[0];
    d->tc_max_abs = mx[1];
    static std::atomic<uint64_t> serial{0};  // process-wide: dictionaries of different contexts / host threads never share one
    d->tc_serial = ++serial;
    d->tc_stats_ready = true;
    return SS_OK;
}

int dtw_tc_dict_build(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    d->tc_ready = false;
    SS_TRY(tc_dict_stats(d));
    if (!d->tc_stats_ready || d->max_len > (uint32_t)kTcMaxLen) return SS_OK;  // longer segments: dtw_h2.cu's strips, or dtw.cu's fp32 scan
    // segments sorted by length (longest first) so that the 4 slots of a tile, and hence both column halves, carry equal work
    std::vector<uint32_t> order;
    order.reserve(d->nseg);
    for (size_t s = 0; s < d->nseg; s++)
        if (d->h_off[s + 1] > d->h_off[s]) order.push_back((uint32_t)s);
    auto len_of = [&](uint32_t s) { return (int)(d->h_off[s + 1] - d->h_off[s]); };
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return len_of(a) > len_of(b); });
    // A tile has 4 slots of 32 columns. A segment longer than 16 frames takes a slot of its own; shorter ones share a slot
    // two by two (the second at column 16), so that the per-step hand-off is paid once for both. Per slot the descriptor is
    // {segment A, length A, segment B, length B}, B = -1 when absent.
    std::vector<int4> desc;
    d->tc_first_pair_tile = 0xFFFFFFFFu;
    d->h_tc_tile_frames.clear();  // per tile: an instruction-count estimate of one pipeline step (slice balancing)
    for (size_t o = 0; o < order.size();) {
        const bool pair = len_of(order[o]) <= kTcPairCol;
        const size_t take = std::min<size_t>(order.size() - o, pair ? 2 * kTcSlots : kTcSlots);
        uint32_t cost = 0;
        for (int sidx = 0; sidx < 4; sidx++) {
            int4 e = make_int4(-1, 0, -1, 0);
            if ((size_t)sidx < take) e.x = (int)order[o + sidx], e.y = len_of(order[o + sidx]);
            if (pair && (size_t)(kTcSlots + sidx) < take) e.z = (int)order[o + kTcSlots + sidx], e.w = len_of(order[o + kTcSlots + sidx]);
            desc.push_back(e);
            cost = std::max<uint32_t>(cost, 32u + 16u * (uint32_t)(pair ? 2 * ((std::max(e.y, e.w) + 3) >> 2) : ((e.y + 3) >> 2)));
        }
        if (pair && d->tc_first_pair_tile == 0xFFFFFFFFu) d->tc_first_pair_tile = (uint32_t)d->h_tc_tile_frames.size();
        d->h_tc_tile_frames.push_back(cost);
        o += take;
    }
    if (d->tc_first_pair_tile == 0xFFFFFFFFu) d->tc_first_pair_tile = (uint32_t)d->h_tc_tile_frames.size();
    const uint32_t ntiles = (uint32_t)(desc.size() / 4);
    d->tc_ntiles = ntiles;
    SS_TRY(upload(ctx, d->d_tc_desc, desc.data(), desc.size()));
    SS_CUDA(ctx, d->d_tc_tiles.reserve((size_t)ntiles * kTcBTileBytes / 2));
    k_tc_dict_tiles<<<ntiles, kTcN, 0, ctx->stream>>>(d->d_mfcc.p, d->d_off.p, d->c, d->d_mu.p, d->d_tc_desc.p, ntiles, d->tc_nb_scale,
                                                     reinterpret_cast<unsigned char*>(d->d_tc_tiles.p));
    SS_LAUNCHED(ctx);
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    d->tc_ready = true;
    return SS_OK;
}

// Length-sorted groups of 128 queries (a counting sort on the host: lengths <= 32 for the scans of <= 32 x <= 32 frames, up
// to kTcGroupMaxLen for dtw_h2.cu's strip kernel). Depends on the lengths only, so it
// runs once per batch, when the batch is filled (ss_queries_create / the fill inside ss_dict_match, where it overlaps the
// host-to-device copy of the frames), not inside the match.
int dtw_tc_queries_group(ss_queries* q) {
    ss_ctx* ctx = q->ctx;
    q->tc_grouped = false;
    q->tc_built = false;
    q->tc_ngroups = 0;
    if (q->max_len > (uint32_t)kTcGroupMaxLen || q->total_frames == 0) return SS_OK;
    auto len_of = [&](uint32_t i) { return (uint32_t)(q->h_off[i + 1] - q->h_off[i]); };
    std::vector<uint32_t> order;
    {
        const uint32_t ml = q->max_len;
        std::vector<uint32_t> start(ml + 1, 0);  // bucket ml - len: the longest first; empty queries are left out
        size_t nonempty = 0;
        for (size_t i = 0; i < q->nq; i++) {
            const uint32_t l = len_of((uint32_t)i);
            if (l) start[ml - l]++, nonempty++;
        }
        uint32_t acc = 0;
        for (uint32_t b = 0; b <= ml; b++) {
            const uint32_t c = start[b];
            start[b] = acc;
            acc += c;
        }
        order.resize(nonempty);
        for (size_t i = 0; i < q->nq; i++) {
            const uint32_t l = len_of((uint32_t)i);
            if (l) order[start[ml - l]++] = (uint32_t)i;
        }
    }
    // consecutive chunks of 128 queries in length order: a group's queries differ in length by a row or two at most
    // (the scan pads the shorter ones with zero rows and captures every lane's result at its own last row)
    std::vector<uint32_t> glen, gqid, slen;
    std::vector<uint64_t> goff;
    uint64_t bytes = 0;
    for (size_t pos = 0; pos < order.size(); pos += kTcM) {
        const size_t end = std::min(order.size(), pos + (size_t)kTcM);
        const uint32_t lmax = len_of(order[pos]), lmin = len_of(order[end - 1]);
        glen.push_back(lmax | (lmin << 16));
        goff.push_back(bytes);
        for (size_t l = 0; l < (size_t)kTcM; l++) {
            gqid.push_back(pos + l < end ? order[pos + l] : 0xFFFFFFFFu);
            slen.push_back(pos + l < end ? len_of(order[pos + l]) : 0u);
        }
        bytes += (uint64_t)lmax * kTcATileBytes;
    }
    // (host-to-device copies from pageable memory are staged before cudaMemcpyAsync returns: the vectors may go out of scope)
    SS_TRY(upload(ctx, q->d_tc_slot_len, slen.data(), slen.size()));
    q->tc_ngroups = (uint32_t)glen.size();
    q->h_tc_group_len = glen;
    q->tc_a_bytes = bytes;
    SS_TRY(upload(ctx, q->d_tc_group_len, glen.data(), glen.size()));
    SS_TRY(upload(ctx, q->d_tc_group_off, goff.data(), goff.size()));
    SS_TRY(upload(ctx, q->d_tc_qid, gqid.data(), gqid.size()));
    q->tc_grouped = true;
    return SS_OK;
}

// the fp16 A blocks of a grouped batch for dictionary d (its mean frame and norm scale); asynchronous, no host round trip
static int tc_queries_build(ss_dict* d, ss_queries* q) {
    ss_ctx* ctx = q->ctx;
    if (q->tc_built && q->tc_dict_serial == d->tc_serial) return SS_OK;  // the A blocks depend on the dictionary's mean frame and scale
    if (!q->tc_grouped) SS_TRY(dtw_tc_queries_group(q));
    SS_CUDA(ctx, q->d_tc_a.reserve(std::max<uint64_t>(q->tc_a_bytes, 16)));
    SS_CUDA(ctx, q->d_tc_slot_max_na.reserve(std::max<size_t>((size_t)q->tc_ngroups * kTcM, 1)));
    SS_CUDA(ctx, q->d_uncert_flag.reserve(std::max<size_t>(q->nq, 1)));
    SS_CUDA(ctx, q->d_tc_max_norm.reserve(1));
    SS_CUDA(ctx, cudaMemsetAsync(q->d_tc_max_norm.p, 0, sizeof(float), ctx->stream));
    if (q->tc_ngroups) {
        SS_CUDA(ctx, cudaMemsetAsync(q->d_tc_slot_max_na.p, 0, (size_t)q->tc_ngroups * kTcM * sizeof(float), ctx->stream));
        k_tc_query_tiles<<<dim3(q->tc_ngroups, q->max_len), kTcM, 0, ctx->stream>>>(q->d_mfcc.p, q->d_off.p, q->c, d->d_mu.p, q->d_tc_group_len.p,
                                                                 q->d_tc_group_off.p, q->d_tc_qid.p, d->tc_nb_scale, 1.0f, q->d_tc_a.p,
                                                                 q->d_tc_max_norm.p, q->d_tc_slot_max_na.p);
        SS_LAUNCHED(ctx);
    }
    q->tc_built = true;
    q->tc_dict_serial = d->tc_serial;
    return SS_OK;
}

template <int KP, bool PAIRED, bool DBG = false>
static int tc_launch_kind(ss_ctx* ctx, TcParams p, uint32_t slice_begin, uint32_t nslices, size_t smem, bool dependent) {
    if (!nslices) return SS_OK;
    p.slice_begin = slice_begin;
    p.nslices = nslices;
    SS_CUDA(ctx, cudaFuncSetAttribute(k_dtw_scan_tc<KP, PAIRED, DBG>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.ngroups * nslices);
    cfg.blockDim = dim3(kTcThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;  // may start while the previous scan launch is still draining
    cfg.attrs = attr;
    cfg.numAttrs = dependent ? 1 : 0;
    SS_CUDA(ctx, cudaLaunchKernelEx(&cfg, k_dtw_scan_tc<KP, PAIRED, DBG>, p));
    SS_LAUNCHED(ctx);
    return SS_OK;
}
// slices [0, nsingle) hold single-segment tiles, [nsingle, nslices) paired ones
template <int KP>
static int tc_launch(ss_ctx* ctx, const TcParams& p, uint32_t nsingle, uint32_t nslices, size_t smem, uint32_t nlists, uint32_t nslots, ss_dict* d,
                     bool timed) {
    if (timed) SS_CUDA(ctx, cudaEventRecord(d->ev_scan0, ctx->stream));
    SS_TRY((tc_launch_kind<KP, false>(ctx, p, 0, nsingle, smem, false)));
    SS_TRY((tc_launch_kind<KP, true>(ctx, p, nsingle, nslices - nsingle, smem, nsingle != 0)));
    if (timed) {
        SS_CUDA(ctx, cudaEventRecord(d->ev_scan1, ctx->stream));
        d->scan_timed = true;
    }
    k_tc_merge<KP><<<ceil_div(nslots, 8), 256, 0, ctx->stream>>>(d->d_tc_partial.p, nlists, nslots, d->d_cand_idx.p, d->d_cand_adist.p);
    SS_LAUNCHED(ctx);
    return SS_OK;
}

constexpr int kTcWaves = 16;  // CTAs per SM over the two launches of one scan

// slices (contiguous tile ranges of ONE kind - single-segment tiles come first, paired tiles after - balanced by the
// tiles' step-cost estimate; about kTcWaves CTAs per SM over the two launches, 1 resident per SM), workspaces and the
// kernel parameters of one scan of query batch q against dictionary d with candidate lists of kp entries
struct TcPlan {
    TcParams p;
    uint32_t nsingle, nslices, nslots;
    size_t smem;
};
static int tc_plan(ss_dict* d, ss_queries* q, int kp, TcPlan* plan) {
    ss_ctx* ctx = d->ctx;
    const uint32_t nslots = q->tc_ngroups * kTcM;
    if (d->slice_for_groups != q->tc_ngroups) {  // the slice table only depends on the dictionary and the number of query groups
        // about kTcWaves CTAs per SM, but never slices of fewer than ~12 tiles: a small batch (nq = 1: one group) would
        // otherwise pay a CTA's fixed cost (TMEM allocation, the A-block copy, list merge) two thousand times
        const uint32_t want = std::max<uint32_t>(1, std::min<uint32_t>(((uint32_t)ctx->sm_count * kTcWaves + q->tc_ngroups - 1) / q->tc_ngroups,
                                                                       std::max<uint32_t>((uint32_t)ctx->sm_count, d->tc_ntiles / 12)));
        std::vector<uint32_t> st;  // (staged by cudaMemcpyAsync before it returns)
        uint64_t total = 0;
        for (uint32_t f : d->h_tc_tile_frames) total += f;
        const uint64_t per = std::max<uint64_t>(1, (total + want - 1) / want);
        uint32_t nsingle = 0;
        for (int kind = 0; kind < 2; kind++) {
            const uint32_t tb = kind ? d->tc_first_pair_tile : 0, te = kind ? d->tc_ntiles : d->tc_first_pair_tile;
            uint64_t acc = per;  // forces a slice start at the first tile of the kind
            for (uint32_t t = tb; t < te; t++) {
                if (acc >= per) st.push_back(t), acc = 0;
                acc += d->h_tc_tile_frames[t];
            }
            if (!kind) nsingle = (uint32_t)st.size();
        }
        st.push_back(d->tc_ntiles);
        d->tc_nsingle = nsingle;
        d->tc_nslices = (uint32_t)st.size() - 1;
        SS_TRY(upload(ctx, d->d_tc_slice_tile, st.data(), st.size()));
        d->slice_for_groups = q->tc_ngroups;
    }
    const uint32_t nsingle = d->tc_nsingle, nslices = d->tc_nslices;
    // one candidate list per (slice, query): the four slots are merged inside the CTA
    SS_CUDA(ctx, d->d_tc_partial.reserve((size_t)nslices * nslots * kp));
    SS_CUDA(ctx, d->d_cand_idx.reserve((size_t)nslots * kp));
    SS_CUDA(ctx, d->d_cand_adist.reserve((size_t)nslots * kp));
    if (!d->ev_scan0) {
        SS_CUDA(ctx, cudaEventCreate(&d->ev_scan0));
        SS_CUDA(ctx, cudaEventCreate(&d->ev_scan1));
    }
    TcParams& p = plan->p;
    p.a_blocks = q->d_tc_a.p;
    p.group_off = q->d_tc_group_off.p;
    p.group_len = q->d_tc_group_len.p;
    p.slot_len = q->d_tc_slot_len.p;
    p.ngroups = q->tc_ngroups;
    p.tiles = reinterpret_cast<const unsigned char*>(d->d_tc_tiles.p);
    p.desc = d->d_tc_desc.p;
    p.slice_tile = d->d_tc_slice_tile.p;
    p.nslices = nslices;
    p.slice_begin = 0;
    p.partial = d->d_tc_partial.p;
    p.max_len = q->max_len;
    p.dbg = nullptr;
    p.dbg_nseg = 0;
    plan->nsingle = nsingle;
    plan->nslices = nslices;
    plan->nslots = nslots;
    plan->smem = (size_t)q->max_len * kTcATileBytes + kTcStages * kTcBTileBytes + 32 * 8 + (size_t)kp * kTcDpThreads * 8 + 1024;
    return SS_OK;
}

// the fp32-DP tensor-core scan takes segments and queries of at most kTcMaxLen frames
bool dtw_tc_applies(const ss_dict* d, const ss_queries* q) {
    return d->tc_ready && q->max_len <= (uint32_t)kTcMaxLen && q->total_frames > 0;
}

// the scan of batch q (dtw_tc_applies), its f64 refine and certification
int dtw_tc_match_dev(ss_dict* d, ss_queries* q, int k, bool timed, uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    SS_TRY(tc_queries_build(d, q));
    const int kp = k <= 2 ? 8 : 16;  // fp16 products are noisier than the fp32 scan: keep a longer candidate list
    TcPlan plan;
    SS_TRY(tc_plan(d, q, kp, &plan));
    if (kp == 8) SS_TRY(tc_launch<8>(ctx, plan.p, plan.nsingle, plan.nslices, plan.smem, plan.nslices, plan.nslots, d, timed));
    else SS_TRY(tc_launch<16>(ctx, plan.p, plan.nsingle, plan.nslices, plan.smem, plan.nslices, plan.nslots, d, timed));
    // certification bound for fp16 inputs: see k_dtw_finalize (bound_mode 1)
    return dtw_rescore_finalize(d, q, k, kp, plan.nslots, q->d_tc_qid.p, 0.0, q->d_tc_max_norm.p, d->d_tc_max_norm.p, q->d_tc_slot_max_na.p, 1,
                                q->d_uncert_flag.p, d_out_idx, d_out_dist);
}

// ss_dict_debug_tc_scan: the tensor-core scan's raw (filter-stage) distance of EVERY (query, segment) pair, plus the mean
// frame and norm scale the fp16 operands were built with. d_out: [nq][nseg] floats on the device, pre-filled by the caller
// (pairs the scan does not evaluate - empty queries / segments - keep that fill). Runs the production kernel with its
// DBG store compiled in; returns SS_ERR_INVALID if these inputs would not take the tensor-core path.
int dtw_tc_debug_scan(ss_dict* d, ss_queries* q, float* d_out, std::vector<uint32_t>* slot_qid, double* mu16, float* scale) {
    ss_ctx* ctx = d->ctx;
    if (!dtw_tc_applies(d, q))
        return set_error(ctx, SS_ERR_INVALID, "debug_tc_scan: the tensor-core scan does not apply (segments / queries > %d frames, or no frame)", kTcMaxLen);
    SS_TRY(tc_queries_build(d, q));
    TcPlan plan;
    SS_TRY(tc_plan(d, q, 8, &plan));
    plan.p.dbg = d_out;
    plan.p.dbg_nseg = (uint32_t)d->nseg;
    SS_TRY((tc_launch_kind<8, false, true>(ctx, plan.p, 0, plan.nsingle, plan.smem, false)));
    SS_TRY((tc_launch_kind<8, true, true>(ctx, plan.p, plan.nsingle, plan.nslices - plan.nsingle, plan.smem, plan.nsingle != 0)));
    slot_qid->resize(plan.nslots);
    SS_CUDA(ctx, cudaMemcpyAsync(slot_qid->data(), q->d_tc_qid.p, plan.nslots * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaMemcpyAsync(mu16, d->d_mu.p, 16 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *scale = d->tc_nb_scale;
    return SS_OK;
}

}  // namespace ss
