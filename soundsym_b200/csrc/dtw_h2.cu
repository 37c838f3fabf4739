// dtw_h2.cu — the FIRST filter stage of the DTW matcher when every segment and query has <= 32 frames: the tensor-core scan
// with the DP recurrence in PACKED HALF precision, two dictionary segments per register.
//
// Why: the fp32 scan (dtw_tc.cu) is bound by CUDA-core issue of one FMNMX3 + one FADD per cell; FMNMX3 issues at 16 lanes /
// clk / SMSP, so 64 cells / clk / SM is its hard ceiling (47.3 measured for the band alone, tools/microbench_band2.cu).
// VHMNMX (three-input min on half2) and HADD2 issue at the same instruction rate and carry two values each: the same band on
// half2 registers reaches 80-86 cells / clk / SM. The tensor core delivers the local costs already in that form: with an F16
// accumulator (instruction-descriptor c_format = 0) tcgen05.mma writes rn_f16(exact sum of the 16 products) - measured
// bit for bit on 16 384 operand pairs shaped like ours, tools/microbench_f16acc.cu - one 16-bit value per TMEM column, and
// tcgen05.ld ... .pack::16b returns two ADJACENT columns in one register. The dictionary tiles therefore interleave the
// columns of two segments (column 2t = frame t of the first, 2t + 1 = frame t of the second), so a register holds the same
// cell of two independent DTW problems and one VHMNMX + one HADD2 advance both.
//
// What the scan value means (the certification in exact.cu, bound_mode 2, rests on exactly this):
//   operands  A_i[m, :] = S [-2 a~ (13), s, s, rd(|a~|^2 / s)],  B[n, :] = [b~ (13), hi, lo, s]  (a~, b~ = fp16-rounded centred
//             frames, S a power of two that keeps path sums inside the fp16 range), so the exact contraction is S c'(i, j) with
//             c' <= c~ = |a~ - b~|^2 (by at most 2^-10 |a~|^2, from the round-down of |a~|^2);
//   cost      h(i, j) = rn16(S c')                         <= S c~ (1 + u) + eta16,        u = 2^-11
//   DP        D16(i, j) = rn16(h + min3(...))              <= (h + min3)(1 + u) + eta16     (min is exact, rn is monotone)
//   so along the optimal path of the rounded-frame DTW (<= Lq + Ld - 1 cells):  D16 <= S DTW~ (1 + u)^(Lq + Ld) + (Lq + Ld) 2 eta16,
//   i.e.  DTW~ / (Lq + Ld) >= [ D16 / (S (Lq + Ld)) - 2 eta16 / S ] (1 + u)^-(Lq + Ld): a pair dropped from a candidate list whose
//   worst entry is w has rounded-frame distance >= (w - eta)(1 + u)^-(Lq + 32). eta16 = 2^-25 covers fp16 subnormals (cost
//   operands scaled by S, running sums); an overflow to +inf only happens above 65504 / S and is capped in the bound.
//
// Geometry: 128 queries per CTA (= MMA M = TMEM lanes), MMA N = 128 TMEM columns per row = 2 slots x 64 columns, K = 16,
// two rows per pipeline step, two 256-column TMEM buffers. 8 DP warps (warp w: lane quadrant w % 4, slot w / 4) + 1 producer
// warp (TMEM allocation, bulk-TMA of the A block and the B-tile ring, MMA issue). A DP thread owns one query x one slot: NB
// bands of 2 interleaved segments each - NB = 1 (segments of 17..32 frames), 2 (9..16) or 4 (<= 8): every step is
// 2 rows x 64 columns = 128 cells per thread whatever the segment length, so the hand-off cost per cell is the same for
// short and long segments (the fp32 scan's paired tiles spent 4.5 instructions per cell on short segments).
// With 8 candidates per query (k <= 2) the NB = 1 and NB = 2 tiles run k_dtw_scan_h2_2p instead: the same geometry twice in
// one CTA, two pipelines of 8 DP warps + 1 producer warp that each own one 2-row TMEM buffer and take every other tile of the
// slice, so that one pipeline's warps issue while the other's wait for their MMAs or close a tile (640 threads, setmaxnreg:
// DP 112 registers, each step's columns pulled in two chunks).
//
// Code: the band recurrence (tc_band / tc_band_row over __half2), the capture-free step driver on the double-buffered cursor
// (tc_steps), TMEM allocation and the CTA's exit (tc_tmem_alloc / tc_cta_exit), the producer lane (tc_produce), the merge
// and write of a query's slot lists (tc_merge_store) and the launch (tc_launch_scan, tc_smem_bytes) come from tc_common.cuh,
// shared with dtw_tc.cu's fp32 scan. This file keeps the packed loads and picks, the single-buffer cursor of the two
// pipelines (H2PipeCursor) and its step loop in h2_tile, the strip of a long segment (h2_tile_strip), the helpers only its
// kernels share (h2_cta_slice: CTA order; h2_timeline_open; h2_push_tile: a tile's results into the unsorted list), the
// streamed-A producer of k_dtw_scan_h2_long, and the host side.
#include <algorithm>
#include <atomic>
#include <type_traits>

#include "match.cuh"
#include "tc_common.cuh"

namespace ss {

int dtw_second_chance(ss_dict* d, ss_queries* q, int k, int kp, uint32_t nslots, const uint32_t* d_slot_qid, const unsigned long long* d_partial,
                      uint32_t nlists, const unsigned long long* d_thr, double eps, const float* d_max_na, const float* d_max_nb,
                      const float* d_slot_max_na, int bound_mode, uint8_t* d_uncert_flag, uint32_t* d_out_idx, double* d_out_dist);

constexpr int kH2Slots = 2;
constexpr int kH2SlotCols = 64;                       // TMEM columns per slot and row
constexpr int kH2DpWarps = 4 * kH2Slots;              // 8
constexpr int kH2DpThreads = kH2DpWarps * 32;         // 256
constexpr int kH2Threads = (kH2DpWarps + 1) * 32;     // 288
constexpr int kH2DescInt4 = 4;                        // per (tile, slot): {seg 0..3}, {seg 4..7}, {columns 0..3 bytes, 4..7 bytes, ng, flags | strip << 8}, {whole length of seg 0..3}
constexpr int kH2In = 1, kH2Out = 2;                   // strip flags: boundary column comes in from / goes out to the neighbouring strip
constexpr int kH2ARing = 32;                          // rows of the A block resident at a time when a query group is longer (4 pieces of 8)
constexpr int kH2MaxLong = 2048;                      // longest segment / query the strip kernel takes (boundary scratch: %nsmid x rows x 1 KB)
// k_dtw_scan_h2_2p: two independent pipelines of 8 DP warps per CTA, each with its own 2-row TMEM buffer and producer warp
constexpr int kH2Pipes = 2;
constexpr int kH2PDpWarps = kH2Pipes * kH2DpWarps;       // 16; warp w: lane quadrant w % 4, slot (w >> 2) & 1, pipeline w >> 3
constexpr int kH2PDpThreads = kH2PDpWarps * 32;          // 512
constexpr int kH2PThreads = (kH2PDpWarps + 4) * 32;      // 640: warps 16, 17 = the producers, 18, 19 = idle register donors
// setmaxnreg: 640 threads launch with 96 registers; DP 112 / producer warpgroup 32 is the whole pool (512 x 112 + 128 x 32)
constexpr int kH2PRegsDp = 112, kH2PRegsProd = 32;
static_assert(kH2PDpThreads * kH2PRegsDp + 128 * kH2PRegsProd == kH2PThreads * 96, "setmaxnreg budget must match the launch pool");

struct H2Params {
    const unsigned char* a_blocks;
    const uint64_t* group_off;
    const uint32_t* group_len;   // longest | shortest << 16 query length of each group of 128
    const uint32_t* slot_len;    // per query slot: its own length (0 = padding lane)
    uint32_t ngroups;
    const unsigned char* tiles;  // ntiles x 4 KB, K-major no-swizzle, interleaved segment columns
    const int4* desc;            // [ntiles][2 slots][3]
    const uint32_t* slice_tile;  // all slices + 1
    uint32_t nslices, slice_begin;
    unsigned long long* partial;  // [nslices][ngroups * 128][KP]
    uint32_t max_len;
    float inv_s;                  // 1 / S
    // [ngroups * 128] per query: the smallest "worst kept key" any finished CTA reported. A CTA that kept KP candidates all
    // below T proves that nothing >= T is in the query's global top-KP, so later CTAs start with that threshold instead of an
    // empty list's +inf and skip almost every insertion (a CTA's first few hundred pairs are otherwise mostly insertions).
    unsigned long long* thr;
    float* dbg;                   // DBG instantiation only: [ngroups * 128][dbg_nseg]
    uint32_t dbg_nseg;
    __half2* bnd;                 // LONG kernel: [%nsmid][bnd_rows][256] boundary columns between the strips of a long segment
    uint32_t bnd_rows;
    float eta;                    // LONG kernel: subtracted from a pair's scan distance before its key is deflated (bound_mode 3)
    // measurement hook (SS_DTW_H2_TIMELINE=<file>, nullptr otherwise): per CTA {start, setup done, DP done, end} in %globaltimer ns,
    // then {smid | kind << 16 | group << 32, SM cycles (clock64) between stamps 1 and 2, end of the first half of the tiles,
    // L << 32 | tiles} - [grid][8] u64, written by thread 0
    unsigned long long* timeline;
};
// this CTA's 8 timeline words (p.timeline != nullptr)
__device__ __forceinline__ unsigned long long* h2_timeline_of(const H2Params& p) {
    return p.timeline + ((size_t)(p.slice_begin * p.ngroups) + blockIdx.x) * 8;
}
__device__ __forceinline__ unsigned long long h2_now() {
    unsigned long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// the timeline's opening stamps (thread 0): start, SM, tile kind NB, group, group length and tiles of the slice
__device__ __forceinline__ void h2_timeline_open(unsigned long long* tl, int nb, uint32_t g, uint32_t L, uint32_t ntiles) {
    unsigned smid;
    asm("mov.u32 %0, %%smid;" : "=r"(smid));
    tl[0] = h2_now(), tl[4] = smid | ((unsigned long long)nb << 16) | ((unsigned long long)g << 32), tl[7] = ((unsigned long long)L << 32) | ntiles;
}
// CTA order of k_dtw_scan_h2 / _2p: the FIRST slice of every group, then the other slices group by group (longest groups first
// in both parts). The slices of a group otherwise start together and none of them ever sees a sibling's threshold: with an
// empty threshold a thread's list takes 8 (1 + ln(n / 8)) sorted insertions over the n pairs of its slice, whatever n - per
// unit of work 5 times more on a 1/8 shard (ncu: 2.8 x the shared-memory wavefronts, + 5.7 % instructions, + 8 % cycles
// per step). With the first slice's threshold published before most of the others start, ~KP pairs per slice pass.
// Measured: 4.90 -> 4.85 ms on a 1/8 shard, 36.08 -> 35.97 ms at config 4 (the insertions were a part of the loss, not all
// of it: profiles/r2_h2_cycles_per_tile_eighth_vs_full.txt). Restricting the order to the first launch measured the same.
__device__ __forceinline__ void h2_cta_slice(const H2Params& p, uint32_t& g, uint32_t& slice) {
    if (blockIdx.x < p.ngroups) {
        g = blockIdx.x, slice = p.slice_begin;
    } else {
        const uint32_t r = blockIdx.x - p.ngroups;
        g = r / (p.nslices - 1), slice = p.slice_begin + 1 + r % (p.nslices - 1);
    }
}

// ---- packed TMEM loads: N registers <- 2 N adjacent columns ---------------------------------------------------------------
template <int N>
__device__ __forceinline__ void h2_ld(uint32_t taddr, __half2* v);
template <>
__device__ __forceinline__ void h2_ld<4>(uint32_t taddr, __half2* v) {
    uint32_t r[4];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.pack::16b.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 4; i++) v[i] = *reinterpret_cast<__half2*>(&r[i]);
}
template <>
__device__ __forceinline__ void h2_ld<8>(uint32_t taddr, __half2* v) {
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.pack::16b.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 8; i++) v[i] = *reinterpret_cast<__half2*>(&r[i]);
}
template <>
__device__ __forceinline__ void h2_ld<16>(uint32_t taddr, __half2* v) {
    uint32_t r[16];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.pack::16b.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 16; i++) v[i] = *reinterpret_cast<__half2*>(&r[i]);
}
// the 4 NG registers (8 NG columns) of one band row, as 16 / 8 / 4-register pieces
template <int NG>
__device__ __forceinline__ void h2_ld_row(uint32_t taddr, __half2 (&v)[4 * NG]) {
    constexpr int N = 4 * NG;
    int done = 0;
    if constexpr (N >= 32) {
        h2_ld<16>(taddr, v);
        h2_ld<16>(taddr + 32, v + 16);
        done = 32;
    } else if constexpr (N >= 16) {
        h2_ld<16>(taddr, v);
        done = 16;
    }
    if constexpr ((N & 8) != 0) {
        h2_ld<8>(taddr + 2 * done, v + done);
        done += 8;
    }
    if constexpr ((N & 4) != 0) h2_ld<4>(taddr + 2 * done, v + done);
}

__device__ __forceinline__ __half2 h2_inf() {
    const uint32_t bits = 0x7C007C00u;
    return *reinterpret_cast<const __half2*>(&bits);
}
__device__ __forceinline__ __half2 h2_zero() {
    const uint32_t bits = 0u;
    return *reinterpret_cast<const __half2*>(&bits);
}
// low half of a, high half of b
__device__ __forceinline__ __half2 h2_combine(__half2 a, __half2 b) {
    const uint32_t r = __byte_perm(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b), 0x7610);
    return *reinterpret_cast<const __half2*>(&r);
}
// element e (0..7) of a slot descriptor; e is a compile-time constant after unrolling, so these fold to register reads
// (arrays indexed in unrolled loops ended up in local memory)
__device__ __forceinline__ int h2_len_of(const int4& sc, int e) { return (int)((((e < 4) ? (uint32_t)sc.x : (uint32_t)sc.y) >> (8 * (e & 3))) & 0xFFu); }
__device__ __forceinline__ int h2_seg_of(const int4& sa, const int4& sb, int e) {
    return e == 0 ? sa.x : e == 1 ? sa.y : e == 2 ? sa.z : e == 3 ? sa.w : e == 4 ? sb.x : e == 5 ? sb.y : e == 6 ? sb.z : sb.w;
}
// v[r], r in 0..3, as three selects on registers (a plain ternary chain over an array is turned into an indexed load from local
// memory by the compiler, which put the capture values on the stack)
__device__ __forceinline__ uint32_t h2_selp(uint32_t a, uint32_t b, int pick_a) {
    uint32_t r;
    asm("{\n.reg .pred q;\nsetp.ne.s32 q, %3, 0;\nselp.b32 %0, %1, %2, q;\n}\n" : "=r"(r) : "r"(a), "r"(b), "r"(pick_a));
    return r;
}
__device__ __forceinline__ __half2 h2_pick4(const __half2* v, int r) {
    const uint32_t v0 = *reinterpret_cast<const uint32_t*>(&v[0]), v1 = *reinterpret_cast<const uint32_t*>(&v[1]);
    const uint32_t v2 = *reinterpret_cast<const uint32_t*>(&v[2]), v3 = *reinterpret_cast<const uint32_t*>(&v[3]);
    const uint32_t lo = h2_selp(v1, v0, r & 1), hi = h2_selp(v3, v2, r & 1);
    const uint32_t o = h2_selp(hi, lo, r & 2);
    return *reinterpret_cast<const __half2*>(&o);
}

// consumer side of one pipeline's single 2-row TMEM buffer (k_dtw_scan_h2_2p): its "empty" barrier sits 16 bytes above its
// "full" barrier, as in TcCursor, but the buffer and the barriers never change - only the parity flips
struct H2PipeCursor {
    uint32_t par, full, taddr;
    __device__ __forceinline__ void wait() const {
        mb_wait_addr(full, par);
        tc_fence_after();
    }
    __device__ __forceinline__ void release() {
        tc_fence_before();
        mb_arrive_elect(full + 16);
        par ^= 1u;
    }
};

// one pipeline step for one thread: wait for the step's MMAs, pull the NB bands' columns of both rows, hand the buffer back,
// advance the bands. With the single-buffer cursor (112 registers) the columns come in two chunks of at most 32 registers:
// the first 16 registers of each row (NB = 1) or the first half of the bands, then the rest; the buffer goes back after the
// second chunk's loads.
template <int NB, int NG, class Cur>
__device__ __forceinline__ void h2_step2(Cur& cur, __half2 (&d)[NB][4 * NG], __half2 dinit, __half2 (&c0l)[NB][4]) {
    constexpr int kBandCols = kH2SlotCols / NB;
    cur.wait();
    const uint32_t taddr = cur.taddr;
    if constexpr (std::is_same<Cur, H2PipeCursor>::value && NB == 1) {
        static_assert(NG >= 5, "NB = 1 tiles have 5..8 column groups");
        TcCarry<__half2> c = {h2_inf(), dinit, h2_inf()};
        {
            __half2 a0[16], a1[16];
            h2_ld_row<4>(taddr, a0);
            h2_ld_row<4>(taddr + kTcN, a1);
            tc_wait_ld();
            tc_band<NG, 0, 16>(a0, a1, d[0], c, c0l[0]);
        }
        __half2 b0[4 * (NG - 4)], b1[4 * (NG - 4)];
        h2_ld_row<NG - 4>(taddr + 32, b0);
        h2_ld_row<NG - 4>(taddr + kTcN + 32, b1);
        tc_wait_ld();
        cur.release();
        tc_band<NG, 16, 4 * NG>(b0, b1, d[0], c, c0l[0]);
    } else if constexpr (std::is_same<Cur, H2PipeCursor>::value) {
        constexpr int H = NB / 2;
        {
            __half2 tm0[H][4 * NG], tm1[H][4 * NG];
#pragma unroll
            for (int b = 0; b < H; b++) {
                h2_ld_row<NG>(taddr + b * kBandCols, tm0[b]);
                h2_ld_row<NG>(taddr + kTcN + b * kBandCols, tm1[b]);
            }
            tc_wait_ld();
#pragma unroll
            for (int b = 0; b < H; b++) {
                TcCarry<__half2> c = {h2_inf(), dinit, h2_inf()};
                tc_band<NG, 0, 4 * NG>(tm0[b], tm1[b], d[b], c, c0l[b]);
            }
        }
        __half2 tm0[H][4 * NG], tm1[H][4 * NG];
#pragma unroll
        for (int b = 0; b < H; b++) {
            h2_ld_row<NG>(taddr + (H + b) * kBandCols, tm0[b]);
            h2_ld_row<NG>(taddr + kTcN + (H + b) * kBandCols, tm1[b]);
        }
        tc_wait_ld();
        cur.release();
#pragma unroll
        for (int b = 0; b < H; b++) {
            TcCarry<__half2> c = {h2_inf(), dinit, h2_inf()};
            tc_band<NG, 0, 4 * NG>(tm0[b], tm1[b], d[H + b], c, c0l[H + b]);
        }
    } else {
        __half2 tm0[NB][4 * NG], tm1[NB][4 * NG];
#pragma unroll
        for (int b = 0; b < NB; b++) {
            h2_ld_row<NG>(taddr + b * kBandCols, tm0[b]);
            h2_ld_row<NG>(taddr + kTcN + b * kBandCols, tm1[b]);
        }
        tc_wait_ld();
        cur.release();
#pragma unroll
        for (int b = 0; b < NB; b++) {
            TcCarry<__half2> c = {h2_inf(), dinit, h2_inf()};
            tc_band<NG, 0, 4 * NG>(tm0[b], tm1[b], d[b], c, c0l[b]);
        }
    }
}

// One dictionary tile for one thread (= one query x one slot = 2 NB segments). ra / rb: position of column len - 1 inside the
// last 4-column group, for the band's first (low halves) and second (high halves) segment. res[b] = D(Lm - 1, len - 1) of both.
// Cur: TcCursor (two TMEM buffers, k_dtw_scan_h2 / _long) or H2PipeCursor (one buffer per pipeline, k_dtw_scan_h2_2p).
// before_capture runs once, after the capture-free steps (k_dtw_scan_h2_2p loads the tile's segment ids there).
struct H2NoHook {
    __device__ __forceinline__ void operator()() const {}
};
template <int NB, int NG, class Cur, class Hook = H2NoHook>
__device__ __forceinline__ void h2_tile(uint32_t L, uint32_t lmin, uint32_t Lm, const int4& sc, Cur& cur, __half2 (&res)[NB],
                                        Hook before_capture = Hook()) {
    __half2 d[NB][4 * NG];
#pragma unroll
    for (int b = 0; b < NB; b++) {
#pragma unroll
        for (int j = 0; j < 4 * NG; j++) d[b][j] = h2_inf();
        res[b] = h2_inf();
    }
    __half2 dinit = h2_zero();
    const uint32_t nfull = L >> 1;                       // steps that carry two rows
    const uint32_t ncap = min((lmin - 1) >> 1, nfull);   // steps before any query of the group can end
    uint32_t st = 0;
    if constexpr (std::is_same<Cur, H2PipeCursor>::value) {
        // steps [0, ncap): no query of the group ends; one buffer, so every step has the same addresses. NB = 1 runs two steps
        // per iteration (the first step, the only one with D(-1, -1) = 0, before the loop): with one step per iteration ptxas
        // made the home registers of d[] the second chunk's TMEM-load destination and copied every new row value back, 22 - 36
        // moves per 80 - 128 band instructions; two steps let the row state and the loads trade registers (1 - 10 moves per
        // two steps, tools/sass_step_mix.py). NB = 2 spills its per-slice state to local memory when unrolled and keeps one.
        if constexpr (NB == 1) {
            if (st < ncap) {
                __half2 c0l[NB][4];
                h2_step2<NB, NG>(cur, d, dinit, c0l);
                dinit = h2_inf();
                st++;
            }
#pragma unroll 1
            for (; st + 2 <= ncap; st += 2) {
                __half2 c0l[NB][4];
                h2_step2<NB, NG>(cur, d, h2_inf(), c0l);
                h2_step2<NB, NG>(cur, d, h2_inf(), c0l);
            }
            if (st < ncap) {
                __half2 c0l[NB][4];
                h2_step2<NB, NG>(cur, d, h2_inf(), c0l);
                st++;
            }
        } else {
#pragma unroll 1
            for (; st < ncap; st++) {
                __half2 c0l[NB][4];
                h2_step2<NB, NG>(cur, d, dinit, c0l);
                dinit = h2_inf();
            }
        }
        before_capture();
    } else {
        st = tc_steps(cur, ncap, dinit, h2_inf(), [&](TcCursor& c, __half2 di) {  // no query of the group ends in steps [0, ncap)
            __half2 c0l[NB][4];
            h2_step2<NB, NG>(c, d, di, c0l);
        });
    }
#pragma unroll 1
    for (; st < nfull; st++) {  // only the last step or two of a tile: some query of the group can end here
        __half2 c0l[NB][4];
        h2_step2<NB, NG>(cur, d, dinit, c0l);
        dinit = h2_inf();
        const bool end0 = 2 * st + 1 == Lm, end1 = 2 * st + 2 == Lm;
#pragma unroll
        for (int b = 0; b < NB; b++) {
            const int ra = (h2_len_of(sc, 2 * b) - 1) & 3, rb = (h2_len_of(sc, 2 * b + 1) - 1) & 3;
            const __half2 e0 = h2_combine(h2_pick4(c0l[b], ra), h2_pick4(c0l[b], rb));
            const __half2 e1 = h2_combine(h2_pick4(&d[b][4 * (NG - 1)], ra), h2_pick4(&d[b][4 * (NG - 1)], rb));
            res[b] = end0 ? e0 : (end1 ? e1 : res[b]);
        }
    }
    if (L & 1) {  // odd group length: the last step carries one row
        constexpr int kBandCols = kH2SlotCols / NB;
        cur.wait();
        __half2 tm0[NB][4 * NG];
#pragma unroll
        for (int b = 0; b < NB; b++) h2_ld_row<NG>(cur.taddr + b * kBandCols, tm0[b]);
        tc_wait_ld();
        cur.release();
#pragma unroll
        for (int b = 0; b < NB; b++) {
            tc_band_row<NG>(tm0[b], d[b], h2_inf(), dinit);
            const int ra = (h2_len_of(sc, 2 * b) - 1) & 3, rb = (h2_len_of(sc, 2 * b + 1) - 1) & 3;
            const __half2 e = h2_combine(h2_pick4(&d[b][4 * (NG - 1)], ra), h2_pick4(&d[b][4 * (NG - 1)], rb));
            res[b] = (L == Lm) ? e : res[b];
        }
    }
}

// One 32-column strip of two long segments for one thread. IN: the strip continues a previous one (boundary column read
// from `bnd`, [row][256 threads]); OUT: another strip follows (this strip's last column written back in place, nothing
// captured). The LAST strip (IN && !OUT) captures D(Lm - 1, len - 1) like a whole-segment tile.
template <int NG, bool IN, bool OUT>
__device__ __forceinline__ void h2_tile_strip(uint32_t L, uint32_t lmin, uint32_t Lm, const int4& sc, TcCursor& cur, __half2* bnd, __half2& res) {
    constexpr uint32_t kStride = kH2DpThreads;
    __half2 d[4 * NG];
#pragma unroll
    for (int j = 0; j < 4 * NG; j++) d[j] = h2_inf();
    res = h2_inf();
    __half2 prev_b = IN ? h2_inf() : h2_zero();  // D(i - 1, -1): +inf above the first row of a later strip, the virtual 0 of D(-1, -1) in the first
    const uint32_t nfull = L >> 1;
    const uint32_t ncap = OUT ? nfull : min((lmin - 1) >> 1, nfull);
    const int ra = (h2_len_of(sc, 0) - 1) & 3, rb = (h2_len_of(sc, 1) - 1) & 3;
#pragma unroll 1
    for (uint32_t st = 0; st < nfull; st++) {
        __half2 b0 = h2_inf(), b1 = h2_inf();
        if (IN) b0 = bnd[(size_t)(2 * st) * kStride], b1 = bnd[(size_t)(2 * st + 1) * kStride];  // issued ahead of the TMEM wait
        cur.wait();
        const uint32_t taddr = cur.taddr;
        __half2 tm0[4 * NG], tm1[4 * NG], c0l[4];
        h2_ld_row<NG>(taddr, tm0);
        h2_ld_row<NG>(taddr + kTcN, tm1);
        tc_wait_ld();
        cur.release();
        TcCarry<__half2> c = {b0, prev_b, b1};  // the previous strip's last column: D(i, -1), D(i-1, -1), D(i+1, -1)
        tc_band<NG, 0, 4 * NG>(tm0, tm1, d, c, c0l);
        prev_b = IN ? b1 : h2_inf();
        if (OUT) {  // this strip's last column, for the next strip
            bnd[(size_t)(2 * st) * kStride] = c.left0;
            bnd[(size_t)(2 * st + 1) * kStride] = c.left1;
        } else if (st >= ncap) {
            const bool end0 = 2 * st + 1 == Lm, end1 = 2 * st + 2 == Lm;
            const __half2 e0 = h2_combine(h2_pick4(c0l, ra), h2_pick4(c0l, rb));
            const __half2 e1 = h2_combine(h2_pick4(&d[4 * (NG - 1)], ra), h2_pick4(&d[4 * (NG - 1)], rb));
            res = end0 ? e0 : (end1 ? e1 : res);
        }
    }
    if (L & 1) {
        __half2 b0 = h2_inf();
        if (IN) b0 = bnd[(size_t)(L - 1) * kStride];
        cur.wait();
        __half2 tm0[4 * NG];
        h2_ld_row<NG>(cur.taddr, tm0);
        tc_wait_ld();
        cur.release();
        const __half2 o0 = tc_band_row<NG>(tm0, d, b0, prev_b);
        if (OUT) {
            bnd[(size_t)(L - 1) * kStride] = o0;
        } else {
            const __half2 e = h2_combine(h2_pick4(&d[4 * (NG - 1)], ra), h2_pick4(&d[4 * (NG - 1)], rb));
            res = (L == Lm) ? e : res;
        }
    }
}

// A tile's results res[b] (two segments per band) for query m of group g as candidates of this thread's list, kept UNSORTED
// while the slice is scanned (see k_dtw_scan_h2): a key below `worst` goes to the next free place (cnt) or, once the list is
// full, replaces its largest key (at wpos), and the new largest key and its place are found with KP independent loads.
// DBG also stores every pair's scan distance.
template <int KP, int STRIDE, int NB, bool DBG>
__device__ __forceinline__ void h2_push_tile(const H2Params& p, uint32_t g, int m, uint32_t Lm, const int4& sa, const int4& sb, const int4& sc,
                                             const __half2 (&res)[NB], unsigned long long* list, unsigned long long& worst, unsigned long long thr0,
                                             int& cnt, int& wpos) {
    if (Lm) {
#pragma unroll
        for (int b = 0; b < NB; b++) {
#pragma unroll
            for (int hsel = 0; hsel < 2; hsel++) {
                const int e = 2 * b + hsel;
                const int seg = h2_seg_of(sa, sb, e);
                if (seg >= 0) {
                    const float v = hsel ? __high2float(res[b]) : __low2float(res[b]);
                    // D16 / (S (Lq + Ld)); an overflowed path sum stays +inf and is never inserted
                    const float dist = __fdividef(v * p.inv_s, (float)(Lm + (uint32_t)h2_len_of(sc, e)));
                    const unsigned long long key = ((unsigned long long)f2ord(dist) << 32) | (uint32_t)seg;
                    if (key < worst && dist == dist) {
                        const bool full = cnt == KP;
                        list[(full ? wpos : cnt) * STRIDE] = key;
                        cnt += full ? 0 : 1;
                        if (cnt == KP) {
                            tc_list_max<KP, STRIDE>(list, worst, wpos);
                            worst = worst < thr0 ? worst : thr0;
                        }
                    }
                    if constexpr (DBG) p.dbg[(size_t)(g * kTcM + m) * p.dbg_nseg + seg] = dist;
                }
            }
        }
    }
}

// NB selects the tile kind the launch covers (the dictionary's tiles are sorted: NB = 1 tiles first, then 2, then 4).
template <int KP, int NB, bool DBG = false>
__global__ void __launch_bounds__(kH2Threads, 1) k_dtw_scan_h2(const H2Params p) {
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
    unsigned long long* topk = reinterpret_cast<unsigned long long*>(bars + 32);  // [KP][256]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t g, slice;
    h2_cta_slice(p, g, slice);
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next tile kind's launch may start filling SMs
    const uint32_t glen = p.group_len[g];
    const uint32_t L = glen & 0xFFFFu, lmin = glen >> 16;
    const uint32_t t0 = p.slice_tile[slice], t1 = p.slice_tile[slice + 1];
    const uint32_t ntiles = t1 - t0;
    unsigned long long* tl = p.timeline ? h2_timeline_of(p) : nullptr;
    if (tl && threadIdx.x == 0) h2_timeline_open(tl, NB, g, L, ntiles);

    if (threadIdx.x == 0) {
        mb_init(a_full, 1);
        for (int s = 0; s < kTcStages; s++) mb_init(&b_full[s], 1), mb_init(&b_empty[s], 1);
        for (int s = 0; s < 2; s++) mb_init(&t_full[s], 1), mb_init(&t_empty[s], kH2DpWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t tmem_base = tc_tmem_alloc(warp == kH2DpWarps, tmem_slot);
    if (tl && threadIdx.x == 0) tl[1] = h2_now(), tl[5] = clock64();
    if (warp == kH2DpWarps) {
        if (lane == 0 && ntiles) {
            const uint32_t bars_s = s32(bars);
            tc_produce<1>(p, g, L, t0, ntiles, 0, kTcIdescF16, s32(sA), s32(sB), bars_s, bars_s + 8, bars_s + 80, tmem_base);
        }
    } else {
        // ---- DP warps ---------------------------------------------------------------------------------------------------
        const int q = warp & 3, slot = warp >> 2;
        const int m = q * 32 + lane;
        unsigned long long* list = topk + threadIdx.x;  // [KP][256] keys, this thread's column
#pragma unroll
        for (int s = 0; s < KP; s++) list[s * kH2DpThreads] = 0xFFFFFFFFFFFFFFFFull;
        const unsigned long long thr0 = __ldcg(p.thr + g * kTcM + m);  // (L2: other CTAs update it)
        unsigned long long worst = thr0;
        // The list is kept UNSORTED while the slice is scanned: a candidate below `worst` goes to the next free place or, once
        // the list is full, replaces its largest key, and the new largest key and its place are found with KP independent loads
        // - the same work for every lane of the warp, where a sorted insertion is a walk of data-dependent length through
        // dependent shared-memory loads and stores that a warp pays at its slowest lane's pace (on a 1/8 shard, where a slice is
        // 80 tiles, that was most of the + 400 SM cycles per tile of profiles/r2_h2_cycles_per_tile_eighth_vs_full.txt). The
        // list is sorted once, at the end of the slice.
        int cnt = 0, wpos = 0;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + slot * kH2SlotCols;
        const uint32_t Lm = p.slot_len[g * kTcM + m];  // this lane's own query length
        TcCursor cur;
        cur.init(s32(t_full), lane_addr);
        // the NEXT tile's descriptors are fetched while the current tile is processed: a tile of a short query group is only 2 - 4
        // steps long, and an L2 round trip at its start stalled the warp - and within two steps the whole pipeline
        const int4* dp = p.desc + ((size_t)t0 * kH2Slots + slot) * kH2DescInt4;
        int4 na = make_int4(0, 0, 0, 0), nb = na, nc = na;
        if (ntiles) na = __ldg(dp), nb = __ldg(dp + 1), nc = __ldg(dp + 2);
        for (uint32_t n = 0; n < ntiles; n++) {
            const int4 sa = na, sb = nb, sc = nc;
            dp += kH2Slots * kH2DescInt4;
            if (n + 1 < ntiles) na = __ldg(dp), nb = __ldg(dp + 1), nc = __ldg(dp + 2);
            const int ng = sc.z;
            __half2 res[NB];
            // every segment of a tile has the same number of 4-column groups: straight-line code over 4 NG registers per band
            if constexpr (NB == 1) {
                switch (ng) {
                    case 5: h2_tile<1, 5>(L, lmin, Lm, sc, cur, res); break;
                    case 6: h2_tile<1, 6>(L, lmin, Lm, sc, cur, res); break;
                    case 7: h2_tile<1, 7>(L, lmin, Lm, sc, cur, res); break;
                    default: h2_tile<1, 8>(L, lmin, Lm, sc, cur, res); break;
                }
            } else if constexpr (NB == 2) {
                if (ng == 3) h2_tile<2, 3>(L, lmin, Lm, sc, cur, res);
                else h2_tile<2, 4>(L, lmin, Lm, sc, cur, res);
            } else {
                if (ng == 1) h2_tile<4, 1>(L, lmin, Lm, sc, cur, res);
                else h2_tile<4, 2>(L, lmin, Lm, sc, cur, res);
            }
            if (tl && threadIdx.x == 0 && n + 1 == (ntiles + 1) / 2) tl[6] = h2_now();  // (measurement: the slice's half-way mark)
            h2_push_tile<KP, kH2DpThreads, NB, DBG>(p, g, m, Lm, sa, sb, sc, res, list, worst, thr0, cnt, wpos);
        }
        tc_sort_list<KP, kH2DpThreads>(list, cnt);  // (the places beyond cnt still hold the initial +inf keys)
        worst = list[(KP - 1) * kH2DpThreads];
        worst = worst < thr0 ? worst : thr0;
        // the two slots' lists of query m (threads m, m + 128) are merged by the slot-0 thread
        asm volatile("bar.sync 1, %0;" ::"n"(kH2DpThreads) : "memory");
        if (tl && threadIdx.x == 0) tl[2] = h2_now(), tl[5] = clock64() - tl[5];  // SM cycles of the DP phase (-> the SM clock under load)
        if (slot == 0)
            tc_merge_store<KP, kH2DpThreads, kH2Slots, true>(list, worst, thr0, [&] {
                return TcListDst{p.thr + g * kTcM + m, p.partial + ((size_t)slice * p.ngroups * kTcM + (size_t)g * kTcM + m) * KP};
            });
    }
    tc_cta_exit<NB != 1>(warp == kH2DpWarps, tmem_base);  // the NB = 2 and 4 launches are the dependent ones
    if (tl && threadIdx.x == 0) tl[3] = h2_now();
}

// ---- the same scan with TWO PIPELINES per CTA (KP = 8, the first stage for k <= 2). In k_dtw_scan_h2 all 8 DP warps wait
// for the same buffer, load it, hand it back and reach the end of a tile together, so nothing covers those latencies (ncu:
// 2.25 eligible warps per scheduler, issue 47 %). Here pipeline p = 0, 1 walks the tiles t0 + p, t0 + p + 2, .. of the
// slice with its own 8 DP warps, its own 2-row TMEM buffer (columns [256 p, 256 p + 256)), its own producer warp with its
// own B ring and barriers: the two run out of phase, and while one waits for its MMAs or closes a tile the other's warps
// issue. The A block is copied once (producer 0) and both producers wait for it. MMA shape, operands and the band code are
// those of k_dtw_scan_h2, so every pair's scan value has the same bits. The 4 lists of a query (2 slots x 2 pipelines) are
// merged before the partial write.
template <int KP, int NB, bool DBG = false>
__global__ void __launch_bounds__(kH2PThreads, 1) k_dtw_scan_h2_2p(const H2Params p) {
    extern __shared__ unsigned char smem_raw[];
    // [A tiles: max_len x 4 KB][B rings: 2 pipelines x 4 x 4 KB][barriers][candidate lists [KP][512]], 128-byte aligned
    unsigned char* smem = smem_raw + ((128u - (s32(smem_raw) & 127u)) & 127u);
    unsigned char* sA = smem;
    unsigned char* sB = smem + (size_t)p.max_len * kTcATileBytes;
    // barriers (u64): a_full | b_full[4], b_empty[4] of pipeline 0 | the same of pipeline 1 | t_full[2] | t_empty[2]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sB + kH2Pipes * kTcStages * kTcBTileBytes);
    uint64_t* a_full = bars;
    uint64_t* t_full = bars + 1 + 2 * kH2Pipes * kTcStages;  // 17
    uint64_t* t_empty = t_full + kH2Pipes;                   // = t_full + 16 bytes (H2PipeCursor::release)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(t_empty + kH2Pipes);
    // the CTA's query group and slice, read back by the list merge at the end: held in registers through the slice, they
    // pushed the NB = 1 kernel's two-step loop into local memory
    uint32_t* cta_gs = reinterpret_cast<uint32_t*>(t_empty + kH2Pipes + 1);
    unsigned long long* topk = reinterpret_cast<unsigned long long*>(bars + 32);  // [KP][512]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t g, slice;
    h2_cta_slice(p, g, slice);
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next tile kind's launch may start filling SMs
    const uint32_t glen = p.group_len[g];
    const uint32_t L = glen & 0xFFFFu, lmin = glen >> 16;
    const uint32_t t0 = p.slice_tile[slice], t1 = p.slice_tile[slice + 1];
    const uint32_t ntiles = t1 - t0;
    unsigned long long* tl = p.timeline ? h2_timeline_of(p) : nullptr;
    if (tl && threadIdx.x == 0) h2_timeline_open(tl, NB, g, L, ntiles);

    if (threadIdx.x == 0) {
        cta_gs[0] = g, cta_gs[1] = slice;
        mb_init(a_full, 1);
        for (int s = 0; s < 2 * kH2Pipes * kTcStages; s++) mb_init(&bars[1 + s], 1);
        for (int s = 0; s < kH2Pipes; s++) mb_init(&t_full[s], 1), mb_init(&t_empty[s], kH2DpWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t tmem_base = tc_tmem_alloc(warp == kH2PDpWarps, tmem_slot);
    if (tl && threadIdx.x == 0) tl[1] = h2_now(), tl[5] = clock64();
    if (warp >= kH2PDpWarps) {
        asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kH2PRegsProd));
        const uint32_t pipe = (uint32_t)(warp - kH2PDpWarps);
        const uint32_t ntp = ntiles > pipe ? (ntiles - pipe + 1) >> 1 : 0u;  // this pipeline's tiles: t0 + pipe, t0 + pipe + 2, ..
        if (pipe < (uint32_t)kH2Pipes && lane == 0 && ntp) {
            const uint32_t bars_s = s32(bars);  // producer of pipeline `pipe`: its B ring, its MMAs; producer 0 also copies the A block
            tc_produce<kH2Pipes>(p, g, L, t0, ntp, pipe, kTcIdescF16, s32(sA), s32(sB), bars_s, bars_s + 8, s32(t_full), tmem_base);
        }
    } else {
        // ---- DP warps ---------------------------------------------------------------------------------------------------
        asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kH2PRegsDp));
        const int q = warp & 3, slot = (warp >> 2) & 1, pipe = warp >> 3;
        const int m = q * 32 + lane;
        unsigned long long* list = topk + threadIdx.x;  // [KP][512] keys, this thread's column
#pragma unroll
        for (int s = 0; s < KP; s++) list[s * kH2PDpThreads] = 0xFFFFFFFFFFFFFFFFull;
        const unsigned long long thr0 = __ldcg(p.thr + g * kTcM + m);  // (L2: other CTAs update it)
        unsigned long long worst = thr0;
        int cnt = 0, wpos = 0;  // unsorted list while the slice is scanned, as in k_dtw_scan_h2
        const uint32_t Lm = p.slot_len[g * kTcM + m];  // this lane's own query length
        H2PipeCursor cur = {0u, s32(t_full + pipe), tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(pipe * kTcBufCols + slot * kH2SlotCols)};
        const uint32_t ntp = ntiles > (uint32_t)pipe ? (ntiles - pipe + 1) >> 1 : 0u;
        // the NEXT tile's lengths and column groups are fetched while the current tile is processed; a tile's segment ids are
        // only read after its last step and are loaded after its capture-free steps, so that those steps hold no descriptor
        // registers beyond the lengths. The position is a 32-bit index into p.desc (its base stays in the constant bank): with
        // a 64-bit pointer held through the slice, the NB = 1 two-step loop spilled to local memory (tools/sass_step_mix.py)
        uint32_t di = ((t0 + pipe) * kH2Slots + slot) * kH2DescInt4;
        int4 nc = make_int4(0, 0, 0, 0);
        if (ntp) nc = __ldg(p.desc + di + 2);
        for (uint32_t n = 0; n < ntp; n++) {
            const int4 sc = nc;
            const uint32_t dcur = di;
            di += kH2Pipes * kH2Slots * kH2DescInt4;
            if (n + 1 < ntp) nc = __ldg(p.desc + di + 2);
            const int ng = sc.z;
            __half2 res[NB];
            int4 sa, sb;
            const auto load_segs = [&] { sa = __ldg(p.desc + dcur), sb = __ldg(p.desc + dcur + 1); };
            if constexpr (NB == 1) {
                switch (ng) {
                    case 5: h2_tile<1, 5>(L, lmin, Lm, sc, cur, res, load_segs); break;
                    case 6: h2_tile<1, 6>(L, lmin, Lm, sc, cur, res, load_segs); break;
                    case 7: h2_tile<1, 7>(L, lmin, Lm, sc, cur, res, load_segs); break;
                    default: h2_tile<1, 8>(L, lmin, Lm, sc, cur, res, load_segs); break;
                }
            } else {
                static_assert(NB == 2, "k_dtw_scan_h2_2p runs the NB = 1 and NB = 2 tiles");
                if (ng == 3) h2_tile<2, 3>(L, lmin, Lm, sc, cur, res, load_segs);
                else h2_tile<2, 4>(L, lmin, Lm, sc, cur, res, load_segs);
            }
            if (p.timeline && threadIdx.x == 0 && n + 1 == (ntp + 1) / 2) h2_timeline_of(p)[6] = h2_now();  // (measurement: half of pipeline 0's tiles)
            h2_push_tile<KP, kH2PDpThreads, NB, DBG>(p, g, m, Lm, sa, sb, sc, res, list, worst, thr0, cnt, wpos);
        }
        tc_sort_list<KP, kH2PDpThreads>(list, cnt);  // (the places beyond cnt still hold the initial +inf keys)
        worst = list[(KP - 1) * kH2PDpThreads];
        worst = worst < thr0 ? worst : thr0;
        // the four lists of query m (threads m + 128 s, s = slot + 2 pipeline) are merged by thread m
        asm volatile("bar.sync 1, %0;" ::"n"(kH2PDpThreads) : "memory");
        if (p.timeline && threadIdx.x == 0) {  // (the pointer is re-derived here: held through the slice it took two of the DP warps' registers)
            unsigned long long* t = h2_timeline_of(p);
            t[2] = h2_now(), t[5] = clock64() - t[5];  // SM cycles of the DP phase (-> the SM clock under load)
        }
        if (threadIdx.x < kTcM)
            tc_merge_store<KP, kH2PDpThreads, kH2Pipes * kH2Slots, true>(list, worst, thr0, [&] {
                const uint32_t gm = cta_gs[0] * kTcM + m;
                return TcListDst{p.thr + gm, p.partial + ((size_t)cta_gs[1] * p.ngroups * kTcM + gm) * KP};
            });
    }
    tc_cta_exit<NB != 1>(warp == kH2PDpWarps, tmem_base);
    if (tl && threadIdx.x == 0) tl[3] = h2_now();
}

// ---- the same scan for LONG sequences: dictionary segments of more than 32 frames are cut into 32-column strips (tiles of the
// NB = 1 kind, consecutive in the tile list) whose boundary column travels through a per-SM scratch in global memory, and a
// query group of more than 32 frames streams its A block through a ring of 4 x 8 rows. Separate kernel: the <= 32 x <= 32 case
// (the headline) keeps its own, simpler code.
template <int KP, int NB, bool DBG = false>
__global__ void __launch_bounds__(kH2Threads, 1) k_dtw_scan_h2_long(const H2Params p) {
    extern __shared__ unsigned char smem_raw[];
    // [A ring: 32 rows x 4 KB = 4 pieces of 8 rows][B ring: 4 x 4 KB][barriers][candidate lists], 128-byte aligned
    unsigned char* smem = smem_raw + ((128u - (s32(smem_raw) & 127u)) & 127u);
    unsigned char* sA = smem;
    unsigned char* sB = smem + (size_t)kH2ARing * kTcATileBytes;
    uint64_t* bars = reinterpret_cast<uint64_t*>(sB + kTcStages * kTcBTileBytes);
    uint64_t* a_full = bars;        // [4]
    uint64_t* a_empty = bars + 4;   // [4]
    uint64_t* b_full = bars + 8;    // [4]
    uint64_t* b_empty = bars + 12;  // [4]
    uint64_t* t_full = bars + 16;
    uint64_t* t_empty = bars + 18;  // = t_full + 16 bytes (TcCursor::release)
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 20);
    unsigned long long* topk = reinterpret_cast<unsigned long long*>(bars + 32);  // [KP][256]

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t g = blockIdx.x / p.nslices, slice = p.slice_begin + blockIdx.x % p.nslices;
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");  // the next tile kind's launch may start filling SMs
    const uint32_t glen = p.group_len[g];
    const uint32_t L = glen & 0xFFFFu, lmin = glen >> 16;
    const uint32_t t0 = p.slice_tile[slice], t1 = p.slice_tile[slice + 1];
    const uint32_t ntiles = t1 - t0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < 4; s++) mb_init(&a_full[s], 1), mb_init(&a_empty[s], 1);
        for (int s = 0; s < kTcStages; s++) mb_init(&b_full[s], 1), mb_init(&b_empty[s], 1);
        for (int s = 0; s < 2; s++) mb_init(&t_full[s], 1), mb_init(&t_empty[s], kH2DpWarps);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    const uint32_t tmem_base = tc_tmem_alloc(warp == kH2DpWarps, tmem_slot);
    if (warp == kH2DpWarps) {
        if (lane == 0 && ntiles) {
            // ---- producer: TMA + MMA issue. The group's A block (L rows) lives in a ring of 4 pieces of 8 rows. Up to 32 rows it
            // is loaded once and stays; a longer group STREAMS it: every tile consumes pieces 0 .. npieces - 1 in order, the
            // piece sequence runs on across tiles (n = tile * npieces + piece -> ring slot n % 4), and a slot is refilled one
            // piece after its MMAs were committed (their completion arrives on a_empty[slot]) -----------------------------------
            const uint32_t bars_s = s32(bars), sA_s = s32(sA), sB_s = s32(sB);
            const uint32_t a_full_s = bars_s, a_empty_s = bars_s + 32, b_full_s = bars_s + 64, b_empty_s = bars_s + 96, t_full_s = bars_s + 128,
                           t_empty_s = bars_s + 144;
            const uint32_t npieces = (L + 7) >> 3;
            const bool streaming = npieces > 4;
            const uint32_t total_pieces = streaming ? ntiles * npieces : npieces;
            const unsigned char* a_src = p.a_blocks + p.group_off[g];
            auto load_piece = [&](uint32_t n) {  // sequence number n -> piece n % npieces into ring slot
                const uint32_t pc = n % npieces, slot = streaming ? (n & 3u) : pc;
                const uint32_t rows = min(8u, L - 8u * pc);
                mbs_expect_tx(a_full_s + 8 * slot, rows * kTcATileBytes);
                tmas_g2s(sA_s + slot * 8 * kTcATileBytes, a_src + (size_t)pc * 8 * kTcATileBytes, rows * kTcATileBytes, a_full_s + 8 * slot);
            };
            for (uint32_t n = 0; n < total_pieces && n < 4; n++) load_piece(n);
            const unsigned char* tile_src = p.tiles + (size_t)t0 * kTcBTileBytes;
            for (uint32_t n = 0; n < ntiles && n < (uint32_t)kTcStages; n++) {
                mbs_expect_tx(b_full_s + 8 * n, kTcBTileBytes);
                tmas_g2s(sB_s + n * kTcBTileBytes, tile_src + (size_t)n * kTcBTileBytes, kTcBTileBytes, b_full_s + 8 * n);
            }
            tile_src += (size_t)kTcStages * kTcBTileBytes;
            const uint32_t idesc = kTcIdescF16;
            uint32_t cnt = 0, stage = 0, sphase = 0, use_n = 0;
            for (uint32_t n = 0; n < ntiles; n++) {
                mbs_wait_sleep(b_full_s + 8 * stage, sphase);
                const uint64_t bdesc = tc_smem_desc_s<kTcN>(sB_s + stage * kTcBTileBytes);
                for (uint32_t pc = 0; pc < npieces; pc++, use_n++) {
                    const uint32_t slot = streaming ? (use_n & 3u) : pc;
                    if (streaming && use_n >= 1 && use_n + 3 < total_pieces) {  // refill the slot the previous piece sat in
                        mbs_wait_sleep(a_empty_s + 8 * ((use_n - 1) & 3u), ((use_n - 1) >> 2) & 1);
                        load_piece(use_n + 3);
                    }
                    if (streaming || n == 0) mbs_wait_sleep(a_full_s + 8 * slot, streaming ? ((use_n >> 2) & 1) : 0u);
                    const uint64_t adesc0 = tc_smem_desc_s<kTcM>(sA_s + slot * 8 * kTcATileBytes);
                    const uint32_t rows = min(8u, L - 8u * pc);
                    for (uint32_t r = 0; r < rows; r += 2, cnt++) {
                        const uint32_t buf = cnt & 1;
                        if (cnt >= 2) mbs_wait_sleep(t_empty_s + 8 * buf, ((cnt >> 1) - 1) & 1);
                        tc_fence_after();
                        const uint32_t tm = tmem_base + buf * kTcBufCols;
                        const uint64_t adesc = adesc0 + (uint64_t)r * (kTcATileBytes >> 4);
                        tc_mma_f16(tm, adesc, bdesc, idesc);
                        if (r + 1 < rows) tc_mma_f16(tm + kTcN, adesc + (kTcATileBytes >> 4), bdesc, idesc);
                        tcs_commit(t_full_s + 8 * buf);
                    }
                    if (streaming) tcs_commit(a_empty_s + 8 * slot);
                }
                tcs_commit(b_empty_s + 8 * stage);
                if (n + kTcStages < ntiles) {
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
        const int q = warp & 3, slot = warp >> 2;
        const int m = q * 32 + lane;
        unsigned long long* list = topk + threadIdx.x;  // [KP][256] keys, this thread's column
#pragma unroll
        for (int s = 0; s < KP; s++) list[s * kH2DpThreads] = 0xFFFFFFFFFFFFFFFFull;
        const unsigned long long thr0 = __ldcg(p.thr + g * kTcM + m);  // (L2: other CTAs update it)
        unsigned long long worst = thr0;
        const uint32_t lane_addr = tmem_base + ((uint32_t)(q * 32) << 16) + slot * kH2SlotCols;
        const uint32_t Lm = p.slot_len[g * kTcM + m];  // this lane's own query length
        TcCursor cur;
        cur.init(s32(t_full), lane_addr);
        const int4* dp = p.desc + ((size_t)t0 * kH2Slots + slot) * kH2DescInt4;  // (next tile's descriptors prefetched, as above)
        int4 na = make_int4(0, 0, 0, 0), nb = na, nc = na, nd = na;
        if (ntiles) na = __ldg(dp), nb = __ldg(dp + 1), nc = __ldg(dp + 2), nd = __ldg(dp + 3);
        for (uint32_t n = 0; n < ntiles; n++) {
            const int4 sa = na, sb = nb, sc = nc, sd = nd;
            dp += kH2Slots * kH2DescInt4;
            if (n + 1 < ntiles) na = __ldg(dp), nb = __ldg(dp + 1), nc = __ldg(dp + 2), nd = __ldg(dp + 3);
            const int ng = sc.z, flags = sc.w & 3;
            __half2 res[NB];
            // every segment of a tile has the same number of 4-column groups: straight-line code over 4 NG registers per band
            if (NB == 1 && flags != 0) {
                // a 32-column strip of two segments longer than 32 frames
                unsigned smid;
                asm("mov.u32 %0, %%smid;" : "=r"(smid));
                __half2* bnd = p.bnd + ((size_t)smid * p.bnd_rows) * kH2DpThreads + threadIdx.x;
                if (flags == kH2Out) h2_tile_strip<8, false, true>(L, lmin, Lm, sc, cur, bnd, res[0]);
                else if (flags == (kH2In | kH2Out)) h2_tile_strip<8, true, true>(L, lmin, Lm, sc, cur, bnd, res[0]);
                else {
                    switch (ng) {
                        case 1: h2_tile_strip<1, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        case 2: h2_tile_strip<2, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        case 3: h2_tile_strip<3, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        case 4: h2_tile_strip<4, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        case 5: h2_tile_strip<5, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        case 6: h2_tile_strip<6, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        case 7: h2_tile_strip<7, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                        default: h2_tile_strip<8, true, false>(L, lmin, Lm, sc, cur, bnd, res[0]); break;
                    }
                }
            } else if constexpr (NB == 1) {
                switch (ng) {
                    case 5: h2_tile<1, 5>(L, lmin, Lm, sc, cur, res); break;
                    case 6: h2_tile<1, 6>(L, lmin, Lm, sc, cur, res); break;
                    case 7: h2_tile<1, 7>(L, lmin, Lm, sc, cur, res); break;
                    default: h2_tile<1, 8>(L, lmin, Lm, sc, cur, res); break;
                }
            } else if constexpr (NB == 2) {
                if (ng == 3) h2_tile<2, 3>(L, lmin, Lm, sc, cur, res);
                else h2_tile<2, 4>(L, lmin, Lm, sc, cur, res);
            } else {
                if (ng == 1) h2_tile<4, 1>(L, lmin, Lm, sc, cur, res);
                else h2_tile<4, 2>(L, lmin, Lm, sc, cur, res);
            }
            if (Lm && !(flags & kH2Out)) {  // (a strip with a successor has no result yet)
#pragma unroll
                for (int b = 0; b < NB; b++) {
#pragma unroll
                    for (int hsel = 0; hsel < 2; hsel++) {
                        const int e = 2 * b + hsel;
                        const int seg = h2_seg_of(sa, sb, e);
                        if (seg >= 0) {
                            const float v = hsel ? __high2float(res[b]) : __low2float(res[b]);
                            // D16 / (S (Lq + Ld)); an overflowed path sum stays +inf and is never inserted
                            // whole length of the segment (a last strip's `columns` field is only its own width)
                            const int whole = NB == 1 ? (e == 0 ? sd.x : sd.y) : h2_len_of(sc, e);
                            // The KEY is a lower bound of the pair's rounded-frame distance, not the raw scan value: the
                            // packed-half roundings can only have inflated D16 by (1 + 2^-11) per cell of the path (header), so
                            // (scan - eta) (1 + 2^-11)^-(Lq + Ld + 2) <= DTW~ / (Lq + Ld) PER PAIR (7.06e-4 > log2(1 + 2^-11), the
                            // excess covers the fp32 roundings of this line). A list's worst key w then bounds every dropped
                            // pair whatever its length (bound_mode 3) - a common factor for the longest segment of the
                            // dictionary would throw away 20 % for 383 frames.
                            const float npath = (float)(Lm + (uint32_t)whole);
                            const float dist = fmaxf(__fdividef(v * p.inv_s, npath) - p.eta, 0.f) * exp2f(-7.06e-4f * (npath + 2.f));
                            tc_insert<KP, kH2DpThreads>(list, worst, dist, (uint32_t)seg);
                            worst = worst < thr0 ? worst : thr0;  // (an insertion reloads `worst` from the list's last place)
                            if constexpr (DBG) p.dbg[(size_t)(g * kTcM + m) * p.dbg_nseg + seg] = dist;
                        }
                    }
                }
            }
        }
        // the two slots' lists of query m (threads m, m + 128) are merged by the slot-0 thread
        asm volatile("bar.sync 1, %0;" ::"n"(kH2DpThreads) : "memory");
        if (slot == 0)
            tc_merge_store<KP, kH2DpThreads, kH2Slots, true>(list, worst, thr0, [&] {
                return TcListDst{p.thr + g * kTcM + m, p.partial + ((size_t)slice * p.ngroups * kTcM + (size_t)g * kTcM + m) * KP};
            });
    }
    tc_cta_exit<NB != 1>(warp == kH2DpWarps, tmem_base);  // the NB = 2 and 4 launches are the dependent ones
}

__global__ void k_h2_nsmid(uint32_t* out) {
    uint32_t n;
    asm("mov.u32 %0, %%nsmid;" : "=r"(n));
    *out = n;
}

// one thread per (tile, TMEM column n): writes row n of the tile's B operand. Slot = n / 64; inside the slot band = column /
// (64 / NB), and inside the band column 2 t + w is frame t of the band's segment w.
__global__ void k_h2_dict_tiles(const double* __restrict__ mfcc, const uint64_t* __restrict__ off, int c, const double* __restrict__ mu,
                                const int4* __restrict__ desc, const uint8_t* __restrict__ tile_nb, uint32_t ntiles, float scale,
                                unsigned char* __restrict__ tiles) {
    const uint32_t t = blockIdx.x, n = threadIdx.x;  // blockDim = 128
    if (t >= ntiles) return;
    const int nb = tile_nb[t];
    const int slot = (int)n / kH2SlotCols, col = (int)n % kH2SlotCols;
    const int band_cols = kH2SlotCols / nb;
    const int e = 2 * (col / band_cols) + (col & 1), j = (col % band_cols) >> 1;
    const int4* dp = desc + ((size_t)t * kH2Slots + slot) * kH2DescInt4;
    const int4 sa = dp[0], sb = dp[1], sc = dp[2];
    const int segs[8] = {sa.x, sa.y, sa.z, sa.w, sb.x, sb.y, sb.z, sb.w};
    const int seg = segs[e];
    const int len = (int)((((e < 4) ? (uint32_t)sc.x : (uint32_t)sc.y) >> (8 * (e & 3))) & 0xFFu);  // columns of this strip
    const int strip = sc.w >> 8;  // the tile covers frames 32 strip .. of its segments
    __align__(16) __half row[kTcK];
#pragma unroll
    for (int k = 0; k < kTcK; k++) row[k] = __float2half_rn(0.f);
    if (seg >= 0 && j < len) {
        const double* src = mfcc + (off[seg] + 32 * strip + j) * c;
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
        row[15] = __float2half_rn(scale);
    }
    unsigned char* base = tiles + (size_t)t * kTcBTileBytes;
    *reinterpret_cast<uint4*>(base + tc_tile_offset<kTcN>((int)n, 0)) = *reinterpret_cast<const uint4*>(&row[0]);
    *reinterpret_cast<uint4*>(base + tc_tile_offset<kTcN>((int)n, 8)) = *reinterpret_cast<const uint4*>(&row[8]);
}

// ---------------------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------------------
// needs dtw_tc_dict_build to have run (mean frame, norm scale, max norms)
int dtw_h2_dict_build(ss_dict* d) {
    ss_ctx* ctx = d->ctx;
    d->h2_ready = false;
    if (!d->tc_stats_ready || d->max_len > (uint32_t)kH2MaxLong) return SS_OK;  // (longer still: dtw.cu's fp32 scan)
    std::vector<uint32_t> order;
    order.reserve(d->nseg);
    for (size_t s = 0; s < d->nseg; s++)
        if (d->h_off[s + 1] > d->h_off[s]) order.push_back((uint32_t)s);
    auto len_of = [&](uint32_t s) { return (int)(d->h_off[s + 1] - d->h_off[s]); };
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return len_of(a) > len_of(b); });
    // Tiles. A segment of <= 32 frames is one column run; all segments of a tile share ng = ceil(len / 4) (and hence the kind
    // NB: ng 5..8 -> 1 band per thread, 3..4 -> 2, 1..2 -> 4); a tile holds 2 slots x 2 NB segments. Element e of a slot =
    // band e / 2, half e % 2; consecutive segments in length order go to the SAME half-pair first, so the two halves of a
    // register carry nearly equal lengths. A LONGER segment is cut into 32-column strips: four segments with the same
    // number of strips and the same ng of their last strip form nstrips consecutive NB = 1 tiles (flags: boundary column
    // in / out), which one CTA processes in order.
    std::vector<int4> desc;
    std::vector<uint8_t> tile_nb;
    d->h_h2_tile_cost.clear();
    d->h_h2_tile_cont.clear();
    d->h2_first_tile[0] = 0;
    d->h2_has_strips = false;
    auto push_tile = [&](int nb, int ng, uint32_t cost, bool cont) {
        tile_nb.push_back((uint8_t)nb);
        d->h_h2_tile_cost.push_back(cost);
        d->h_h2_tile_cont.push_back(cont ? 1 : 0);
        (void)ng;
    };
    int cur_kind = 1;
    for (size_t o = 0; o < order.size();) {
        const int len0 = len_of(order[o]);
        if (len0 > 32) {
            // ---- a quad of long segments: equal strip count, equal ng of the last strip ------------------------------------
            const int nstrips = (len0 + 31) / 32, ngl = ((len0 - 32 * (nstrips - 1)) + 3) >> 2;
            size_t take = 0;
            while (take < 4 && o + take < order.size()) {
                const int l = len_of(order[o + take]);
                if ((l + 31) / 32 != nstrips || (((l - 32 * (nstrips - 1)) + 3) >> 2) != ngl) break;
                take++;
            }
            for (int st = 0; st < nstrips; st++) {
                const bool last = st == nstrips - 1;
                const int flags = (st > 0 ? kH2In : 0) | (!last ? kH2Out : 0);
                for (int slot = 0; slot < kH2Slots; slot++) {
                    int segs[2] = {-1, -1}, whole[2] = {0, 0};
                    uint32_t lens = 0;
                    for (int e = 0; e < 2; e++) {
                        const size_t pos = (size_t)slot * 2 + e;
                        if (pos < take) {
                            const int l = len_of(order[o + pos]);
                            segs[e] = (int)order[o + pos];
                            whole[e] = l;
                            lens |= (uint32_t)(last ? l - 32 * (nstrips - 1) : 32) << (8 * e);
                        }
                    }
                    desc.push_back(make_int4(segs[0], segs[1], -1, -1));
                    desc.push_back(make_int4(-1, -1, -1, -1));
                    desc.push_back(make_int4((int)lens, 0, last ? ngl : 8, flags | (st << 8)));
                    desc.push_back(make_int4(whole[0], whole[1], 0, 0));
                }
                push_tile(1, last ? ngl : 8, 24u + 16u * (uint32_t)(last ? ngl : 8), st > 0);
            }
            d->h2_has_strips = true;
            o += take;
            continue;
        }
        const int ng = (len0 + 3) >> 2;
        const int nb = ng >= 5 ? 1 : (ng >= 3 ? 2 : 4);
        while (cur_kind < nb) {  // kinds in launch order 1, 2, 4
            d->h2_first_tile[cur_kind == 1 ? 1 : 2] = (uint32_t)tile_nb.size();
            cur_kind *= 2;
        }
        const size_t cap = (size_t)kH2Slots * 2 * nb;
        size_t take = 0;
        while (take < cap && o + take < order.size() && ((len_of(order[o + take]) + 3) >> 2) == ng) take++;
        for (int slot = 0; slot < kH2Slots; slot++) {
            int segs[8] = {-1, -1, -1, -1, -1, -1, -1, -1}, whole[4] = {0, 0, 0, 0};
            uint32_t lens[2] = {0, 0};
            for (int e = 0; e < 2 * nb; e++) {
                const size_t pos = (size_t)slot * 2 * nb + e;
                if (pos < take) {
                    segs[e] = (int)order[o + pos];
                    lens[e >> 2] |= (uint32_t)len_of(order[o + pos]) << (8 * (e & 3));
                    if (e < 4) whole[e] = len_of(order[o + pos]);
                }
            }
            desc.push_back(make_int4(segs[0], segs[1], segs[2], segs[3]));
            desc.push_back(make_int4(segs[4], segs[5], segs[6], segs[7]));
            desc.push_back(make_int4((int)lens[0], (int)lens[1], ng, 0));
            desc.push_back(make_int4(whole[0], whole[1], whole[2], whole[3]));
        }
        // cost of one two-row step of the tile, relative: measured per kind with the per-CTA timeline (SS_DTW_H2_TIMELINE,
        // tools/h2_timeline.py): 0.385 / 0.399 / 0.575 us for NB = 1 / 2 / 4 - four short bands cost 1.5 x what the column count says
        push_tile(nb, ng, (24u + 16u * (uint32_t)(nb * ng)) * (nb == 4 ? 3u : 2u) / 2u, false);
        o += take;
    }
    while (cur_kind < 4) {
        d->h2_first_tile[cur_kind == 1 ? 1 : 2] = (uint32_t)tile_nb.size();
        cur_kind *= 2;
    }
    d->h2_first_tile[3] = (uint32_t)tile_nb.size();
    const uint32_t ntiles = (uint32_t)tile_nb.size();
    d->h2_ntiles = ntiles;
    d->h2_slices.clear();
    if (!ntiles) return SS_OK;
    SS_TRY(upload(ctx, d->d_h2_desc, desc.data(), desc.size()));
    DevBuf<uint8_t> d_nb;
    SS_TRY(upload(ctx, d_nb, tile_nb.data(), tile_nb.size()));
    SS_CUDA(ctx, d->d_h2_tiles.reserve((size_t)ntiles * kTcBTileBytes / 2));
    k_h2_dict_tiles<<<ntiles, kTcN, 0, ctx->stream>>>(d->d_mfcc.p, d->d_off.p, d->c, d->d_mu.p, d->d_h2_desc.p, d_nb.p, ntiles, d->tc_nb_scale,
                                                     reinterpret_cast<unsigned char*>(d->d_h2_tiles.p));
    SS_LAUNCHED(ctx);
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // d_nb is released on return
    // cost scale S: S |b|^2_max <= 4096, so that a path of 64 typical cells stays far below 65504 (an overflow is not an error:
    // the pair reads +inf and the bound is capped, see the header); longer paths scale it down further, per query batch
    // (h2_cost_scale: S only enters the query side's A blocks)
    float S = 1.0f;
    while (S * d->tc_max_nb > 4096.f) S *= 0.5f;
    while (S * d->tc_max_nb < 2048.f && S < 64.f) S *= 2.0f;
    d->h2_s0 = S;
    d->h2_s = S;
    d->h2_bmax = d->tc_max_abs;
    {   // the strip kernel's boundary scratch has one area per SM id
        DevBuf<uint32_t> d_n;
        SS_CUDA(ctx, d_n.reserve(1));
        k_h2_nsmid<<<1, 1, 0, ctx->stream>>>(d_n.p);
        SS_LAUNCHED(ctx);
        SS_CUDA(ctx, cudaMemcpyAsync(&d->h2_nsmid, d_n.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    }
    d->h2_ready = true;
    return SS_OK;
}

// S for one (dictionary, query batch): halved for every doubling of the longest possible path (Lq + Ld cells) beyond 64, so that
// path sums of the longest sequences still fit the fp16 range. Sets d->h2_s (what the launch, eta and the bound read).
static void h2_cost_scale(ss_dict* d, const ss_queries* q) {
    float S = d->h2_s0;
    for (uint64_t l = 64; l < (uint64_t)d->max_len + q->max_len && S > 1.0f / 65536.f; l *= 2) S *= 0.5f;
    d->h2_s = S;
}

static int h2_queries_build(ss_dict* d, ss_queries* q) {
    ss_ctx* ctx = q->ctx;
    h2_cost_scale(d, q);
    if (q->h2_built && q->h2_dict_serial == d->tc_serial && q->h2_s_built == d->h2_s) return SS_OK;
    if (!q->tc_grouped) SS_TRY(dtw_tc_queries_group(q));
    SS_CUDA(ctx, q->d_h2_a.reserve(std::max<uint64_t>(q->tc_a_bytes, 16)));
    SS_CUDA(ctx, q->d_tc_slot_max_na.reserve(std::max<size_t>((size_t)q->tc_ngroups * kTcM, 1)));
    SS_CUDA(ctx, q->d_uncert_flag.reserve(std::max<size_t>(q->nq, 1)));
    SS_CUDA(ctx, q->d_tc_max_norm.reserve(1));
    SS_CUDA(ctx, cudaMemsetAsync(q->d_tc_max_norm.p, 0, sizeof(float), ctx->stream));
    if (q->tc_ngroups) {
        SS_CUDA(ctx, cudaMemsetAsync(q->d_tc_slot_max_na.p, 0, (size_t)q->tc_ngroups * kTcM * sizeof(float), ctx->stream));
        k_tc_query_tiles<<<dim3(q->tc_ngroups, q->max_len), kTcM, 0, ctx->stream>>>(q->d_mfcc.p, q->d_off.p, q->c, d->d_mu.p, q->d_tc_group_len.p,
                                                                 q->d_tc_group_off.p, q->d_tc_qid.p, d->tc_nb_scale, d->h2_s, q->d_h2_a.p,
                                                                 q->d_tc_max_norm.p, q->d_tc_slot_max_na.p);
        SS_LAUNCHED(ctx);
    }
    q->h2_built = true;
    q->h2_dict_serial = d->tc_serial;
    q->h2_s_built = d->h2_s;
    return SS_OK;
}

// Candidates kept per query for k <= 2. Measured at config 4 (profiles/bench/r2_h2_kp_sweep.json): 8 leaves 47 of the 10 000
// queries uncertified by the merged list, but the scan itself is 3 ms faster than with 16.
constexpr int kH2Kp = 8;

template <int KP, int NB, bool DBG, bool LONG>
static int h2_launch_kind(ss_ctx* ctx, H2Params p, uint32_t slice_begin, uint32_t nslices, size_t smem, bool dependent) {
    if (!nslices) return SS_OK;
    p.slice_begin = slice_begin;
    p.nslices = nslices;
    // KP = 8 (k <= 2) runs the two-pipeline kernel for NB = 1 and 2. Its 32-entry lists (H2_WIDE, k > 2) would need 128 KB of
    // shared memory, and NB = 4 does not fit its 112 DP registers without spilling: both keep the one-pipeline kernel.
    if constexpr (LONG) return tc_launch_scan(ctx, k_dtw_scan_h2_long<KP, NB, DBG>, p, kH2Threads, smem, dependent);
    else if constexpr (KP == kH2Kp && NB != 4)
        return tc_launch_scan(ctx, k_dtw_scan_h2_2p<KP, NB, DBG>, p, kH2PThreads, tc_smem_bytes(p.max_len, kH2Pipes, KP, kH2PDpThreads), dependent);
    else return tc_launch_scan(ctx, k_dtw_scan_h2<KP, NB, DBG>, p, kH2Threads, smem, dependent);
}

// eta of the bound (true units, per normalised distance): fp16 subnormal roundings of the S-scaled operands and sums
static double h2_eta(const ss_dict* d) { return (13.0 * (double)d->h2_bmax + 4.0) * 5.9604644775390625e-08 /* 2^-24 */ / (double)d->h2_s; }

struct H2Plan {
    H2Params p;
    uint32_t kind_begin[4];  // first slice of each kind (1, 2, 4) and the total
    uint32_t nslots;
    size_t smem;
    bool use_long;  // segments or queries of more than 32 frames: k_dtw_scan_h2_long (strips, streamed A block, deflated keys)
};
constexpr int kH2Waves = 16;  // CTAs per SM over the launches of one scan

static int h2_plan(ss_dict* d, ss_queries* q, int kp, H2Plan* plan) {
    ss_ctx* ctx = d->ctx;
    const uint32_t nslots = q->tc_ngroups * kTcM;
    if (d->h2_slices.size() > 64 && !d->h2_slices.count(q->tc_ngroups)) {  // (many different batch sizes: start over)
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        d->h2_slices.clear();
    }
    std::unique_ptr<ss_dict::H2Slices>& sl = d->h2_slices[q->tc_ngroups];
    if (!sl) {
        sl.reset(new ss_dict::H2Slices());
        // about kH2Waves CTAs per SM, but never slices of fewer than ~12 tiles: a small batch (nq = 1: one group) would
        // otherwise pay a CTA's fixed cost (TMEM allocation, the A-block copy, list merge) two thousand times
        const uint32_t want = std::max<uint32_t>(1, std::min<uint32_t>(((uint32_t)ctx->sm_count * kH2Waves + q->tc_ngroups - 1) / q->tc_ngroups,
                                                                       std::max<uint32_t>((uint32_t)ctx->sm_count, d->h2_ntiles / 12)));
        std::vector<uint32_t> st;
        uint64_t total = 0;
        for (uint32_t f : d->h_h2_tile_cost) total += f;
        const uint64_t per0 = std::max<uint64_t>(1, (total + want - 1) / want);
        // the kind that is launched LAST gets slices of half the cost: the step ends when its slowest CTA does, and the timeline
        // showed 2.7 % of the step's SM-time idle behind the last CTAs (one wave of 158 CTAs of 1.0 - 4.4 ms each at config 4)
        int last_kind = -1, nkinds = 0;
        for (int kind = 0; kind < 3; kind++)
            if (d->h2_first_tile[kind + 1] > d->h2_first_tile[kind]) last_kind = kind, nkinds++;
        if (nkinds < 2) last_kind = -1;  // (a single kind keeps its wave count)
        for (int kind = 0; kind < 3; kind++) {
            sl->kind_slice[kind] = (uint32_t)st.size();
            const uint64_t per = kind == last_kind ? std::max<uint64_t>(1, per0 / 2) : per0;
            uint64_t acc = per;  // forces a slice start at the first tile of the kind
            for (uint32_t t = d->h2_first_tile[kind]; t < d->h2_first_tile[kind + 1]; t++) {
                if (acc >= per && !d->h_h2_tile_cont[t]) st.push_back(t), acc = 0;  // (the strips of a long segment stay in one slice)
                acc += d->h_h2_tile_cost[t];
            }
        }
        sl->kind_slice[3] = (uint32_t)st.size();
        st.push_back(d->h2_ntiles);
        SS_TRY(upload(ctx, sl->d_slice_tile, st.data(), st.size()));
    }
    const uint32_t nslices = sl->kind_slice[3];
    SS_CUDA(ctx, d->d_tc_partial.reserve((size_t)nslices * nslots * kp));
    SS_CUDA(ctx, d->d_cand_idx.reserve((size_t)nslots * kp));
    SS_CUDA(ctx, d->d_cand_adist.reserve((size_t)nslots * kp));
    if (!d->ev_scan0) {
        SS_CUDA(ctx, cudaEventCreate(&d->ev_scan0));
        SS_CUDA(ctx, cudaEventCreate(&d->ev_scan1));
    }
    H2Params& p = plan->p;
    p.a_blocks = q->d_h2_a.p;
    p.group_off = q->d_tc_group_off.p;
    p.group_len = q->d_tc_group_len.p;
    p.slot_len = q->d_tc_slot_len.p;
    p.ngroups = q->tc_ngroups;
    p.tiles = reinterpret_cast<const unsigned char*>(d->d_h2_tiles.p);
    p.desc = d->d_h2_desc.p;
    p.slice_tile = sl->d_slice_tile.p;
    p.nslices = nslices;
    p.slice_begin = 0;
    p.partial = d->d_tc_partial.p;
    p.max_len = q->max_len;
    p.inv_s = 1.0f / d->h2_s;
    SS_CUDA(ctx, d->d_h2_thr.reserve(std::max<uint32_t>(nslots, 1)));
    SS_CUDA(ctx, cudaMemsetAsync(d->d_h2_thr.p, 0xFF, (size_t)nslots * sizeof(unsigned long long), ctx->stream));
    p.thr = d->d_h2_thr.p;
    p.dbg = nullptr;
    p.dbg_nseg = 0;
    for (int i = 0; i < 4; i++) plan->kind_begin[i] = sl->kind_slice[i];
    plan->nslots = nslots;
    plan->use_long = d->h2_has_strips || q->max_len > (uint32_t)kTcMaxLen;
    p.bnd = nullptr;
    p.bnd_rows = 0;
    p.eta = 0.f;
    p.timeline = nullptr;
    if (plan->use_long) {
        if (d->h2_has_strips) {
            p.bnd_rows = (q->max_len + 1) & ~1u;
            SS_CUDA(ctx, d->d_h2_bnd.reserve((size_t)d->h2_nsmid * p.bnd_rows * kH2DpThreads));
            p.bnd = d->d_h2_bnd.p;
        }
        p.eta = (float)h2_eta(d) * 1.0001f;
        plan->smem = tc_smem_bytes(kH2ARing, 1, kp, kH2DpThreads);
    } else {
        plan->smem = tc_smem_bytes(q->max_len, 1, kp, kH2DpThreads);
    }
    return SS_OK;
}

template <int KP, bool DBG, bool LONG>
static int h2_launch_kinds(ss_ctx* ctx, const H2Plan& plan) {
    bool dep = false;
    const uint32_t* kb = plan.kind_begin;
    SS_TRY((h2_launch_kind<KP, 1, DBG, LONG>(ctx, plan.p, kb[0], kb[1] - kb[0], plan.smem, dep)));
    dep = dep || kb[1] > kb[0];
    SS_TRY((h2_launch_kind<KP, 2, DBG, LONG>(ctx, plan.p, kb[1], kb[2] - kb[1], plan.smem, dep)));
    dep = dep || kb[2] > kb[1];
    SS_TRY((h2_launch_kind<KP, 4, DBG, LONG>(ctx, plan.p, kb[2], kb[3] - kb[2], plan.smem, dep)));
    return SS_OK;
}
template <int KP, bool DBG>
static int h2_launch_all(ss_ctx* ctx, const H2Plan& plan) {
    return plan.use_long ? h2_launch_kinds<KP, DBG, true>(ctx, plan) : h2_launch_kinds<KP, DBG, false>(ctx, plan);
}

// the packed-half scan takes segments and queries of at most kH2MaxLong frames
bool dtw_h2_applies(const ss_dict* d, const ss_queries* q) {
    return d->h2_ready && q->max_len <= (uint32_t)kH2MaxLong && q->total_frames > 0;
}

// The scan of batch q (dtw_h2_applies), its f64 refine and certification. wide: 32 candidates per query whatever k (the re-run
// of queries an earlier pass could not certify); second_chance: refine the union of the per-slice lists for the queries the
// merged list leaves uncertified.
int dtw_h2_match_dev(ss_dict* d, ss_queries* q, int k, bool wide, bool second_chance, bool timed, uint32_t* d_out_idx, double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    TraceTimer tt(ctx);
    SS_TRY(h2_queries_build(d, q));
    tt.lap("  h2: query A blocks");
    // k > 2: the k-th and the kp-th neighbour must be further apart than the filter's ~4 % margin: a longer list
    const int kp = wide || k > 2 ? 32 : kH2Kp;
    H2Plan plan;
    SS_TRY(h2_plan(d, q, kp, &plan));
    tt.lap("  h2: plan (slices, workspaces)");
    const char* timeline = timed && !plan.use_long ? getenv("SS_DTW_H2_TIMELINE") : nullptr;  // (set and unset between matches)
    if (timeline) {
        const size_t n = (size_t)plan.p.ngroups * plan.p.nslices * 8;
        SS_CUDA(ctx, d->d_h2_timeline.reserve(n));
        SS_CUDA(ctx, cudaMemsetAsync(d->d_h2_timeline.p, 0, n * sizeof(unsigned long long), ctx->stream));
        plan.p.timeline = d->d_h2_timeline.p;
    }
    if (timed) SS_CUDA(ctx, cudaEventRecord(d->ev_scan0, ctx->stream));
    if (kp == kH2Kp) SS_TRY((h2_launch_all<kH2Kp, false>(ctx, plan)));
    else SS_TRY((h2_launch_all<32, false>(ctx, plan)));
    if (timed) {
        SS_CUDA(ctx, cudaEventRecord(d->ev_scan1, ctx->stream));
        d->scan_timed = true;
    }
    if (kp == kH2Kp) k_tc_merge<kH2Kp><<<ceil_div(plan.nslots, 8), 256, 0, ctx->stream>>>(d->d_tc_partial.p, plan.p.nslices, plan.nslots, d->d_cand_idx.p, d->d_cand_adist.p);
    else k_tc_merge<32><<<ceil_div(plan.nslots, 8), 256, 0, ctx->stream>>>(d->d_tc_partial.p, plan.p.nslices, plan.nslots, d->d_cand_idx.p, d->d_cand_adist.p);
    SS_LAUNCHED(ctx);
    tt.lap("  h2: scan + merge");
    if (timeline) {  // SS_DTW_H2_TIMELINE: one line per CTA (measurement only; synchronises)
        const size_t n = (size_t)plan.p.ngroups * plan.p.nslices;
        std::vector<unsigned long long> h(n * 8);
        SS_CUDA(ctx, cudaMemcpyAsync(h.data(), plan.p.timeline, n * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        if (FILE* f = fopen(timeline, "w")) {
            fprintf(f, "# cta start_ns setup_ns dp_done_ns end_ns smid kind group L ntiles dp_cycles half_ns\n");
            for (size_t i = 0; i < n; i++)
                fprintf(f, "%zu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu %llu\n", i, h[i * 8], h[i * 8 + 1], h[i * 8 + 2], h[i * 8 + 3],
                        h[i * 8 + 4] & 0xFFFFull, (h[i * 8 + 4] >> 16) & 0xFFFFull, h[i * 8 + 4] >> 32, h[i * 8 + 7] >> 32, h[i * 8 + 7] & 0xFFFFFFFFull,
                        h[i * 8 + 5], h[i * 8 + 6]);
            fclose(f);
        }
    }
    // bound_mode 2: eps carries eta; the cap (an overflowed path reads +inf) is 60000 / (S (Lq + 32)), passed as the scale 1 / S.
    // bound_mode 3 (strip kernel): the keys are per-pair lower bounds already; eta and the longest segment go into the cap.
    d->h2_bound_inv_s = 1.0 / (double)d->h2_s;
    SS_TRY(dtw_rescore_finalize(d, q, k, kp, plan.nslots, q->d_tc_qid.p, h2_eta(d), q->d_tc_max_norm.p, d->d_tc_max_norm.p, q->d_tc_slot_max_na.p,
                                plan.use_long ? 3 : 2, q->d_uncert_flag.p, d_out_idx, d_out_dist));
    tt.lap("  h2: f64 refine + certification");
    // the queries the merged list could not certify: refine what the union of the per-slice lists still holds below the scan's
    // own insertion threshold, and certify against that threshold (exact.cu, k_dtw_second_chance)
    if (second_chance) {
        SS_TRY(dtw_second_chance(d, q, k, kp, plan.nslots, q->d_tc_qid.p, d->d_tc_partial.p, plan.p.nslices, d->d_h2_thr.p, h2_eta(d), q->d_tc_max_norm.p,
                                 d->d_tc_max_norm.p, q->d_tc_slot_max_na.p, plan.use_long ? 3 : 2, q->d_uncert_flag.p, d_out_idx, d_out_dist));
        tt.lap("  h2: second chance (union of the slice lists)");
    }
    return SS_OK;
}

// ss_dict_debug_tc_scan's half-precision counterpart: the raw scan distance of every pair (see dtw_tc_debug_scan)
int dtw_h2_debug_scan(ss_dict* d, ss_queries* q, float* d_out, std::vector<uint32_t>* slot_qid, double* mu16, float* scale, float* s_out) {
    ss_ctx* ctx = d->ctx;
    if (!dtw_h2_applies(d, q))
        return set_error(ctx, SS_ERR_INVALID, "debug_h2_scan: the packed-half scan does not apply (segments / queries > %d frames, or no frame)", kH2MaxLong);
    SS_TRY(h2_queries_build(d, q));
    H2Plan plan;
    SS_TRY(h2_plan(d, q, 8, &plan));
    plan.p.dbg = d_out;
    plan.p.dbg_nseg = (uint32_t)d->nseg;
    SS_TRY((h2_launch_all<8, true>(ctx, plan)));
    slot_qid->resize(plan.nslots);
    SS_CUDA(ctx, cudaMemcpyAsync(slot_qid->data(), q->d_tc_qid.p, plan.nslots * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaMemcpyAsync(mu16, d->d_mu.p, 16 * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    *scale = d->tc_nb_scale;
    *s_out = d->h2_s;
    return SS_OK;
}

}  // namespace ss
