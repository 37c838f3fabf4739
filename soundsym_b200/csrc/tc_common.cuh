// tc_common.cuh — what the two tensor-core DTW scans (dtw_tc.cu: fp32 DP, dtw_h2.cu: packed-half DP) share: tile geometry,
// the PTX wrappers (mbarrier, bulk TMA, tcgen05.mma / commit / fences, UMMA descriptors), the packed candidate keys and the
// consumer-side cursor over the double-buffered TMEM accumulators.
#pragma once
#include <cuda_fp16.h>

#include "match.cuh"

namespace ss {

constexpr int kTcM = 128;          // queries per CTA = MMA M = TMEM lanes
constexpr int kTcSlots = 4;        // slots per tile (32 columns each) = DP warps per TMEM lane quadrant
constexpr int kTcN = kTcSlots * 32;  // 128 columns per tile = MMA N
constexpr int kTcK = 16;           // fp16 elements per row = one MMA K step
constexpr int kTcATileBytes = kTcM * kTcK * 2;  // 4096: one query row of the CTA's 128 queries
constexpr int kTcBTileBytes = kTcN * kTcK * 2;  // 4096: one dictionary tile
constexpr int kTcStages = 4;       // B-tile ring
constexpr int kTcBufCols = 2 * kTcN;  // one pipeline step = two rows of the tile = 256 TMEM columns; two buffers = all 512
constexpr int kTcMaxLen = 32;
constexpr int kTcGroupMaxLen = 2048;  // longest query the length-sorted groups of 128 are built for (dtw_h2.cu's strip kernel)
constexpr int kTcPairCol = 16;     // segments of <= 16 frames share a slot two by two: the second one's columns start here
constexpr int kTcDpWarps = 4 * kTcSlots;             // 16; warp w: TMEM lane quadrant w % 4, slot w / 4
// The producer warp sits in a warpgroup of its own (three idle warps) that hands its registers to the DP warpgroups
// (setmaxnreg): 640 threads, 96 registers at launch, DP 112 / producer group 32 = the whole pool. 112 is why the DP step
// pulls its costs from TMEM in 16-column chunks (kTcChunked).
constexpr int kTcRegsDp = 112, kTcRegsProd = 32;
constexpr bool kTcChunked = true;
constexpr int kTcThreads = (kTcDpWarps + 4) * 32;    // 640
constexpr int kTcDpThreads = kTcDpWarps * 32;

// byte offset of element (row, k) inside a ROWS x 16 fp16 K-major no-swizzle UMMA tile: core matrix = 8 rows x 16 B;
// SBO (between 8-row groups) = 128 B, LBO (between the two K chunks) = ROWS / 8 * 128 B
template <int ROWS>
__host__ __device__ __forceinline__ int tc_tile_offset(int row, int k) {
    return ((k >> 3) * (ROWS / 8) + (row >> 3)) * 128 + (row & 7) * 16 + (k & 7) * 2;
}

// ---------------------------------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t s32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mb_init(uint64_t* bar, unsigned count) { asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(s32(bar)), "r"(count)); }
__device__ __forceinline__ void mb_expect_tx(uint64_t* bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(s32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mb_arrive(uint64_t* bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(s32(bar)) : "memory"); }
// blocking wait: try_wait suspends the thread in hardware (up to the hint) instead of hot-spinning, and a failed
// probe backs off with nanosleep — a spinning high-id warp otherwise starves the DP warps that share its scheduler
// (measured: 33 issued instructions per cell with a plain try_wait loop).
__device__ __forceinline__ void mb_wait(uint64_t* bar, unsigned parity) {
    const uint32_t addr = s32(bar);
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(addr), "r"(parity), "r"(20000u)
            : "memory");
        if (done) break;
        __nanosleep(32);
    }
}
// DP-warp side of the TMEM hand-off, by shared-memory address. The wait is the bare try_wait loop (the instruction itself
// suspends the thread up to the hint); the arrive is issued by one elected lane once the whole warp has reached it.
__device__ __forceinline__ void mb_wait_addr(uint32_t addr, unsigned parity) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "TC_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n"
        "@p bra TC_DONE;\n"
        "bra TC_WAIT;\n"
        "TC_DONE:\n"
        "}\n" ::"r"(addr),
        "r"(parity), "r"(20000u)
        : "memory");
}
__device__ __forceinline__ void mb_arrive_elect(uint32_t addr) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "elect.sync _|p, 0xffffffff;\n"
        "@p mbarrier.arrive.shared::cta.b64 _, [%0];\n"
        "}\n" ::"r"(addr)
        : "memory");
}
__device__ __forceinline__ void tma_g2s(void* dst, const void* src, unsigned bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(s32(dst)), "l"(src),
                 "r"(bytes), "r"(s32(bar))
                 : "memory");
}
// the same primitives by 32-bit shared address (the producer lane keeps no generic pointers)
__device__ __forceinline__ void mbs_expect_tx(uint32_t bar, unsigned bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbs_wait_sleep(uint32_t bar, unsigned parity) {
    for (;;) {
        uint32_t done;
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n"
            "selp.u32 %0, 1, 0, p;\n"
            "}\n"
            : "=r"(done)
            : "r"(bar), "r"(parity), "r"(20000u)
            : "memory");
        if (done) break;
        __nanosleep(32);
    }
}
__device__ __forceinline__ void tmas_g2s(uint32_t dst, const void* src, unsigned bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src), "r"(bytes),
                 "r"(bar)
                 : "memory");
}
__device__ __forceinline__ void tcs_commit(uint32_t bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(s32(bar)) : "memory");
}
// D[tmem] = A[smem] * B[smem]^T (overwrite), kind::f16, fp32 accumulate
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(0u)
        : "memory");
}
template <int ROWS>
__device__ __forceinline__ uint64_t tc_smem_desc(const void* p) {
    // start >> 4 | LBO >> 4 << 16 | SBO (128 B) >> 4 << 32 | version 1 << 46 | SWIZZLE_NONE
    return (uint64_t)((s32(p) & 0x3FFFF) >> 4) | ((uint64_t)((ROWS / 8 * 128) >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | (1ull << 46);
}
template <int ROWS>
__device__ __forceinline__ uint64_t tc_smem_desc_s(uint32_t saddr) {
    return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)((ROWS / 8 * 128) >> 4) << 16) | ((uint64_t)(128 >> 4) << 32) | (1ull << 46);
}
__device__ __forceinline__ void tc_ld32(uint32_t taddr, float* v) {
    uint32_t r[32];
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, "
        "%20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]),
          "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
          "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]),
          "=r"(r[31])
        : "r"(taddr));
#pragma unroll
    for (int i = 0; i < 32; i++) v[i] = __uint_as_float(r[i]);
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float tc_min3(float a, float b, float c) {
    float d;
    asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// per-thread candidate list kept in shared memory as packed (ord(dist) << 32 | idx) keys, ascending; only the worst kept
// key lives in a register for the per-pair test, so the hot loop pays two registers for the list
// (STRIDE = number of DP threads of the kernel: entry s of a thread's list sits at list[s * STRIDE])
template <int KP, int STRIDE = kTcDpThreads>
__device__ __forceinline__ void tc_insert_key(unsigned long long* list, unsigned long long& worst, unsigned long long key) {
    int s = KP - 1;
    while (s > 0 && list[(s - 1) * STRIDE] > key) {
        list[s * STRIDE] = list[(s - 1) * STRIDE];
        s--;
    }
    list[s * STRIDE] = key;
    worst = list[(KP - 1) * STRIDE];
}
// unsorted lists (dtw_h2.cu): the largest key of a full list and its place - KP independent loads, no data-dependent loop
template <int KP, int STRIDE = kTcDpThreads>
__device__ __forceinline__ void tc_list_max(const unsigned long long* list, unsigned long long& mx, int& pos) {
    unsigned long long m = list[0];
    int p = 0;
#pragma unroll
    for (int s = 1; s < KP; s++) {
        const unsigned long long v = list[s * STRIDE];
        p = v > m ? s : p;
        m = v > m ? v : m;
    }
    mx = m, pos = p;
}
// ascending insertion sort of the first n places of a list that was filled in no particular order
template <int KP, int STRIDE = kTcDpThreads>
__device__ __forceinline__ void tc_sort_list(unsigned long long* list, int n) {
    for (int i = 1; i < n; i++) {
        const unsigned long long key = list[i * STRIDE];
        int s = i;
        while (s > 0 && list[(s - 1) * STRIDE] > key) {
            list[s * STRIDE] = list[(s - 1) * STRIDE];
            s--;
        }
        list[s * STRIDE] = key;
    }
}
template <int KP, int STRIDE = kTcDpThreads>
__device__ __forceinline__ void tc_insert(unsigned long long* list, unsigned long long& worst, float dist, uint32_t idx) {
    const unsigned long long key = ((unsigned long long)f2ord(dist) << 32) | idx;
    if (key < worst && dist == dist) tc_insert_key<KP, STRIDE>(list, worst, key);
}

// consumer side of the TMEM double buffer: the address of the next buffer's "full" barrier (its "empty" barrier sits 16
// bytes above), the parity to wait for, and this thread's TMEM address in that buffer. The two barriers / buffers are
// flipped by subtracting from their sum.
struct TcCursor {
    uint32_t buf, par, full, taddr, full_sum, taddr_sum;
    __device__ __forceinline__ void init(uint32_t full0, uint32_t lane_addr) {
        buf = 0, par = 0, full = full0, taddr = lane_addr;
        full_sum = 2 * full0 + 8, taddr_sum = 2 * lane_addr + (uint32_t)kTcBufCols;
    }
    __device__ __forceinline__ void wait() const {
        mb_wait_addr(full, par);
        tc_fence_after();
    }
    // the step's costs are in registers: hand the TMEM buffer back and move to the other one
    __device__ __forceinline__ void release() {
        tc_fence_before();
        mb_arrive_elect(full + 16);
        par ^= buf;
        buf ^= 1u;
        full = full_sum - full;
        taddr = taddr_sum - taddr;
    }
};

// one thread per (group g = blockIdx.x, row i = blockIdx.y, query m): A_i[m, :] = [-2 (a_i - mu) (13), s, s, rd(|a_i|^2 / s)],
// written as the two 16-byte K chunks of row m (K-major core matrices). slot_max_na (per query: max |a_i|^2 over its rows)
// and max_norm[0] must be zeroed before the launch. A query that leaves the fp16 range (a coefficient beyond +-3e4 after
// centring, or |a_i|^2 / s beyond 60000: far louder than the dictionary) is clamped and gets slot_max_na = +inf: its scan
// result is then never certified (scan_lower_bound = -inf) and the fp32 scan re-runs it - no host decision needed.
static __global__ void k_tc_query_tiles(const double* __restrict__ mfcc, const uint64_t* __restrict__ off, int c, const double* __restrict__ mu,
                                 const uint32_t* __restrict__ group_len, const uint64_t* __restrict__ group_off,
                                 const uint32_t* __restrict__ qid, float scale, float ascale, unsigned char* __restrict__ a_blocks,
                                 float* __restrict__ max_norm, float* __restrict__ slot_max_na) {
    // ascale: a power of two multiplied into every A entry (1 for the fp32-DP scan; the packed-half scan's cost scale S)
    const uint32_t g = blockIdx.x, i = blockIdx.y, m = threadIdx.x;  // blockDim = 128
    const uint32_t L = group_len[g] & 0xFFFFu;                        // longest query of the group; shorter ones are zero-padded
    if (i >= L) return;
    const uint32_t id = qid[g * kTcM + m];
    const uint32_t Lm = id != 0xFFFFFFFFu ? (uint32_t)(off[id + 1] - off[id]) : 0u;
    unsigned char* blk = a_blocks + group_off[g];
    const float inv_scale = 1.0f / scale;  // power of two: exact
    __align__(16) __half row[kTcK];
#pragma unroll
    for (int k = 0; k < kTcK; k++) row[k] = __float2half_rn(0.f);
    float nrm = 0.f;
    if (i < Lm) {
        const double* src = mfcc + (off[id] + i) * c;
        bool clamped = false;
        for (int k = 0; k < c; k++) {
            float x = (float)(src[k] - mu[k]);
            if (!(fabsf(x) <= 3.0e4f)) x = x > 0.f ? 3.0e4f : (x < 0.f ? -3.0e4f : 0.f), clamped = true;  // also catches NaN
            const __half h = __float2half_rn(x);
            const float v = __half2float(h);
            nrm += v * v;
            row[k] = __float2half_rn(-2.f * v * ascale);  // exact (short of fp16 subnormals, which the bound's eta covers)
        }
        row[13] = __float2half_rn(scale * ascale);
        row[14] = __float2half_rn(scale * ascale);
        // |a_i|^2 rides in the spare K slot, rounded DOWN: the scan cost never exceeds the cost of the rounded frames
        if (!(nrm * inv_scale <= 60000.f)) clamped = true;
        row[15] = __float2half_rn(__half2float(__float2half_rd(fminf(nrm * inv_scale, 60000.f))) * ascale);  // rd first, then the exact scaling
        if (clamped) nrm = __int_as_float(0x7f800000);
    }
    unsigned char* base = blk + (size_t)i * kTcATileBytes;
    *reinterpret_cast<uint4*>(base + tc_tile_offset<kTcM>((int)m, 0)) = *reinterpret_cast<const uint4*>(&row[0]);
    *reinterpret_cast<uint4*>(base + tc_tile_offset<kTcM>((int)m, 8)) = *reinterpret_cast<const uint4*>(&row[8]);
    if (i < Lm) atomicMax(reinterpret_cast<unsigned*>(slot_max_na + g * kTcM + m), __float_as_uint(nrm));  // nrm >= 0 (or +inf)
    float mx = nrm < __int_as_float(0x7f800000) ? nrm : 0.f;
    for (int o = 16; o; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    if ((m & 31) == 0) atomicMax(reinterpret_cast<unsigned*>(max_norm), __float_as_uint(mx));
}

// per query slot: merge the per-slice candidate lists (each ascending) by packed (ord(dist), idx) key. One WARP per slot:
// lane l folds lists l, l + 32, .. into its own ascending top-KP (normally one list per lane: a 64-byte load), then KP
// rounds of "smallest head over the warp" (two redux.sync) pop the merged list, lane r keeping output r.
template <int KP>
__global__ void __launch_bounds__(256) k_tc_merge(const unsigned long long* __restrict__ partial, uint32_t nlists, uint32_t nslots,
                                                  uint32_t* __restrict__ cand_idx, float* __restrict__ cand_adist) {
    const uint32_t slot = blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (slot >= nslots) return;
    unsigned long long best[KP];
#pragma unroll
    for (int s = 0; s < KP; s++) best[s] = kEmptyKey;
    for (uint32_t l = lane; l < nlists; l += 32) {
        const ulonglong2* src = reinterpret_cast<const ulonglong2*>(partial + ((size_t)l * nslots + slot) * KP);
        unsigned long long key[KP];
#pragma unroll
        for (int s = 0; s < KP; s += 2) {
            const ulonglong2 v = __ldg(src + s / 2);
            key[s] = v.x, key[s + 1] = v.y;
        }
        if (l < 32) {
#pragma unroll
            for (int s = 0; s < KP; s++) best[s] = key[s];
        } else {
#pragma unroll
            for (int s = 0; s < KP; s++) {
                if (key[s] < best[KP - 1]) {
                    best[KP - 1] = key[s];
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
    }
    unsigned long long mine = kEmptyKey;
#pragma unroll
    for (int r = 0; r < KP; r++) {
        const uint32_t hi = (uint32_t)(best[0] >> 32), lo = (uint32_t)best[0];
        const uint32_t mhi = __reduce_min_sync(0xffffffffu, hi);
        const uint32_t mlo = __reduce_min_sync(0xffffffffu, hi == mhi ? lo : 0xFFFFFFFFu);
        const unsigned long long m = ((unsigned long long)mhi << 32) | mlo;
        if (best[0] == m && m != kEmptyKey) {  // keys are unique (a segment sits in exactly one slice): one lane pops
#pragma unroll
            for (int s = 0; s + 1 < KP; s++) best[s] = best[s + 1];
            best[KP - 1] = kEmptyKey;
        }
        if (lane == r) mine = m;
    }
    if (lane < KP) {
        const bool empty = mine == kEmptyKey;
        cand_idx[(size_t)slot * KP + lane] = empty ? 0xFFFFFFFFu : (uint32_t)mine;
        const float dist = key_dist(mine);
        cand_adist[(size_t)slot * KP + lane] = empty ? __int_as_float(0x7f800000) : dist;
    }
}

}  // namespace ss
