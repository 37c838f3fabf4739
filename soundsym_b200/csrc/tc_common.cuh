// tc_common.cuh — what the two tensor-core DTW scans (dtw_tc.cu: fp32 DP, dtw_h2.cu: packed-half DP) share: tile geometry,
// the PTX wrappers (mbarrier, bulk TMA, tcgen05.mma / commit / fences, UMMA descriptors), the packed candidate keys, and the
// pieces every scan kernel is built from: the DP band recurrence over float or __half2 (tc_band, tc_band_row), the consumer-side
// cursor over the double-buffered TMEM accumulators and the step driver of a tile's capture-free steps (TcCursor, tc_steps), the
// CTA skeleton (tc_tmem_alloc, tc_cta_exit), the producer lane (tc_produce), the merge and write of a query's slot lists
// (tc_merge_store), and on the host the launch (tc_launch_scan) and the shared-memory size (tc_smem_bytes).
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
// instruction descriptors of the scans' MMA: f16 x f16, K-major both, N = 128, M = 128, into an fp32 (c_format = 1) or an
// F16 (c_format = 0) accumulator
constexpr uint32_t kTcIdescF32 = (1u << 4) | ((uint32_t)(kTcN >> 3) << 17) | ((uint32_t)(kTcM >> 4) << 24);
constexpr uint32_t kTcIdescF16 = (0u << 4) | ((uint32_t)(kTcN >> 3) << 17) | ((uint32_t)(kTcM >> 4) << 24);

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
__device__ __forceinline__ __half2 tc_min3(__half2 a, __half2 b, __half2 c) { return __hmin2(__hmin2(a, b), c); }  // one VHMNMX
__device__ __forceinline__ float tc_add(float a, float b) { return a + b; }
__device__ __forceinline__ __half2 tc_add(__half2 a, __half2 b) { return __hadd2(a, b); }

// ---------------------------------------------------------------------------------------------------------------
// the DP band, over float (dtw_tc.cu) or __half2 (dtw_h2.cu: two segments per register)
// ---------------------------------------------------------------------------------------------------------------
// what a band carries from column j-1 to column j: D(i, j-1), D(i-1, j-1), D(i+1, j-1)
template <class T>
struct TcCarry {
    T left0, diag0, left1;
};
// TWO rows (i, i+1) of a band over columns [J0, J1), row state updated in place: cell (i, j) reads d[j] (row i-1) and feeds
// cell (i+1, j), which overwrites d[j]. Two independent dependency chains per thread, no register copies, no guards: per cell
// one three-input min and one add. tm0 / tm1 hold the costs of columns J0 .. J1 - 1 of the two rows. The carries come in and
// go out through c, so a band split into column chunks (or a strip of a longer band) does the same operations in the same
// order as the whole band. c0l receives row i's values of the last 4-column group (row i+1's are d[4 NG - 4 ..]): the
// column len - 1 lies in that group, and the caller picks D(i, len-1) / D(i+1, len-1) from them in the steps where a query
// can end.
template <int NG, int J0, int J1, class T>
__device__ __forceinline__ void tc_band(const T* tm0, const T* tm1, T (&d)[4 * NG], TcCarry<T>& c, T (&c0l)[4]) {
#pragma unroll
    for (int j = J0; j < J1; j++) {
        const T up0 = d[j];
        const T c0 = tc_add(tm0[j - J0], tc_min3(c.left0, up0, c.diag0));
        const T c1 = tc_add(tm1[j - J0], tc_min3(c.left1, c0, c.left0));  // up = D(i, j), diag = D(i, j-1)
        c.diag0 = up0;
        c.left0 = c0;
        c.left1 = c1;
        d[j] = c1;
        if (j >= 4 * (NG - 1)) c0l[j - 4 * (NG - 1)] = c0;
    }
}
// a single row of a band, in place (the odd last row of a tile): carries D(i, -1) = left, D(i-1, -1) = diag in; returns the
// row's last column, the left carry of whatever follows
template <int NG, class T>
__device__ __forceinline__ T tc_band_row(const T* tm, T (&d)[4 * NG], T left, T diag) {
#pragma unroll
    for (int j = 0; j < 4 * NG; j++) {
        const T up = d[j];
        const T cur = tc_add(tm[j], tc_min3(left, up, diag));
        diag = up;
        left = cur;
        d[j] = cur;
    }
    return left;
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

// Steps [0, ncap) of a tile on the double-buffered cursor, the ones in which no query of the group ends. They run two per
// iteration on buffer 0 then buffer 1, from cursors rebuilt out of loop invariants - barrier and TMEM addresses are then
// constants of the loop and only the parity flips (once per pair) - after one plain step if the tile happens to start on
// buffer 1. step(cursor, dinit) is one pipeline step; dinit = D(i-1, -1) of its first row: the caller's value for the tile's
// first step (the virtual D(-1, -1) = 0), inf after; dinit is left at inf once a step has run. Returns the next step (ncap).
template <class T, class Step>
__device__ __forceinline__ uint32_t tc_steps(TcCursor& cur, uint32_t ncap, T& dinit, T inf, Step step) {
    uint32_t st = 0;
    if (st < ncap && cur.buf) {
        step(cur, dinit);
        dinit = inf;
        st++;
    }
    if (st + 2 <= ncap) {
        const uint32_t full0 = cur.full, taddr0 = cur.taddr;
        uint32_t par = cur.par;
#pragma unroll 1
        for (; st + 2 <= ncap; st += 2) {
            TcCursor c0 = {0u, par, full0, taddr0, cur.full_sum, cur.taddr_sum};
            step(c0, dinit);
            TcCursor c1 = {1u, par, full0 + 8u, taddr0 + (uint32_t)kTcBufCols, cur.full_sum, cur.taddr_sum};
            step(c1, inf);
            dinit = inf;
            par ^= 1u;
        }
        cur.par = par;
    }
    if (st < ncap) {
        step(cur, dinit);
        dinit = inf;
        st++;
    }
    return st;
}

// ---------------------------------------------------------------------------------------------------------------
// CTA skeleton of the scan kernels
// ---------------------------------------------------------------------------------------------------------------
// all 512 TMEM columns, allocated by the warp alloc_warp into *slot; every thread returns with their base address (the
// mbarriers must be initialised before: the __syncthreads here publishes them too)
__device__ __forceinline__ uint32_t tc_tmem_alloc(bool alloc_warp, uint32_t* slot) {
    if (alloc_warp) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(s32(slot)), "r"(512u) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    return *slot;
}
// the CTA's way out: the allocating warp hands TMEM back once every thread is done with it. DEPENDENT: the launch may have
// started early (programmatic dependent launch) and may finish its own work before the launch ahead of it has: it must not
// be seen as complete (the merge kernel is ordered after THIS grid) until that one is, so every CTA waits for it on the
// way out. By then all of the earlier grid's CTAs are at least resident, so nothing is held up.
template <bool DEPENDENT>
__device__ __forceinline__ void tc_cta_exit(bool alloc_warp, uint32_t tmem_base) {
    if constexpr (DEPENDENT) asm volatile("griddepcontrol.wait;" ::: "memory");
    tc_fence_before();
    __syncthreads();
    if (alloc_warp) {
        tc_fence_after();
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512u) : "memory");
    }
}

// The producer lane of pipeline `pipe` of a scan CTA: bulk-TMA copies and MMA issue. It lives in kTcRegsProd registers, so it
// keeps 32-bit shared addresses and running counters only. Pipeline 0's producer copies the group's A block (L rows) into
// sA_s; every producer waits for it. The ntiles B tiles t0 + pipe, t0 + pipe + PIPES, .. stream through the pipeline's ring of
// kTcStages tiles (the rings from sB_s on, one per pipeline; per pipeline b_full[kTcStages], b_empty[kTcStages] barriers from
// b_full_s on); per tile, one step per two query rows: two MMAs and one commit to the step's t_full barrier (t_empty 16
// bytes above; one per pipeline from t_full_s on). PIPES = 1: the steps alternate between the TMEM buffers tmem_base and
// tmem_base + kTcBufCols; PIPES = 2: every step goes to the pipeline's one buffer, tmem_base + pipe kTcBufCols.
template <int PIPES, class Params>
__device__ __forceinline__ void tc_produce(const Params& p, uint32_t g, uint32_t L, uint32_t t0, uint32_t ntiles, uint32_t pipe, uint32_t idesc,
                                           uint32_t sA_s, uint32_t sB_s, uint32_t a_full_s, uint32_t b_full_s, uint32_t t_full_s, uint32_t tmem_base) {
    constexpr uint32_t kBufs = PIPES == 1 ? 2 : 1;  // TMEM buffers the steps go round
    constexpr size_t kStride = (size_t)PIPES * kTcBTileBytes;  // from one of this producer's tiles to the next
    sB_s += pipe * (kTcStages * kTcBTileBytes);
    b_full_s += pipe * (16 * kTcStages);
    t_full_s += 8 * pipe;
    const uint32_t b_empty_s = b_full_s + 8 * kTcStages, t_empty_s = t_full_s + 16;
    if (pipe == 0) {
        mbs_expect_tx(a_full_s, L * kTcATileBytes);
        tmas_g2s(sA_s, p.a_blocks + p.group_off[g], L * kTcATileBytes, a_full_s);
    }
    const unsigned char* tile_src = p.tiles + (size_t)(t0 + pipe) * kTcBTileBytes;
    for (uint32_t n = 0; n < ntiles && n < (uint32_t)kTcStages; n++) {
        mbs_expect_tx(b_full_s + 8 * n, kTcBTileBytes);
        tmas_g2s(sB_s + n * kTcBTileBytes, tile_src + n * kStride, kTcBTileBytes, b_full_s + 8 * n);
    }
    tile_src += kTcStages * kStride;  // the next tile to fetch
    mbs_wait_sleep(a_full_s, 0);
    const uint64_t adesc0 = tc_smem_desc_s<kTcM>(sA_s);
    const uint32_t tm = tmem_base + pipe * kTcBufCols;
    uint32_t cnt = 0, stage = 0, sphase = 0;
    for (uint32_t n = 0; n < ntiles; n++) {
        mbs_wait_sleep(b_full_s + 8 * stage, sphase);
        const uint64_t bdesc = tc_smem_desc_s<kTcN>(sB_s + stage * kTcBTileBytes);
        uint64_t adesc = adesc0;  // advances by one A tile (4 KB = 256 descriptor units) per row
        for (uint32_t row = 0; row < L; row += 2, cnt++) {
            const uint32_t buf = cnt % kBufs;
            if (cnt >= kBufs) mbs_wait_sleep(t_empty_s + 8 * buf, (cnt / kBufs - 1) & 1);  // the DP warps have pulled the step before
            tc_fence_after();
            const uint32_t tmb = tm + buf * kTcBufCols;
            tc_mma_f16(tmb, adesc, bdesc, idesc);
            if (row + 1 < L) tc_mma_f16(tmb + kTcN, adesc + (kTcATileBytes >> 4), bdesc, idesc);
            tcs_commit(t_full_s + 8 * buf);
            adesc += 2 * (kTcATileBytes >> 4);
        }
        tcs_commit(b_empty_s + 8 * stage);
        if (n + kTcStages < ntiles) {  // refill this stage once its MMAs have completed
            mbs_wait_sleep(b_empty_s + 8 * stage, sphase);
            mbs_expect_tx(b_full_s + 8 * stage, kTcBTileBytes);
            tmas_g2s(sB_s + stage * kTcBTileBytes, tile_src, kTcBTileBytes, b_full_s + 8 * stage);
            tile_src += kStride;
        }
        if (++stage == (uint32_t)kTcStages) stage = 0, sphase ^= 1;
    }
}

// The end of a slice for the thread that owns query m's first list: the other NLISTS - 1 lists of the query (list + o kTcM,
// each ascending) are merged into its own ascending list, which then leaves the CTA as the (slice, query) partial dst().out.
// THR (packed-half scans): `worst` never rises above the query's threshold thr0, and a kept worst key below it is published
// to the query's threshold word dst().thr. dst is evaluated once the lists are merged, so that what it reads (k_dtw_scan_h2_2p:
// its group and slice, from shared memory) is not held through the merge.
struct TcListDst {
    unsigned long long* thr;
    unsigned long long* out;
};
template <int KP, int STRIDE, int NLISTS, bool THR, class Dst>
__device__ __forceinline__ void tc_merge_store(unsigned long long* list, unsigned long long worst, unsigned long long thr0, Dst dst) {
    for (int o = 1; o < NLISTS; o++) {
        const unsigned long long* other = list + o * kTcM;
        for (int s = 0; s < KP; s++) {  // ascending: stop at the first key that does not make the cut
            const unsigned long long key = other[s * STRIDE];
            if (key >= worst) break;
            tc_insert_key<KP, STRIDE>(list, worst, key);
            if constexpr (THR) worst = worst < thr0 ? worst : thr0;
        }
    }
    const TcListDst to = dst();
    if constexpr (THR) {
        const unsigned long long kept_worst = list[(KP - 1) * STRIDE];
        if (kept_worst != 0xFFFFFFFFFFFFFFFFull && kept_worst < thr0) atomicMin(to.thr, kept_worst);
    }
#pragma unroll
    for (int s = 0; s < KP; s++) to.out[s] = list[s * STRIDE];
}

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

// ---------------------------------------------------------------------------------------------------------------
// host side of the scan launches
// ---------------------------------------------------------------------------------------------------------------
// dynamic shared memory of a scan CTA: a_rows A tiles, b_rings B-tile rings, the barriers, kp candidate keys per DP thread,
// and the slack of the 128-byte alignment
static inline size_t tc_smem_bytes(uint32_t a_rows, int b_rings, int kp, int dp_threads) {
    return (size_t)a_rows * kTcATileBytes + b_rings * kTcStages * kTcBTileBytes + 32 * 8 + (size_t)kp * dp_threads * 8 + 1024;
}
// one scan launch of p.ngroups x p.nslices CTAs. dependent: it may start while the previous scan launch is still draining
// (programmatic dependent launch; the launches write disjoint candidate lists and none reads another's output)
template <class Params>
static int tc_launch_scan(ss_ctx* ctx, void (*kern)(Params), const Params& p, unsigned threads, size_t smem, bool dependent) {
    SS_CUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(p.ngroups * p.nslices);
    cfg.blockDim = dim3(threads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = ctx->stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = dependent ? 1 : 0;
    SS_CUDA(ctx, cudaLaunchKernelEx(&cfg, kern, p));
    SS_LAUNCHED(ctx);
    return SS_OK;
}

}  // namespace ss
