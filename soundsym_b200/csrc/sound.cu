// sound.cu — the MFCC subsystem (SURVEY.md §8a rows 1-8) and the sample-domain helpers of the matcher (row 17).
//
//   k_decode_pcm   Sound::from_path's sample conversion                      src/sound.rs:118-120
//   k_mfcc         analyze_mfccs: frame 1024/256, Hann, FFT, 12/13 mel bands, log10, DCT-II x2   src/sound.rs:215-242
//                  (arithmetic of sample::window + vox_box::spectrum::MFCC, [RECALL] A1-A4 in oracle/ASSUMPTIONS.h)
//   k_max_power    analyze_max_power: rectangular 128/64 frames, max RMS         src/sound.rs:244-256 (bit-exact fold)
//   k_colsum_*     analyze_mean_mfccs                                            src/sound.rs:271-286
//   k_resynth      clone_from_dictionary's pad / truncate + to_sound's concat   src/sound.rs:451-483
//   k_resynth_warped  the same along the DTW warping path of each match (ss_resynth_warped; no reference counterpart, A11)
//
// k_mfcc: one warp per frame, all arithmetic in f64. The real 1024-point transform is done as a 512-point complex
// Stockham FFT (three radix-8 passes, 2 butterflies per lane per pass, the first pass reading the windowed samples
// straight from global memory with coalesced 16-byte loads, the others exchanging through the warp's 8 KB of shared
// memory), followed by the even/odd split for the bins the mel bank needs (2..229 for C = 12 at 44.1 kHz).
// What bounds it is the SM's L1 data pipe (shared-memory and global-load wavefronts share it: 93 % busy in round 2's
// profile), so every table the warp reads is stored in the order the warp reads it - twiddles per (pass, t, lane), mel
// weights per (step, half band), the DCT matrix transposed: one coalesced load where a gather touched up to 32 lines.
#include <cmath>
#include <map>

#include "sound.cuh"

namespace ss {

struct SoundTables {
    double sample_rate = 0;
    int c = 0;
    int bins[SS_MAX_NCOEFFS + 2] = {0};
    DevBuf<double> d_win;     // 1024 Hann weights (A2)
    DevBuf<double2> d_tw;     // exp(-2 pi i j / 1024), j = 0..1023
    DevBuf<double> d_dct;     // c x c: cos(pi k (2n+1) / (2c))
    DevBuf<int> d_bins;       // c + 2
    // triangle weights of the mel bank, one run per half band (2 f = rising part of band f, 2 f + 1 = falling part): the
    // values (double)i / width and 1.0 - (double)i / width the CPU path forms per element, computed once on the host with
    // the same IEEE operations. d_half: per half band {first bin, count, offset into d_melw}.
    DevBuf<double> d_melw;
    DevBuf<int> d_half;       // 2 c x 3 ints (padded to 4)
    int melw_count = 0;
    // the same tables in the order the warp reads them (one coalesced load per step instead of a gather over up to 32 cache
    // lines - the gathers were half of the kernel's L1 wavefronts, and the L1 data pipe is what bounds it):
    DevBuf<double2> d_tw1;    // [t - 1][lane]      pass 1: tw[16 t (lane & 7)],       t = 1..7
    DevBuf<double2> d_tw2;    // [h][t - 1][lane]   pass 2: tw[2 t (lane + 32 h)],     t = 1..7
    DevBuf<double> d_melw_t;  // [i][lane]          weight i of half band `lane` (0 beyond its count)
    DevBuf<double> d_dct_t;   // [n][16]            dct[k][n] at [n][k]
    int melw_rows = 0;
};

struct MfccTabs {  // device pointers of one SoundTables, by value into k_mfcc
    const double* win;
    const double2* tw;
    const double2* tw1;
    const double2* tw2;
    const double* dct_t;
    const int* bins;
    const double* melw_t;
    const int4* half;
};

struct SoundState {
    std::vector<SoundTables*> tables;
    DevBuf<double> d_samples, d_mfcc, d_partial, d_small;
    DevBuf<int32_t> d_pcm;
    DevBuf<unsigned long long> d_maxbits;
    DevBuf<uint64_t> d_off_a, d_off_b, d_off_pf;
    DevBuf<uint32_t> d_idx;
    DevBuf<uint64_t> d_path_off;  // ss_resynth_warped: path offsets (in cells) and (i, j) cells
    DevBuf<uint2> d_path;
    // chunked ingest (ss_sound_analyze / _pcm on long inputs): the H2D copy of chunk k+1 runs on copy_stream while chunk k is
    // converted and analysed on the ctx stream
    cudaStream_t copy_stream = nullptr;
    cudaEvent_t ev_chunk[2] = {nullptr, nullptr};
    ~SoundState() {
        for (auto* t : tables) delete t;
        for (auto& e : ev_chunk)
            if (e) cudaEventDestroy(e);
        if (copy_stream) cudaStreamDestroy(copy_stream);
    }
};

static void sound_state_free(void* p) { delete static_cast<SoundState*>(p); }

SoundState* sound_state(ss_ctx* ctx) {
    if (!ctx->sound_state) {
        ctx->sound_state = new SoundState();
        ctx->sound_state_free = sound_state_free;
    }
    return static_cast<SoundState*>(ctx->sound_state);
}

static inline double hz_to_mel(double hz) { return 1125.0 * std::log1p(hz / 700.0); }   // [RECALL] vox_box::spectrum
static inline double mel_to_hz(double mel) { return 700.0 * (std::exp(mel / 1125.0) - 1.0); }

static int get_tables(ss_ctx* ctx, double sample_rate, int c, SoundTables** out) {
    SoundState* st = sound_state(ctx);
    for (auto* t : st->tables)
        if (t->sample_rate == sample_rate && t->c == c) {
            *out = t;
            return SS_OK;
        }
    const double kPi = 3.14159265358979323846264338327950288;
    SoundTables* t = new SoundTables();
    t->sample_rate = sample_rate;
    t->c = c;
    // mel band edges (A3b-c): c+2 points spaced (hi-lo)/c in mel, bin = floor((N+1) hz / sr)
    const double lo = hz_to_mel(SS_F_LO), range = hz_to_mel(SS_F_HI) - lo;
    for (int i = 0; i < c + 2; i++) {
        const double point = ((double)i / (double)c) * range + lo;
        t->bins[i] = (int)std::floor((double)(SS_BIN + 1) * mel_to_hz(point) / sample_rate);
    }
    bool ok = t->bins[0] >= 0 && t->bins[c + 1] <= SS_BIN / 2;
    for (int i = 0; i < c + 1; i++) ok = ok && t->bins[i + 1] > t->bins[i];
    if (!ok) {
        delete t;
        return set_error(ctx, SS_ERR_INVALID, "sample rate %.1f Hz: mel band edges leave [0, %d] or collapse (needs sr >= ~17.9 kHz)",
                         sample_rate, SS_BIN / 2);
    }
    std::vector<double> win(SS_BIN), dct((size_t)c * c);
    std::vector<double2> tw(SS_BIN);
    for (int i = 0; i < SS_BIN; i++) {
        win[i] = 0.5 * (1.0 - std::cos(2.0 * kPi * (double)i / (double)(SS_BIN - 1)));  // A2: symmetric Hann
        const double ang = -2.0 * kPi * (double)i / (double)SS_BIN;
        tw[i] = make_double2(std::cos(ang), std::sin(ang));
    }
    for (int k = 0; k < c; k++)
        for (int n = 0; n < c; n++) dct[(size_t)k * c + n] = std::cos(kPi * (double)k * (2.0 * (double)n + 1.0) / (2.0 * (double)c));
    std::vector<double> melw;
    std::vector<int> half;
    for (int f = 0; f < c; f++) {
        const int b0 = t->bins[f], b1 = t->bins[f + 1], b2 = t->bins[f + 2];
        const double up = (double)(b1 - b0), down = (double)(b2 - b1);
        half.insert(half.end(), {b0, b1 - b0, (int)melw.size(), 0});
        for (int i = 0; i < b1 - b0; i++) melw.push_back((double)i / up);
        half.insert(half.end(), {b1, b2 - b1, (int)melw.size(), 0});
        for (int i = 0; i < b2 - b1; i++) melw.push_back(1.0 - (double)i / down);
    }
    t->melw_count = (int)melw.size();
    std::vector<double2> tw1(7 * 32), tw2(2 * 7 * 32);
    for (int tt = 1; tt < 8; tt++)
        for (int l = 0; l < 32; l++) {
            tw1[(tt - 1) * 32 + l] = tw[(tt * (l & 7) * 16) & (SS_BIN - 1)];
            for (int h = 0; h < 2; h++) tw2[(h * 7 + tt - 1) * 32 + l] = tw[(tt * (l + 32 * h) * 2) & (SS_BIN - 1)];
        }
    int rows = 1;
    for (int h = 0; h < 2 * c; h++) rows = std::max(rows, half[4 * h + 1]);
    t->melw_rows = rows;
    std::vector<double> melw_t((size_t)rows * 32, 0.0), dct_t((size_t)c * 16, 0.0);
    for (int h = 0; h < 2 * c; h++)
        for (int i = 0; i < half[4 * h + 1]; i++) melw_t[(size_t)i * 32 + h] = melw[half[4 * h + 2] + i];
    for (int k = 0; k < c; k++)
        for (int n = 0; n < c; n++) dct_t[(size_t)n * 16 + k] = dct[(size_t)k * c + n];
    int rc = upload(ctx, t->d_win, win.data(), win.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_melw, melw.data(), melw.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_half, half.data(), half.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_tw, tw.data(), tw.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_dct, dct.data(), dct.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_bins, t->bins, (size_t)c + 2);
    if (rc == SS_OK) rc = upload(ctx, t->d_tw1, tw1.data(), tw1.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_tw2, tw2.data(), tw2.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_melw_t, melw_t.data(), melw_t.size());
    if (rc == SS_OK) rc = upload(ctx, t->d_dct_t, dct_t.data(), dct_t.size());
    if (rc == SS_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = set_error(ctx, SS_ERR_CUDA, "table upload failed");
    if (rc != SS_OK) {
        delete t;
        return rc;
    }
    st->tables.push_back(t);
    *out = t;
    return SS_OK;
}

static MfccTabs mfcc_tabs(const SoundTables* t) {
    return MfccTabs{t->d_win.p, t->d_tw.p, t->d_tw1.p, t->d_tw2.p, t->d_dct_t.p, t->d_bins.p, t->d_melw_t.p, reinterpret_cast<const int4*>(t->d_half.p)};
}

// ---------------------------------------------------------------------------------------------------------------
__global__ void k_decode_pcm(const int32_t* __restrict__ pcm, size_t n, double denom, double* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __ddiv_rn((double)pcm[i], denom);
}
__global__ void k_decode_pcm16(const int16_t* __restrict__ pcm, size_t n, double denom, double* __restrict__ out) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = __ddiv_rn((double)pcm[i], denom);
}

// ---------------------------------------------------------------------------------------------------------------
struct cplx {
    double x, y;
};
__device__ __forceinline__ cplx cadd(cplx a, cplx b) { return {a.x + b.x, a.y + b.y}; }
__device__ __forceinline__ cplx csub(cplx a, cplx b) { return {a.x - b.x, a.y - b.y}; }
__device__ __forceinline__ cplx cmul(cplx a, cplx b) { return {a.x * b.x - a.y * b.y, a.x * b.y + a.y * b.x}; }
__device__ __forceinline__ cplx mul_negi(cplx a) { return {a.y, -a.x}; }  // a * (-i)

// natural-order 8-point DFT (decimation in frequency), in place
__device__ __forceinline__ void dft8(cplx* u) {
    const double s = 0.70710678118654752440084436210485;
    cplx a0 = cadd(u[0], u[4]), a1 = cadd(u[1], u[5]), a2 = cadd(u[2], u[6]), a3 = cadd(u[3], u[7]);
    cplx b0 = csub(u[0], u[4]), b1 = csub(u[1], u[5]), b2 = csub(u[2], u[6]), b3 = csub(u[3], u[7]);
    b1 = cmul(b1, cplx{s, -s});
    b2 = mul_negi(b2);
    b3 = cmul(b3, cplx{-s, -s});
    const cplx c0 = cadd(a0, a2), c1 = cadd(a1, a3), c2 = csub(a0, a2), c3 = mul_negi(csub(a1, a3));
    const cplx d0 = cadd(b0, b2), d1 = cadd(b1, b3), d2 = csub(b0, b2), d3 = mul_negi(csub(b1, b3));
    u[0] = cadd(c0, c1);
    u[1] = cadd(d0, d1);
    u[2] = cadd(c2, c3);
    u[3] = cadd(d2, d3);
    u[4] = csub(c0, c1);
    u[5] = csub(d0, d1);
    u[6] = csub(c2, c3);
    u[7] = csub(d2, d3);
}

constexpr int kMfccWarps = 4;
constexpr int kHalf = SS_BIN / 2;  // 512
// Where element `idx` of the warp's 512 x double2 exchange buffer lives: the low three index bits are XOR-ed with the next
// three. A quarter-warp's 16-byte accesses are conflict-free when its 8 addresses cover 8 different 16-byte bank groups; the
// Stockham stores of passes 0 and 1 go to idx = 8 i + t and (i & ~7) 8 + (i & 7) + 8 t (lane i, fixed t) - stride 8 in the low
// bits, an 8-way conflict in the natural layout (pass 0 alone was half of the kernel's shared-memory wavefronts) - and the
// loads to idx = i + 64 t; with the swizzle every one of them touches 8 distinct groups.
__device__ __forceinline__ int mfcc_sw(int idx) { return idx ^ ((idx >> 3) & 7); }

// largest s in [0, n) with off[s] <= x (off ascending, off[0] = 0 <= x < off[n])
__device__ __forceinline__ uint32_t seg_of(const uint64_t* __restrict__ off, uint32_t n, uint64_t x) {
    uint32_t lo = 0, hi = n;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (off[mid] <= x) lo = mid;
        else hi = mid;
    }
    return lo;
}

// (min CTAs per SM: 4 -> 128 registers per thread without spills, 16 warps / SM; left to itself the compiler takes 168
// registers = 12 warps / SM. 40.5 KB of shared memory per CTA at 44.1 kHz.)
#ifndef SS_MFCC_MINBLOCKS
#define SS_MFCC_MINBLOCKS 4
#endif
// Measured and NOT kept (1 h of audio, same commit; the kernel sits at the 128-register edge and every variant below spills
// 90 - 670 B per thread through the L1 data pipe, which is the unit that bounds the kernel):
//   SS_MFCC_PREFETCH 1 (first half of the next frame's samples fetched before the band / DCT stages)  2.91 - 3.16 ms
//   SS_MFCC_PREFETCH 2 (prefetch.global.L2 of the next frame, no registers)                           2.60 ms with SPLIT 2
//   SS_MFCC_SPLIT 2 / 4 (independent bins per lane and step in the even/odd split)                     2.54 / 2.72 ms
// against 2.39 ms for the plain loop.
#ifndef SS_MFCC_PREFETCH
#define SS_MFCC_PREFETCH 0
#endif
#ifndef SS_MFCC_SPLIT
#define SS_MFCC_SPLIT 1
#endif
__global__ void __launch_bounds__(kMfccWarps * 32, SS_MFCC_MINBLOCKS)
k_mfcc(const double* __restrict__ samples, size_t frames, const MfccTabs tabs, int c, int pw_len, double energy_floor,
       double* __restrict__ out, const uint64_t* __restrict__ frame_off = nullptr, const uint64_t* __restrict__ samp_off = nullptr,
       uint32_t nsounds = 0) {
    const double* __restrict__ win = tabs.win;
    const double2* __restrict__ tw = tabs.tw;
    const double2* __restrict__ tw1 = tabs.tw1 + (threadIdx.x & 31);
    const double2* __restrict__ tw2 = tabs.tw2 + (threadIdx.x & 31);
    const double* __restrict__ dct_t = tabs.dct_t;
    const int* __restrict__ bins = tabs.bins;
    const int4* __restrict__ halfband = tabs.half;
    extern __shared__ __align__(16) unsigned char mfcc_smem[];
    double2* s_buf = reinterpret_cast<double2*>(mfcc_smem);                                   // [warps][512]  32 KB
    double* s_pw = reinterpret_cast<double*>(mfcc_smem + sizeof(double2) * kMfccWarps * kHalf);  // [warps][pw_len]: bins below the bank's top edge
    double* s_le_all = s_pw + kMfccWarps * pw_len;                                            // [warps][16]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double2* buf = s_buf + warp * kHalf;
    double* pw = s_pw + warp * pw_len;         // power spectrum of the bins the bank reads
    double* s_le = s_le_all + warp * 16;
    const int kb0 = bins[0], kb1 = bins[c + 1];
    // lane h < 2 c sums half band h (rising or falling part of band h / 2) sequentially, in the CPU path's element order
    const int4 hb = lane < 2 * c ? __ldg(&halfband[lane]) : make_int4(0, 0, 0, 0);
    const double* hw = tabs.melw_t + lane;  // weight i of this lane's half band at hw[32 i]

    // first sample of frame f. One sound: f * HOP. Batch (ss_sound_analyze_batch): frame f belongs to the sound whose frame
    // range holds it and starts at that sound's first sample + local frame * HOP (any alignment: scalar loads)
    auto frame_start = [&](size_t f) -> size_t {
        if (!frame_off) return f * SS_HOP;
        const uint32_t snd = seg_of(frame_off, nsounds, f);
        return samp_off[snd] + (f - frame_off[snd]) * SS_HOP;
    };
    // half h of the frame's 1024 samples as double2: element i + 64 t of lane i = lane + 32 h in sv[t]
    auto load_half = [&](size_t f, int h, double2 (&sv)[8]) {
        const size_t start = frame_start(f);
        const double* s1 = samples + start;
        if ((start & 1) == 0) {
            const double2* s2 = reinterpret_cast<const double2*>(s1);
#pragma unroll
            for (int t = 0; t < 8; t++) sv[t] = s2[lane + 32 * h + 64 * t];
        } else {
#pragma unroll
            for (int t = 0; t < 8; t++) {
                const int n = lane + 32 * h + 64 * t;
                sv[t] = make_double2(s1[2 * n], s1[2 * n + 1]);
            }
        }
    };
    const size_t fstride = (size_t)gridDim.x * kMfccWarps;
    size_t f = (size_t)blockIdx.x * kMfccWarps + warp;
    double2 sv0[8];
#if SS_MFCC_PREFETCH == 1
    if (f < frames) load_half(f, 0, sv0);
#endif
    for (; f < frames; f += fstride) {
        const double2* w2 = reinterpret_cast<const double2*>(win);
        // ---- pass 0 (Ns = 1): z[n] = (x[2n] w[2n], x[2n+1] w[2n+1]) straight from global memory (coalesced 16-byte loads) ---
        cplx u[2][8];
        double2 sv1[8];
#if SS_MFCC_PREFETCH != 1
        load_half(f, 0, sv0);
#endif
        load_half(f, 1, sv1);
#pragma unroll
        for (int h = 0; h < 2; h++) {
            const int i = lane + 32 * h;
#pragma unroll
            for (int t = 0; t < 8; t++) {
                const double2 wv = __ldg(&w2[i + 64 * t]);
                const double2 x = h == 0 ? sv0[t] : sv1[t];
                u[h][t] = cplx{x.x * wv.x, x.y * wv.y};
            }
            dft8(u[h]);
#pragma unroll
            for (int t = 0; t < 8; t++) buf[8 * i + (t ^ (i & 7))] = make_double2(u[h][t].x, u[h][t].y);  // = mfcc_sw(8 i + t)
        }
        __syncwarp();
        // ---- passes 1, 2 (Ns = 8, 64) -------------------------------------------------------------------------------
#pragma unroll
        for (int pass = 1; pass <= 2; pass++) {
            const int p = pass == 1 ? 8 : 64;
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int i = lane + 32 * h;
                const int bi = mfcc_sw(i);  // mfcc_sw(i + 64 t) = mfcc_sw(i) + 64 t
                // twiddle exp(-2 pi i t k / (8 p)) = tw[t k 128 / p], k = i & (p - 1), from the lane-ordered tables; t = 0 is 1
                const double2* twp = pass == 1 ? tw1 : tw2 + h * 7 * 32;
                {
                    const double2 v = buf[bi];
                    u[h][0] = cplx{v.x, v.y};
                }
#pragma unroll
                for (int t = 1; t < 8; t++) {
                    const double2 v = buf[bi + 64 * t];
                    const double2 w = __ldg(&twp[(t - 1) * 32]);
                    u[h][t] = cmul(cplx{v.x, v.y}, cplx{w.x, w.y});
                }
                dft8(u[h]);
            }
            __syncwarp();
#pragma unroll
            for (int h = 0; h < 2; h++) {
                const int i = lane + 32 * h;
                const int k = i & (p - 1);
                const int jo = ((i - k) << 3) + k;
                // mfcc_sw(jo + t p): p = 8 -> (i - k) 8 + 8 t + (k ^ t);  p = 64 -> mfcc_sw(jo) + 64 t
                const int js = mfcc_sw(jo);
#pragma unroll
                for (int t = 0; t < 8; t++)
                    buf[pass == 1 ? ((i - k) << 3) + 8 * t + (k ^ t) : js + 64 * t] = make_double2(u[h][t].x, u[h][t].y);
            }
            __syncwarp();
        }
#if SS_MFCC_PREFETCH == 1
        if (f + fstride < frames) load_half(f + fstride, 0, sv0);  // consumed by the next iteration's pass 0
#elif SS_MFCC_PREFETCH == 2
        if (f + fstride < frames) {  // the next frame's 64 cache lines towards L2, two per lane (no registers held)
            const char* nx = reinterpret_cast<const char*>(samples + frame_start(f + fstride)) + 128 * lane;
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nx));
            asm volatile("prefetch.global.L2 [%0];" ::"l"(nx + 4096));
        }
#endif
        // ---- even/odd split: X[k] = E[k] + W_1024^k O[k] for the bins of the mel bank; power |X|^2 (A3) -------------
        for (int k0 = kb0 + lane; k0 < kb1; k0 += 32 * SS_MFCC_SPLIT) {
            double2 zk[SS_MFCC_SPLIT], zm[SS_MFCC_SPLIT], w[SS_MFCC_SPLIT];
#pragma unroll
            for (int j = 0; j < SS_MFCC_SPLIT; j++) {
                const int k = k0 + 32 * j;
                if (k < kb1) {
                    zk[j] = buf[mfcc_sw(k & (kHalf - 1))];
                    zm[j] = buf[mfcc_sw((kHalf - k) & (kHalf - 1))];
                    w[j] = __ldg(&tw[k]);
                }
            }
#pragma unroll
            for (int j = 0; j < SS_MFCC_SPLIT; j++) {
                const int k = k0 + 32 * j;
                if (k < kb1) {
                    const cplx e = {0.5 * (zk[j].x + zm[j].x), 0.5 * (zk[j].y - zm[j].y)};
                    const cplx o = {0.5 * (zk[j].y + zm[j].y), -0.5 * (zk[j].x - zm[j].x)};  // (Zk - conj(Zm)) / (2i)
                    const cplx x = cadd(e, cmul(cplx{w[j].x, w[j].y}, o));
                    pw[k] = x.x * x.x + x.y * x.y;
                }
            }
        }
        __syncwarp();
        // ---- triangular bands (un-normalised; rise starts at 0, fall starts at 1), log10 with the A4 floor ------------
        // 2 c lanes each fold one half band (weights from the table: no division in the loop), then band f = rise + fall
        {
            double part = 0.0;
            for (int i = 0; i < hb.y; i++) part = part + pw[hb.x + i] * __ldg(&hw[32 * i]);
            const double up_sum = __shfl_sync(0xffffffffu, part, (2 * lane) & 31), down_sum = __shfl_sync(0xffffffffu, part, (2 * lane + 1) & 31);
            if (lane < c) {
                const double e = up_sum + down_sum;
                s_le[lane] = log10(e > energy_floor ? e : energy_floor);
            }
        }
        __syncwarp();
        // ---- DCT-II x 2 ---------------------------------------------------------------------------------------------
        if (lane < c) {
            double acc = 0.0;
            for (int n = 0; n < c; n++) acc = acc + s_le[n] * __ldg(&dct_t[n * 16 + lane]);
            out[f * c + lane] = 2.0 * acc;
        }
        __syncwarp();
    }
}

// analyze_max_power: one thread per 128/64 frame, the reference's sequential fold with separate multiply and add
__global__ void k_max_power(const double* __restrict__ samples, size_t frames, unsigned long long* __restrict__ out_bits) {
    const size_t f = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    double rms = 0.0;
    if (f < frames) {
        const double* s = samples + f * 64;
        double acc = 0.0;
        for (int i = 0; i < 128; i++) acc = __dadd_rn(acc, __dmul_rn(s[i], s[i]));
        rms = __dsqrt_rn(__ddiv_rn(acc, 128.0));
        if (!(rms == rms)) rms = 0.0;  // f64::max ignores NaN (src/sound.rs:255)
    }
    for (int o = 16; o; o >>= 1) rms = fmax(rms, __shfl_xor_sync(0xffffffffu, rms, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out_bits, (unsigned long long)__double_as_longlong(rms));  // rms >= 0
}

// batch forms (ss_sound_analyze_batch): per-sound max power and per-sound mean MFCC
__global__ void k_max_power_batch(const double* __restrict__ samples, const uint64_t* __restrict__ samp_off, const uint64_t* __restrict__ pf_off,
                                  uint32_t nsounds, size_t pframes, unsigned long long* __restrict__ out_bits /* nsounds, zeroed */) {
    const size_t f = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= pframes) return;
    const uint32_t snd = seg_of(pf_off, nsounds, f);
    const double* s = samples + samp_off[snd] + (f - pf_off[snd]) * 64;
    double acc = 0.0;
    for (int i = 0; i < 128; i++) acc = __dadd_rn(acc, __dmul_rn(s[i], s[i]));
    double rms = __dsqrt_rn(__ddiv_rn(acc, 128.0));
    if (!(rms == rms)) rms = 0.0;
    atomicMax(&out_bits[snd], (unsigned long long)__double_as_longlong(rms));  // rms >= 0
}
// one thread per (sound, coefficient): the reference's row-by-row accumulation, then / frames (NaN for an empty sound)
__global__ void k_mean_batch(const double* __restrict__ mfcc, const uint64_t* __restrict__ frame_off, uint32_t nsounds, int c,
                             double* __restrict__ out /* nsounds x c */) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (size_t)nsounds * c) return;
    const uint32_t snd = (uint32_t)(t / c);
    const int col = (int)(t % c);
    const uint64_t f0 = frame_off[snd], f1 = frame_off[snd + 1];
    double acc = 0.0;
    for (uint64_t f = f0; f < f1; f++) acc = acc + mfcc[f * c + col];
    out[t] = acc / (double)(f1 - f0);
}

// column sums in two deterministic stages
__global__ void k_colsum_partial(const double* __restrict__ m, size_t rows, int c, double* __restrict__ partial) {
    __shared__ double s[256];
    const int col = threadIdx.x % 16, rl = threadIdx.x / 16;  // 16 row-lanes x 16 columns
    double acc = 0.0;
    if (col < c)
        for (size_t r = (size_t)blockIdx.x * 16 + rl; r < rows; r += (size_t)gridDim.x * 16) acc += m[r * c + col];
    s[threadIdx.x] = acc;
    __syncthreads();
    if (rl == 0) {
        for (int j = 1; j < 16; j++) acc += s[j * 16 + col];
        partial[(size_t)blockIdx.x * 16 + col] = acc;
    }
}
__global__ void k_colsum_final(const double* __restrict__ partial, int nblocks, size_t rows, int c, double* __restrict__ out) {
    const int col = threadIdx.x;
    if (col >= c) return;
    double acc = 0.0;
    for (int b = 0; b < nblocks; b++) acc += partial[(size_t)b * 16 + col];
    out[col] = acc / (double)rows;  // 0/0 = NaN for an empty sound, as the reference
}

// clone_from_dictionary + to_sound: output sample -> (target segment by binary search) -> dictionary sample or 0
__global__ void k_resynth(const double* __restrict__ dict_samples, const uint64_t* __restrict__ dict_off,
                          const uint32_t* __restrict__ match_idx, const uint64_t* __restrict__ out_off, size_t nseg, size_t total,
                          double* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        size_t lo = 0, hi = nseg;  // last segment whose out_off <= i
        while (hi - lo > 1) {
            const size_t mid = (lo + hi) >> 1;
            if (out_off[mid] <= i) lo = mid;
            else hi = mid;
        }
        const uint64_t within = i - out_off[lo];
        const uint32_t m = match_idx[lo];
        const uint64_t b = dict_off[m], e = dict_off[m + 1];
        out[i] = within < e - b ? dict_samples[b + within] : 0.0;
    }
}

// Resynthesis along the DTW warping path (ss_resynth_warped, DESIGN.md §3.5, A11): output block b (SS_HOP samples) of segment t
// plays dictionary frame j(b) = the j of the first path cell of row b; past the path's last row the source runs on at unit speed.
// Where j(b - 1) -> j(b) is not a unit step, the block crossfades linearly from where the previous block would have gone on.
// Path cells are in forward order, so their i is non-decreasing and every row 0..Lq-1 occurs: the first cell of row b is the
// lower bound of b in the segment's i values. The 32 lanes of a warp share b (SS_HOP is a multiple of 32) unless the warp
// straddles two segments, so the search reads broadcast.
__device__ __forceinline__ uint64_t warp_src_frame(const uint2* __restrict__ path, uint64_t p0, uint64_t p1, uint64_t b) {
    if (p0 == p1) return b;  // empty path: the diagonal
    const uint64_t lq = (uint64_t)path[p1 - 1].x + 1;
    const uint64_t row = b < lq ? b : lq - 1;
    uint64_t lo = p0, hi = p1 - 1;  // first cell with i >= row; row <= the last cell's i, so it lies in [p0, p1 - 1]
    while (lo < hi) {
        const uint64_t mid = (lo + hi) >> 1;
        if ((uint64_t)path[mid].x < row) lo = mid + 1;
        else hi = mid;
    }
    return (uint64_t)path[lo].y + (b - row);
}

__global__ void k_resynth_warped(const double* __restrict__ dict_samples, const uint64_t* __restrict__ dict_off,
                                 const uint32_t* __restrict__ match_idx, const uint2* __restrict__ path, const uint64_t* __restrict__ path_off,
                                 const uint64_t* __restrict__ out_off, size_t nseg, size_t total, double* __restrict__ out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        size_t lo = 0, hi = nseg;  // last segment whose out_off <= i
        while (hi - lo > 1) {
            const size_t mid = (lo + hi) >> 1;
            if (out_off[mid] <= i) lo = mid;
            else hi = mid;
        }
        const uint64_t within = i - out_off[lo], b = within / SS_HOP, r = within % SS_HOP;
        const uint32_t m = match_idx[lo];
        const uint64_t base = dict_off[m], len = dict_off[m + 1] - base, p0 = path_off[lo], p1 = path_off[lo + 1];
        auto x = [&](uint64_t p) { return p < len ? dict_samples[base + p] : 0.0; };
        const uint64_t s = warp_src_frame(path, p0, p1, b) * SS_HOP;
        const double a = x(s + r);
        double v = a;
        if (b > 0) {
            const uint64_t prev = warp_src_frame(path, p0, p1, b - 1) * SS_HOP;
            if (s != prev + SS_HOP) {  // not contiguous: c (H - r) / H + a r / H, weights exact, no FMA
                const double c = x(prev + SS_HOP + r);
                v = __dadd_rn(__dmul_rn(c, (double)(SS_HOP - r) * (1.0 / SS_HOP)), __dmul_rn(a, (double)r * (1.0 / SS_HOP)));
            }
        }
        out[i] = v;
    }
}

// ---------------------------------------------------------------------------------------------------------------
static int mfcc_launch(ss_ctx* ctx, const double* d_samples, size_t n, double sample_rate, int c, double* d_out, size_t frames) {
    if (!frames) return SS_OK;
    SoundTables* t = nullptr;
    SS_TRY(get_tables(ctx, sample_rate, c, &t));
    const int grid = (int)std::min<size_t>((frames + kMfccWarps - 1) / kMfccWarps, (size_t)ctx->sm_count * 4 * SS_MFCC_MINBLOCKS);
    const int pw_len = (t->bins[c + 1] + 32) & ~31;  // 256 at 44.1 kHz (top edge bin 230)
    const int smem = (int)(sizeof(double2) * kMfccWarps * kHalf + sizeof(double) * kMfccWarps * pw_len + sizeof(double) * kMfccWarps * 16);
    SS_CUDA(ctx, cudaFuncSetAttribute(k_mfcc, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    k_mfcc<<<grid, kMfccWarps * 32, smem, ctx->stream>>>(d_samples, frames, mfcc_tabs(t), c, pw_len, 1e-10, d_out);
    SS_LAUNCHED(ctx);
    (void)n;
    return SS_OK;
}

static int check_c(ss_ctx* ctx, int c) {
    if (c < 1 || c > SS_MAX_NCOEFFS) return set_error(ctx, SS_ERR_INVALID, "ncoeffs must be in 1..%d (got %d)", SS_MAX_NCOEFFS, c);
    return SS_OK;
}

}  // namespace ss

using namespace ss;

extern "C" {

int ss_decode_pcm(ss_ctx* ctx, const int32_t* pcm, size_t n, int bits, double* out_samples) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (bits < 1 || bits > 32) return set_error(ctx, SS_ERR_INVALID, "bits_per_sample must be in 1..32 (got %d)", bits);
    if (n && (!pcm || !out_samples)) return set_error(ctx, SS_ERR_INVALID, "NULL buffer");
    if (!n) return SS_OK;
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SoundState* st = sound_state(ctx);
    SS_TRY(upload(ctx, st->d_pcm, pcm, n));
    SS_CUDA(ctx, st->d_samples.reserve(n));
    const double denom = (double)(INT32_MAX >> (32 - bits));  // i32::max_value().wrapping_shr(32 - bits)
    k_decode_pcm<<<ceil_div((long long)n, 256), 256, 0, ctx->stream>>>(st->d_pcm.p, n, denom, st->d_samples.p);
    SS_LAUNCHED(ctx);
    SS_CUDA(ctx, cudaMemcpyAsync(out_samples, st->d_samples.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SS_OK;
}

int ss_mfcc_dev(ss_ctx* ctx, const double* d_samples, size_t n, double sample_rate, int ncoeffs, double* d_out_mfcc) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    SS_TRY(check_c(ctx, ncoeffs));
    size_t frames = 0;
    ss_frame_count(n, &frames);
    if (frames && (!d_samples || !d_out_mfcc)) return set_error(ctx, SS_ERR_INVALID, "NULL buffer");
    if (((uintptr_t)d_samples & 15) != 0) return set_error(ctx, SS_ERR_INVALID, "d_samples must be 16-byte aligned");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    return mfcc_launch(ctx, d_samples, n, sample_rate, ncoeffs, d_out_mfcc, frames);
}

// Chunked, double-buffered ingest (SURVEY.md §8f item 2): samples arrive in chunks of kChunkSamples; chunk k+1 is copied
// host -> device on copy_stream while chunk k is converted (integer PCM) and the MFCC frames it completes are computed on
// the ctx stream. Works for pinned and pageable host memory alike (with pageable memory the copy call blocks the host,
// but the previous chunk's kernels are already enqueued). Results are identical to the one-shot path: the same kernels
// run on sub-ranges, and every frame is independent.
constexpr size_t kChunkSamples = size_t(4) << 20;

// bits = 0: f64 samples; 16: int16 PCM; 24 / 32: int32 PCM. Leaves the samples in st->d_samples and, if want_mfcc, the MFCC
// frames in st->d_mfcc.
static int ingest_chunked(ss_ctx* ctx, SoundState* st, const void* src, size_t n, int bits, double sample_rate, int ncoeffs, bool want_mfcc) {
    if (!st->copy_stream) {
        SS_CUDA(ctx, cudaStreamCreateWithFlags(&st->copy_stream, cudaStreamNonBlocking));
        for (auto& e : st->ev_chunk) SS_CUDA(ctx, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    size_t frames = 0;
    ss_frame_count(n, &frames);
    SS_CUDA(ctx, st->d_samples.reserve(n));
    if (want_mfcc && frames) SS_CUDA(ctx, st->d_mfcc.reserve(frames * (size_t)ncoeffs));
    const size_t esz = bits == 0 ? sizeof(double) : (bits == 16 ? sizeof(int16_t) : sizeof(int32_t));
    if (bits) SS_CUDA(ctx, st->d_pcm.reserve(bits == 16 ? (n + 1) / 2 : n));
    const double denom = bits ? (double)(INT32_MAX >> (32 - bits)) : 1.0;  // src/sound.rs:118-120
    // the copy stream must not overwrite buffers that earlier work on the ctx stream still reads
    SS_CUDA(ctx, cudaEventRecord(st->ev_chunk[0], ctx->stream));
    SS_CUDA(ctx, cudaStreamWaitEvent(st->copy_stream, st->ev_chunk[0], 0));
    size_t frames_done = 0;
    int k = 0;
    for (size_t s0 = 0; s0 < n; s0 += kChunkSamples, k++) {
        const size_t s1 = std::min(n, s0 + kChunkSamples), cn = s1 - s0;
        unsigned char* dst = bits == 0 ? reinterpret_cast<unsigned char*>(st->d_samples.p) : reinterpret_cast<unsigned char*>(st->d_pcm.p);
        SS_CUDA(ctx, cudaMemcpyAsync(dst + s0 * esz, static_cast<const unsigned char*>(src) + s0 * esz, cn * esz, cudaMemcpyHostToDevice,
                                     st->copy_stream));
        SS_CUDA(ctx, cudaEventRecord(st->ev_chunk[k & 1], st->copy_stream));
        SS_CUDA(ctx, cudaStreamWaitEvent(ctx->stream, st->ev_chunk[k & 1], 0));
        if (bits == 16) {
            k_decode_pcm16<<<ceil_div((long long)cn, 256), 256, 0, ctx->stream>>>(reinterpret_cast<const int16_t*>(st->d_pcm.p) + s0, cn, denom,
                                                                                st->d_samples.p + s0);
            SS_LAUNCHED(ctx);
        } else if (bits) {
            k_decode_pcm<<<ceil_div((long long)cn, 256), 256, 0, ctx->stream>>>(st->d_pcm.p + s0, cn, denom, st->d_samples.p + s0);
            SS_LAUNCHED(ctx);
        }
        if (want_mfcc) {
            size_t f1 = 0;
            ss_frame_count(s1, &f1);  // frames that lie entirely inside the samples received so far
            if (f1 > frames_done) {
                SS_TRY(mfcc_launch(ctx, st->d_samples.p + frames_done * 256, s1 - frames_done * 256, sample_rate, ncoeffs,
                                   st->d_mfcc.p + frames_done * (size_t)ncoeffs, f1 - frames_done));
                frames_done = f1;
            }
        }
    }
    return SS_OK;
}

// the three analyses on samples already in st->d_samples (mfcc_done: st->d_mfcc already holds the frames);
// stream-synchronised on return
static int analyze_resident(ss_ctx* ctx, SoundState* st, size_t n, double sample_rate, int ncoeffs, double* out_mfcc, size_t* out_frames,
                            double* out_max_power, double* out_mean_mfccs, bool mfcc_done = false) {
    size_t frames = 0;
    ss_frame_count(n, &frames);
    if (out_frames) *out_frames = frames;
    const bool want_mfcc = out_mfcc || out_mean_mfccs;
    if (want_mfcc && frames) {
        if (!mfcc_done) {
            SS_CUDA(ctx, st->d_mfcc.reserve(frames * (size_t)ncoeffs));
            SS_TRY(mfcc_launch(ctx, st->d_samples.p, n, sample_rate, ncoeffs, st->d_mfcc.p, frames));
        }
        if (out_mfcc)
            SS_CUDA(ctx, cudaMemcpyAsync(out_mfcc, st->d_mfcc.p, frames * (size_t)ncoeffs * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (out_mean_mfccs) {
        SS_CUDA(ctx, st->d_small.reserve(16));
        const int nb = (int)std::min<size_t>(std::max<size_t>(frames / 64, 1), 1024);
        SS_CUDA(ctx, st->d_partial.reserve((size_t)nb * 16));
        k_colsum_partial<<<nb, 256, 0, ctx->stream>>>(st->d_mfcc.p, frames, ncoeffs, st->d_partial.p);
        SS_LAUNCHED(ctx);
        k_colsum_final<<<1, 32, 0, ctx->stream>>>(st->d_partial.p, nb, frames, ncoeffs, st->d_small.p);
        SS_LAUNCHED(ctx);
        SS_CUDA(ctx, cudaMemcpyAsync(out_mean_mfccs, st->d_small.p, (size_t)ncoeffs * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    unsigned long long bits = 0;
    if (out_max_power) {
        SS_CUDA(ctx, st->d_maxbits.reserve(1));
        SS_CUDA(ctx, cudaMemsetAsync(st->d_maxbits.p, 0, sizeof(unsigned long long), ctx->stream));
        const size_t pframes = n >= 128 ? (n - 128) / 64 + 1 : 0;
        if (pframes) {
            k_max_power<<<ceil_div((long long)pframes, 128), 128, 0, ctx->stream>>>(st->d_samples.p, pframes, st->d_maxbits.p);
            SS_LAUNCHED(ctx);
        }
        SS_CUDA(ctx, cudaMemcpyAsync(&bits, st->d_maxbits.p, sizeof(bits), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (out_max_power) memcpy(out_max_power, &bits, sizeof(double));
    return SS_OK;
}

int ss_sound_analyze(ss_ctx* ctx, const double* samples, size_t n, double sample_rate, int ncoeffs, double* out_mfcc,
                     size_t* out_frames, double* out_max_power, double* out_mean_mfccs) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    SS_TRY(check_c(ctx, ncoeffs));
    if (n && !samples) return set_error(ctx, SS_ERR_INVALID, "samples is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SoundState* st = sound_state(ctx);
    if (n > kChunkSamples) {
        SS_TRY(ingest_chunked(ctx, st, samples, n, 0, sample_rate, ncoeffs, out_mfcc || out_mean_mfccs));
        return analyze_resident(ctx, st, n, sample_rate, ncoeffs, out_mfcc, out_frames, out_max_power, out_mean_mfccs, true);
    }
    SS_TRY(upload(ctx, st->d_samples, samples, n));
    return analyze_resident(ctx, st, n, sample_rate, ncoeffs, out_mfcc, out_frames, out_max_power, out_mean_mfccs);
}

int ss_sound_analyze_pcm(ss_ctx* ctx, const void* pcm, size_t n, int bits_per_sample, double sample_rate, int ncoeffs, double* out_samples,
                         double* out_mfcc, size_t* out_frames, double* out_max_power, double* out_mean_mfccs) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    SS_TRY(check_c(ctx, ncoeffs));
    if (bits_per_sample != 16 && bits_per_sample != 24 && bits_per_sample != 32)
        return set_error(ctx, SS_ERR_INVALID, "bits_per_sample must be 16 (int16 buffer), 24 or 32 (int32 buffer); got %d", bits_per_sample);
    if (n && !pcm) return set_error(ctx, SS_ERR_INVALID, "pcm is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SoundState* st = sound_state(ctx);
    if (n > kChunkSamples) {
        SS_TRY(ingest_chunked(ctx, st, pcm, n, bits_per_sample, sample_rate, ncoeffs, out_mfcc || out_mean_mfccs));
        if (out_samples) SS_CUDA(ctx, cudaMemcpyAsync(out_samples, st->d_samples.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        return analyze_resident(ctx, st, n, sample_rate, ncoeffs, out_mfcc, out_frames, out_max_power, out_mean_mfccs, true);
    }
    SS_CUDA(ctx, st->d_samples.reserve(n));
    const double denom = (double)(INT32_MAX >> (32 - bits_per_sample));  // src/sound.rs:118-120
    if (n) {
        if (bits_per_sample == 16) {
            SS_CUDA(ctx, st->d_pcm.reserve((n + 1) / 2));  // int16 samples packed in the int32 staging buffer
            SS_CUDA(ctx, cudaMemcpyAsync(st->d_pcm.p, pcm, n * sizeof(int16_t), cudaMemcpyHostToDevice, ctx->stream));
            k_decode_pcm16<<<ceil_div((long long)n, 256), 256, 0, ctx->stream>>>(reinterpret_cast<const int16_t*>(st->d_pcm.p), n, denom,
                                                                               st->d_samples.p);
        } else {
            SS_TRY(upload(ctx, st->d_pcm, static_cast<const int32_t*>(pcm), n));
            k_decode_pcm<<<ceil_div((long long)n, 256), 256, 0, ctx->stream>>>(st->d_pcm.p, n, denom, st->d_samples.p);
        }
        SS_LAUNCHED(ctx);
        if (out_samples) SS_CUDA(ctx, cudaMemcpyAsync(out_samples, st->d_samples.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    return analyze_resident(ctx, st, n, sample_rate, ncoeffs, out_mfcc, out_frames, out_max_power, out_mean_mfccs);
}

int ss_sound_analyze_batch(ss_ctx* ctx, const double* samples, const uint64_t* sample_offsets, size_t nsounds, double sample_rate, int ncoeffs,
                           double* out_mfcc, uint64_t* out_frame_offsets, double* out_max_power, double* out_mean_mfccs) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    SS_TRY(check_c(ctx, ncoeffs));
    if (!sample_offsets || !out_frame_offsets) return set_error(ctx, SS_ERR_INVALID, "sample_offsets / out_frame_offsets is NULL");
    if (nsounds >= 0xFFFFFFFFull) return set_error(ctx, SS_ERR_INVALID, "too many sounds");
    if (sample_offsets[0] != 0) return set_error(ctx, SS_ERR_INVALID, "sample_offsets[0] must be 0");
    std::vector<uint64_t> foff(nsounds + 1, 0), poff(nsounds + 1, 0);
    for (size_t i = 0; i < nsounds; i++) {
        if (sample_offsets[i + 1] < sample_offsets[i]) return set_error(ctx, SS_ERR_INVALID, "sample_offsets must be non-decreasing");
        const size_t n = sample_offsets[i + 1] - sample_offsets[i];
        size_t fr = 0;
        ss_frame_count(n, &fr);
        foff[i + 1] = foff[i] + fr;
        poff[i + 1] = poff[i] + (n >= 128 ? (n - 128) / 64 + 1 : 0);
    }
    memcpy(out_frame_offsets, foff.data(), (nsounds + 1) * sizeof(uint64_t));
    const size_t n = sample_offsets[nsounds], frames = foff[nsounds], pframes = poff[nsounds];
    if (n && !samples) return set_error(ctx, SS_ERR_INVALID, "samples is NULL");
    if (!nsounds) return SS_OK;
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SoundState* st = sound_state(ctx);
    SS_TRY(upload(ctx, st->d_samples, samples, n));
    SS_TRY(upload(ctx, st->d_off_a, sample_offsets, nsounds + 1));
    const bool want_mfcc = (out_mfcc || out_mean_mfccs) && frames;
    if (want_mfcc) {
        SS_TRY(upload(ctx, st->d_off_b, foff.data(), nsounds + 1));
        SS_CUDA(ctx, st->d_mfcc.reserve(frames * (size_t)ncoeffs));
        SoundTables* t = nullptr;
        SS_TRY(get_tables(ctx, sample_rate, ncoeffs, &t));
        const int grid = (int)std::min<size_t>((frames + kMfccWarps - 1) / kMfccWarps, (size_t)ctx->sm_count * 4 * SS_MFCC_MINBLOCKS);
        const int pw_len = (t->bins[ncoeffs + 1] + 32) & ~31;
        const int smem = (int)(sizeof(double2) * kMfccWarps * kHalf + sizeof(double) * kMfccWarps * pw_len + sizeof(double) * kMfccWarps * 16);
        SS_CUDA(ctx, cudaFuncSetAttribute(k_mfcc, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        k_mfcc<<<grid, kMfccWarps * 32, smem, ctx->stream>>>(st->d_samples.p, frames, mfcc_tabs(t), ncoeffs, pw_len, 1e-10, st->d_mfcc.p, st->d_off_b.p,
                                                             st->d_off_a.p, (uint32_t)nsounds);
        SS_LAUNCHED(ctx);
        if (out_mfcc)
            SS_CUDA(ctx, cudaMemcpyAsync(out_mfcc, st->d_mfcc.p, frames * (size_t)ncoeffs * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    if (out_mean_mfccs) {
        if (!frames) SS_TRY(upload(ctx, st->d_off_b, foff.data(), nsounds + 1));
        SS_CUDA(ctx, st->d_partial.reserve(nsounds * (size_t)ncoeffs));
        k_mean_batch<<<ceil_div((long long)nsounds * ncoeffs, 128), 128, 0, ctx->stream>>>(st->d_mfcc.p, st->d_off_b.p, (uint32_t)nsounds, ncoeffs,
                                                                                         st->d_partial.p);
        SS_LAUNCHED(ctx);
        SS_CUDA(ctx, cudaMemcpyAsync(out_mean_mfccs, st->d_partial.p, nsounds * (size_t)ncoeffs * sizeof(double), cudaMemcpyDeviceToHost,
                                     ctx->stream));
    }
    if (out_max_power) {
        static_assert(sizeof(unsigned long long) == sizeof(double), "max power travels as the bit pattern of a non-negative double");
        SS_CUDA(ctx, st->d_maxbits.reserve(nsounds));
        SS_CUDA(ctx, cudaMemsetAsync(st->d_maxbits.p, 0, nsounds * sizeof(unsigned long long), ctx->stream));
        if (pframes) {
            DevBuf<uint64_t>& d_poff = st->d_off_pf;
            SS_TRY(upload(ctx, d_poff, poff.data(), nsounds + 1));
            k_max_power_batch<<<ceil_div((long long)pframes, 128), 128, 0, ctx->stream>>>(st->d_samples.p, st->d_off_a.p, d_poff.p, (uint32_t)nsounds,
                                                                                         pframes, st->d_maxbits.p);
            SS_LAUNCHED(ctx);
        }
        SS_CUDA(ctx, cudaMemcpyAsync(out_max_power, st->d_maxbits.p, nsounds * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // host staging vectors (foff, poff) go out of scope
    return SS_OK;
}

int ss_mfcc(ss_ctx* ctx, const double* samples, size_t n, double sample_rate, int ncoeffs, double* out_mfcc, size_t* out_frames) {
    return ss_sound_analyze(ctx, samples, n, sample_rate, ncoeffs, out_mfcc, out_frames, nullptr, nullptr);
}

int ss_max_power(ss_ctx* ctx, const double* samples, size_t n, double* out) {
    if (!out) return set_error(ctx, SS_ERR_INVALID, "out is NULL");
    return ss_sound_analyze(ctx, samples, n, 44100.0, SS_NCOEFFS, nullptr, nullptr, out, nullptr);
}

int ss_resynth(ss_ctx* ctx, const double* dict_samples, const uint64_t* dict_sample_offsets, size_t ndict, const uint32_t* match_idx,
               const uint64_t* target_lens, size_t nseg, double* out_samples) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (!nseg) return SS_OK;
    if (!dict_sample_offsets || !match_idx || !target_lens || !out_samples) return set_error(ctx, SS_ERR_INVALID, "NULL buffer");
    if (!ndict) return set_error(ctx, SS_ERR_EMPTY_DICT, "resynthesis from an empty dictionary");
    for (size_t i = 0; i < ndict; i++)
        if (dict_sample_offsets[i + 1] < dict_sample_offsets[i]) return set_error(ctx, SS_ERR_INVALID, "dictionary offsets not monotone at %zu", i);
    std::vector<uint64_t> out_off(nseg + 1, 0);
    for (size_t i = 0; i < nseg; i++) {
        if (match_idx[i] >= ndict) return set_error(ctx, SS_ERR_INVALID, "match_idx[%zu] = %u out of range", i, match_idx[i]);
        out_off[i + 1] = out_off[i] + target_lens[i];
    }
    const size_t total = out_off[nseg], dtotal = dict_sample_offsets[ndict];
    if (!total) return SS_OK;
    if (dtotal && !dict_samples) return set_error(ctx, SS_ERR_INVALID, "dict_samples is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SoundState* st = sound_state(ctx);
    SS_TRY(upload(ctx, st->d_samples, dict_samples, dtotal));
    SS_TRY(upload(ctx, st->d_off_a, dict_sample_offsets, ndict + 1));
    SS_TRY(upload(ctx, st->d_off_b, out_off.data(), nseg + 1));
    SS_TRY(upload(ctx, st->d_idx, match_idx, nseg));
    SS_CUDA(ctx, st->d_mfcc.reserve(total));
    const int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)ctx->sm_count * 16);
    k_resynth<<<grid, 256, 0, ctx->stream>>>(st->d_samples.p, st->d_off_a.p, st->d_idx.p, st->d_off_b.p, nseg, total, st->d_mfcc.p);
    SS_LAUNCHED(ctx);
    SS_CUDA(ctx, cudaMemcpyAsync(out_samples, st->d_mfcc.p, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SS_OK;
}

int ss_resynth_warped(ss_ctx* ctx, const double* dict_samples, const uint64_t* dict_sample_offsets, size_t ndict, const uint32_t* match_idx,
                      const uint32_t* paths, const uint64_t* path_offsets, const uint64_t* target_lens, size_t nseg, double* out_samples) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (!nseg) return SS_OK;
    if (!dict_sample_offsets || !match_idx || !path_offsets || !target_lens || !out_samples) return set_error(ctx, SS_ERR_INVALID, "NULL buffer");
    if (!ndict) return set_error(ctx, SS_ERR_EMPTY_DICT, "resynthesis from an empty dictionary");
    for (size_t i = 0; i < ndict; i++)
        if (dict_sample_offsets[i + 1] < dict_sample_offsets[i]) return set_error(ctx, SS_ERR_INVALID, "dictionary offsets not monotone at %zu", i);
    if (path_offsets[0] != 0) return set_error(ctx, SS_ERR_INVALID, "path_offsets[0] must be 0");
    std::vector<uint64_t> out_off(nseg + 1, 0);
    for (size_t t = 0; t < nseg; t++) {
        if (match_idx[t] >= ndict) return set_error(ctx, SS_ERR_INVALID, "match_idx[%zu] = %u out of range", t, match_idx[t]);
        if (path_offsets[t + 1] < path_offsets[t]) return set_error(ctx, SS_ERR_INVALID, "path offsets not monotone at %zu", t);
        out_off[t + 1] = out_off[t] + target_lens[t];
    }
    const size_t cells = path_offsets[nseg];
    if (cells && !paths) return set_error(ctx, SS_ERR_INVALID, "paths is NULL");
    for (size_t t = 0; t < nseg; t++) {  // each path runs from (0, 0) in steps (1, 0), (0, 1) or (1, 1): what the kernel's search relies on
        const uint64_t p0 = path_offsets[t], p1 = path_offsets[t + 1];
        if (p0 == p1) continue;
        if (paths[2 * p0] != 0 || paths[2 * p0 + 1] != 0) return set_error(ctx, SS_ERR_INVALID, "path %zu does not start at (0, 0)", t);
        for (uint64_t e = p0 + 1; e < p1; e++) {
            const uint32_t di = paths[2 * e] - paths[2 * e - 2], dj = paths[2 * e + 1] - paths[2 * e - 1];
            if (di > 1 || dj > 1 || (di | dj) == 0)
                return set_error(ctx, SS_ERR_INVALID, "path %zu: step %llu -> %llu is not (1, 0), (0, 1) or (1, 1)", t,
                                 (unsigned long long)(e - 1 - p0), (unsigned long long)(e - p0));
        }
    }
    const size_t total = out_off[nseg], dtotal = dict_sample_offsets[ndict];
    if (!total) return SS_OK;
    if (dtotal && !dict_samples) return set_error(ctx, SS_ERR_INVALID, "dict_samples is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SoundState* st = sound_state(ctx);
    SS_TRY(upload(ctx, st->d_samples, dict_samples, dtotal));
    SS_TRY(upload(ctx, st->d_off_a, dict_sample_offsets, ndict + 1));
    SS_TRY(upload(ctx, st->d_off_b, out_off.data(), nseg + 1));
    SS_TRY(upload(ctx, st->d_idx, match_idx, nseg));
    SS_TRY(upload(ctx, st->d_path_off, path_offsets, nseg + 1));
    SS_TRY(upload(ctx, st->d_path, reinterpret_cast<const uint2*>(paths), cells));
    SS_CUDA(ctx, st->d_mfcc.reserve(total));
    const int grid = (int)std::min<size_t>((total + 255) / 256, (size_t)ctx->sm_count * 16);
    k_resynth_warped<<<grid, 256, 0, ctx->stream>>>(st->d_samples.p, st->d_off_a.p, st->d_idx.p, st->d_path.p, st->d_path_off.p, st->d_off_b.p, nseg,
                                                    total, st->d_mfcc.p);
    SS_LAUNCHED(ctx);
    SS_CUDA(ctx, cudaMemcpyAsync(out_samples, st->d_mfcc.p, total * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SS_OK;
}

}  // extern "C"
