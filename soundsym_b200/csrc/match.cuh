// match.cuh — HBM-resident dictionary / query-batch handles shared by the DTW (dtw.cu) and cosine-ref (cosine.cu) matchers.
#pragma once
#include <cuda_fp16.h>

#include <chrono>
#include <map>
#include <memory>

#include "common.cuh"

namespace ss {

// ---- layout constants of the DTW scan -----------------------------------------------------------------------------
constexpr int kSlots = 16;        // floats per frame in the fp32 scan layouts (13 coefficient slots + norm slot + pad)
constexpr int kNormSlot = 13;     // stream side: |b|^2 ; lane side: 1.0f
constexpr int kLaneNaSlot = 14;   // lane side: |a|^2 (accumulator seed)
constexpr int kStrip = 32;        // DP columns held in registers per strip
constexpr int kTileFrames = 128;  // frames per TMA tile (8 KB)
constexpr int kStages = 3;        // tile ring depth
constexpr int kWarpsPerCta = 4;
constexpr int kMaxKeep = 32;      // largest candidate list per query kept by a scan

// the stages of an SS_DTW match, in cascade order (dtw.cu)
enum class DtwStage { H2, H2_WIDE, TC, FP32, EXHAUSTIVE };

struct StripDesc {  // 16 B, read as int4
    uint32_t frame_begin;  // first frame of the strip in the shard's frame stream
    uint32_t seg;          // local segment index
    uint32_t len_flags;    // bits 0..15 frames in strip (1..32), bit 16 first strip of its segment, bit 17 last
    uint32_t seg_len;      // frames of the whole segment
};
struct TileDesc {  // 16 B, read as int4
    uint32_t frame_begin, nframes, strip_begin, nstrips;
};

}  // namespace ss

struct ss_dict {
    ss_ctx* ctx = nullptr;
    size_t nseg = 0;
    int c = 0;
    uint32_t index_base = 0;
    uint64_t total_frames = 0;
    uint32_t max_len = 0;
    std::vector<uint64_t> h_off;  // nseg+1, frames
    ss::DevBuf<double> d_mfcc;    // frames x c (f64, as given)
    ss::DevBuf<uint64_t> d_off;   // nseg+1
    // cosine-ref
    ss::DevBuf<double> d_norm;  // per segment: norm(mfccs) (src/sound.rs:36-38)
    std::vector<uint64_t> h_len_sorted, h_len_prefix;  // work accounting (sum of min(Kq, Kd)), built on first use
    ss::DevBuf<uint4> d_cos_seg;     // the cosine scan's walk order: {first frame lo, hi, frames, index} by (length, index)
    ss::DevBuf<double> d_cos_norm;   // d_norm in that order
    std::vector<uint4> h_cos_seg;    // host copy (source of the asynchronous upload)
    // DTW scan
    ss::DevBuf<float> d_stream;  // frames x kSlots
    ss::DevBuf<int4> d_strips, d_tiles;
    uint32_t nstrips = 0, ntiles = 0;
    std::vector<uint32_t> h_tile_frames;    // frames per tile (slice balancing)
    std::vector<uint8_t> h_tile_segstart;   // 1 if the tile begins at a segment boundary
    ss::DevBuf<float> d_max_norm;           // [0] = max |b|^2 over the shard (error bound of the fp32 scan)
    // per-call workspaces (grow-only)
    ss::DevBuf<uint32_t> d_slice_tile;
    ss::DevBuf<unsigned long long> d_partial;
    ss::DevBuf<float> d_scratch;
    ss::DevBuf<uint32_t> d_cand_idx;
    ss::DevBuf<float> d_cand_adist;
    ss::DevBuf<double> d_cand_exact;
    ss::DevBuf<double> d_rescore_rows;
    ss::DevBuf<double> d_second_bnd;  // boundary rows of the long second-chance kernel (exact.cu)
    ss::DevBuf<unsigned long long> d_counters;  // [0] uncertified
    std::vector<uint32_t> h_slice_tile;
    uint64_t last_work = 0;         // work of the last match (SS_DTW: dictionary frames x query frames, the first stage's cells)
    uint64_t last_uncertified = 0;  // queries of the last match whose rows are not final (0 unless a stage failed)
    uint64_t last_tc_fallback = 0;  // queries of the last match that its first stage, a tensor-core scan, left uncertified
    uint64_t last_exhaustive = 0;   // queries of the last match sent to the exhaustive f64 stage
    ss::DevBuf<double> d_exh_dist;
    ss::DevBuf<uint32_t> d_exh_qid;
    cudaEvent_t ev_scan0 = nullptr, ev_scan1 = nullptr;  // around the first stage's scan of the last match
    bool scan_timed = false;
    int last_scan_kind = 0;    // first-stage scan of the last match: 1 packed-half tensor-core, 2 fp32-DP tensor-core, 3 fp32 CUDA-core, 4 cosine-ref
    // tensor-core scan (dtw_tc.cu): fp16 UMMA tiles of 4 segment slots x 32 columns, segments sorted by length
    bool tc_ready = false;
    bool tc_stats_ready = false;             // mean frame, norm scale, max norms (both tensor-core scans)
    float tc_max_nb = 0.f, tc_max_abs = 0.f;  // max |fp16(b - mu)|^2, max |fp16(b - mu)|
    uint64_t tc_serial = 0;                  // identifies this build of the tiles (query A blocks are keyed on it)
    uint32_t tc_ntiles = 0;
    uint32_t tc_first_pair_tile = 0;         // tiles [0, first_pair) hold one segment per slot, the rest two short ones
    float tc_nb_scale = 1.f;                 // power of two s: the |b|^2 columns hold |b|^2 / s
    ss::DevBuf<double> d_mu;                 // per-coefficient mean of the dictionary frames (both sides are centred on it)
    ss::DevBuf<uint16_t> d_tc_tiles;         // ntiles x 4 KB
    ss::DevBuf<int4> d_tc_desc;              // ntiles x 2 = four {segment, length} pairs per tile
    std::vector<uint32_t> h_tc_tile_frames;  // per tile: instruction estimate of one pipeline step (slice balancing)
    ss::DevBuf<unsigned long long> d_tc_partial;
    ss::DevBuf<float> d_tc_max_norm;         // [0] = max |fp16(b - mu)|^2
    // packed-half tensor-core scan (dtw_h2.cu): tiles of 2 slots x 64 TMEM columns, two interleaved segments per register
    bool h2_ready = false;
    uint32_t h2_ntiles = 0;
    uint32_t h2_first_tile[4] = {0, 0, 0, 0};   // first tile of the kinds NB = 1, 2, 4 (launch order) and the total
    // slice tables of the packed-half scan, cached per number of query groups (the main batch and the one-group re-run of
    // its uncertified queries alternate within a match)
    struct H2Slices {
        uint32_t kind_slice[4] = {0, 0, 0, 0};  // first slice of the kinds NB = 1, 2, 4 and the total
        ss::DevBuf<uint32_t> d_slice_tile;
    };
    std::map<uint32_t, std::unique_ptr<H2Slices>> h2_slices;
    float h2_s = 1.f;                           // power-of-two cost scale S of the current match (h2_cost_scale)
    float h2_s0 = 1.f;                          // S for paths of <= 64 cells (from the dictionary's largest frame norm)
    float h2_bmax = 0.f;                        // max |fp16(b - mu)| (bound's eta)
    double h2_bound_inv_s = 1.0;
    std::vector<uint32_t> h_h2_tile_cost;
    std::vector<uint8_t> h_h2_tile_cont;        // 1 if the tile continues the previous one (a later strip of the same long segments)
    bool h2_has_strips = false;
    ss::DevBuf<__half2> d_h2_bnd;               // boundary-column scratch of the long kernel, [192 SM ids][rows][256]
    uint32_t h2_nsmid = 0;                      // %nsmid of the device
    ss::DevBuf<uint16_t> d_h2_tiles;
    ss::DevBuf<int4> d_h2_desc;
    ss::DevBuf<unsigned long long> d_h2_timeline;  // SS_DTW_H2_TIMELINE measurement hook
    ss::DevBuf<unsigned long long> d_h2_thr;   // per query slot: running bound on the global KP-th key (dtw_h2.cu)
    uint32_t dtw_band = 0;  // Sakoe-Chiba radius of the exact DTW stages and of ss_dict_align (ss_dict_set_dtw_band); 0 = no band
    int scan_pref = 0;  // test / A-B hook (ss_dict_set_scan): 0 = packed-half scan first, 1 = start at the fp32 tensor-core scan, 2 = fp32 CUDA-core scan, 3 = packed-half scan without its second chance
    // the last SS_DTW match is asynchronous up to its fallback decision: ss::dtw_match_finish waits for ev_done, reads the
    // uncertified count from pinned memory and runs the later stages for the queries that need them
    struct Pending {
        bool active = false;
        ss::DtwStage first = ss::DtwStage::FP32;  // the stage dtw_match_dev ran on the whole batch
        struct ss_queries* q = nullptr;
        int k = 0;
        uint32_t* d_out_idx = nullptr;
        double* d_out_dist = nullptr;
    } pending;
    unsigned long long* h_counters = nullptr;  // pinned, 4 entries: [0] uncertified queries, [1] extra candidates refined
    cudaEvent_t ev_done = nullptr;
    ss::DevBuf<uint32_t> d_tc_slice_tile;       // the tensor-core scan's own slice table (cached)
    uint32_t slice_for_groups = 0xFFFFFFFFu;  // tc_ngroups the cached slice table (d_slice_tile / h_slice_tile) was built for
    uint32_t tc_nsingle = 0, tc_nslices = 0;
    // the few queries a stage could not certify, as a batch of their own for the next stage (dtw.cu gather_queries)
    struct ss_queries* sub_q = nullptr;
    ss::DevBuf<uint32_t> d_sub_ids, d_sub_idx;
    ss::DevBuf<double> d_sub_dist;
    // host-buffer entry point (ss_dict_match): query batch + result buffers reused across calls (grow-only)
    struct ss_queries* scratch_q = nullptr;
    ss::DevBuf<uint32_t> d_res_idx;
    ss::DevBuf<double> d_res_dist, d_res_targets;
    // ss_dict_walk (exact.cu cosine_walk_dev): its own buffers, so that a walk never touches a match's workspaces or the
    // last_* counters. state = {ticket of the last-CTA reduction, local index of the next step's query}
    ss::DevBuf<double> d_walk_part_dist, d_walk_qnorm;
    ss::DevBuf<uint32_t> d_walk_part_idx, d_walk_state;
    ss::DevBuf<double> d_walk_start, d_walk_targets, d_walk_dist;  // host-buffer entry point: start frames, targets, results
    ss::DevBuf<uint64_t> d_walk_off;
    ss::DevBuf<uint32_t> d_walk_idx;
    uint64_t h_walk_off[2] = {0, 0};
    // ss_dict_align (exact.cu dtw_align_dev): staging slots of the paths, path lengths, direction blocks and boundary rows of
    // the long pairs, the scan's temporary storage; then the host-buffer entry point's inputs and outputs
    ss::DevBuf<uint2> d_align_stage;
    ss::DevBuf<uint64_t> d_align_len, d_align_dir;
    ss::DevBuf<double> d_align_bnd;
    ss::DevBuf<unsigned char> d_align_cub;
    ss::DevBuf<double> d_align_q, d_align_dist;
    ss::DevBuf<uint64_t> d_align_qoff, d_align_off;
    ss::DevBuf<uint32_t> d_align_seg, d_align_path;
    ~ss_dict();
};

struct ss_queries {
    ss_ctx* ctx = nullptr;
    size_t nq = 0;
    size_t nonempty = 0;  // queries with at least one frame
    int c = 0;
    uint64_t total_frames = 0;
    uint32_t max_len = 0;
    std::vector<uint64_t> h_off;
    ss::DevBuf<double> d_mfcc;
    ss::DevBuf<uint64_t> d_off;
    ss::DevBuf<double> d_norm;  // cosine-ref: norm of every query
    // lane layout: queries sorted by length (descending) into length-homogeneous groups of 32 lanes
    uint32_t ngroups = 0;
    uint64_t total_rows = 0;  // sum over groups of padded row counts
    std::vector<uint32_t> h_group_len;
    ss::DevBuf<uint32_t> d_group_len, d_group_rowbase, d_group_qid;  // qid: ngroups x 32, 0xFFFFFFFF = padding lane
    ss::DevBuf<float4> d_lane;                                       // [row][4][32] float4 (DTW)
    ss::DevBuf<float> d_max_norm;                                    // [0] = max |a|^2
    ss::DevBuf<double> d_lane64;                                     // [row*c + e][32] f64 (cosine-ref), built on first use
    ss::DevBuf<uint2> d_cos_items;                                   // cosine-ref work items: {g0, g1} pairs of one length, then single groups
    uint32_t cos_npairs = 0, cos_nsingles = 0;
    bool cos_built = false;
    bool lane_built = false;
    // tensor-core scan: groups of 128 (nearly) equal-length queries. The grouping only depends on the lengths: it is built
    // (host counting sort + uploads) when the batch is filled; the fp16 A blocks depend on the dictionary and are built by
    // the first match against it.
    bool tc_grouped = false;
    bool tc_built = false;
    uint64_t tc_dict_serial = 0;             // ss_dict::tc_serial the A blocks were built for
    uint64_t tc_a_bytes = 0;
    bool h2_built = false;                   // the packed-half scan's A blocks (the same rows scaled by S)
    uint64_t h2_dict_serial = 0;
    float h2_s_built = 0.f;                  // the cost scale S those A blocks carry
    ss::DevBuf<unsigned char> d_h2_a;
    uint32_t tc_ngroups = 0;
    std::vector<uint32_t> h_tc_group_len;
    ss::DevBuf<uint32_t> d_tc_group_len, d_tc_qid, d_tc_slot_len;  // qid / slot_len: ngroups x 128
    ss::DevBuf<uint64_t> d_tc_group_off;            // byte offset of each group's block of L x 4 KB A tiles
    ss::DevBuf<unsigned char> d_tc_a;
    ss::DevBuf<float> d_tc_max_norm;                // [0] = max |fp16(a - mu)|^2
    ss::DevBuf<float> d_tc_slot_max_na;             // per query slot: max over its rows of |fp16(a - mu)|^2
    ss::DevBuf<uint8_t> d_uncert_flag;              // per query: 1 if the last stage run on the batch could not certify its top-k
};

inline ss_dict::~ss_dict() {
    if (ev_scan0) cudaEventDestroy(ev_scan0);
    if (ev_scan1) cudaEventDestroy(ev_scan1);
    if (ev_done) cudaEventDestroy(ev_done);
    if (h_counters) {
        if (ctx) ctx->pinned_free.push_back(h_counters);
        else cudaFreeHost(h_counters);
    }
    delete scratch_q;
    delete sub_q;
}

namespace ss {
// SS_DTW_TRACE=1: wall-clock of a match's steps and the stages it takes, on stderr (each step is followed by a stream synchronisation)
inline bool dtw_trace() {
    static const bool on = [] {
        const char* e = getenv("SS_DTW_TRACE");
        return e && atoi(e) != 0;
    }();
    return on;
}
struct TraceTimer {
    ss_ctx* ctx;
    std::chrono::steady_clock::time_point t0;
    explicit TraceTimer(ss_ctx* c) : ctx(c), t0(std::chrono::steady_clock::now()) {}
    void lap(const char* what) {
        if (!dtw_trace()) return;
        cudaStreamSynchronize(ctx->stream);
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[ss dtw trace] %-28s %8.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

// Sakoe-Chiba band (A10, DESIGN.md §3.1f): the rows [*lo, *hi] of column j (0 <= j < lb; la, lb >= 1) that lie inside the band
// of radius r >= 1, |i (lb - 1) - j (la - 1)| <= r max(la - 1, lb - 1). Both ends are monotone in j. r is capped at max(la, lb),
// beyond which the band covers the whole matrix anyway, so that the products stay inside 64 bits. The exact kernels (exact.cu)
// and the host's cost estimate of the exhaustive stage (dtw.cu) use the same rows.
__host__ __device__ __forceinline__ void band_rows(int j, int la, int lb, uint32_t r, int* lo, int* hi) {
    const long long A = lb - 1, B = la - 1;
    if (A == 0) {  // one column: every row
        *lo = 0, *hi = la - 1;
        return;
    }
    const long long rr = r < (uint32_t)(la > lb ? la : lb) ? r : (la > lb ? la : lb);
    const long long w = rr * (A > B ? A : B), x = (long long)j * B;
    *lo = x - w <= 0 ? 0 : (int)((x - w + A - 1) / A);
    const long long h = (x + w) / A;
    *hi = h < la - 1 ? (int)h : la - 1;
}

int dtw_dict_build(ss_dict* d);       // builds the fp32 stream + strip / tile tables (dtw.cu)
int dtw_tc_dict_build(ss_dict* d);    // builds the fp16 UMMA tiles (dtw_tc.cu)
int dtw_queries_build(ss_queries* q); // builds the lane layout (dtw.cu)
int dtw_tc_queries_group(ss_queries* q);  // length-sorted groups of 128 for the tensor-core scan (dtw_tc.cu); no-op for long queries
// asynchronous on the ctx stream up to the fallback decision; dtw_match_finish completes it (a no-op when nothing is pending)
int dtw_match_dev(ss_dict* d, ss_queries* q, int k, uint32_t* d_out_idx, double* d_out_dist);
int dtw_match_finish(ss_dict* d);
int dtw_h2_dict_build(ss_dict* d);    // builds the interleaved fp16 tiles of the packed-half scan (dtw_h2.cu; after dtw_tc_dict_build)
int dtw_h2_debug_scan(ss_dict* d, ss_queries* q, float* d_out, std::vector<uint32_t>* slot_qid, double* mu16, float* scale, float* s_out);
int dtw_tc_debug_scan(ss_dict* d, ss_queries* q, float* d_out, std::vector<uint32_t>* slot_qid, double* mu16, float* scale);
int queries_check(ss_ctx* ctx, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int ncoeffs);  // capi.cu
int queries_prepare(ss_queries* q, const uint64_t* q_frame_offsets, size_t nq);
int queries_fill(ss_queries* q, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq);
int fill_result(ss_ctx* ctx, uint32_t* d_idx, double* d_dist, size_t n);  // (inf, 0xFFFFFFFF) rows (exact.cu)
int cosine_dict_build(ss_dict* d);    // per-segment norms (cosine.cu)
int cosine_queries_build(ss_queries* q);
int cosine_match_dev(ss_dict* d, ss_queries* q, const double* d_targets, uint32_t* d_out_idx, double* d_out_dist);
// SoundSequence::from_distances for SS_COSINE_REF: nsteps + 1 launches on the ctx stream, no host synchronisation (exact.cu)
int cosine_walk_dev(ss_dict* d, const double* d_start, const uint64_t* d_start_off, const double* d_targets, size_t nsteps,
                    uint32_t* d_out_idx, double* d_out_dist);
// the DTW warping path (DESIGN.md §3.1e) of query p (frames d_qoff[p] .. d_qoff[p+1], h_qoff its host copy) against segment
// d_seg_idx[p]: 1 + (waves of long pairs) + 2 launches on the ctx stream, no host synchronisation (exact.cu). d_out_path must
// hold sum over non-empty queries of (Lq + max(longest segment, 1) - 1) (i, j) pairs.
int dtw_align_dev(ss_dict* d, const double* d_qmfcc, const uint64_t* d_qoff, const uint64_t* h_qoff, size_t nq, const uint32_t* d_seg_idx,
                  uint32_t* d_out_path, uint64_t* d_out_off, double* d_out_dist);
int topk_merge_dev(ss_ctx* ctx, const uint32_t* d_idx, const double* d_dist, int nlists, size_t nq, int k,
                   uint32_t* d_out_idx, double* d_out_dist);
}  // namespace ss
