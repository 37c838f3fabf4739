/* soundsym_b200.h — C ABI of the B200-native soundsym hot path (MFCC -> segmentation -> dictionary matching).
 *
 * The reference (andrewcsmith/soundsym, Rust) has no FFI of its own; its boundary for this path is the crate's public
 * API (src/lib.rs:30 re-exports, src/lib.rs:32-210, src/sound.rs:71-506). Each entry point below names the reference
 * function(s) whose body it replaces; INTEGRATION.md shows the `extern "C"` block and the thin Rust shim that keeps the
 * original signatures on top of it.
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns SS_OK (0) or a negative ss_status; no exceptions cross.
 *   - ss_last_error(ctx) returns a ctx-owned NUL-terminated string (maps to CosError(&'static str), src/lib.rs:181-198,
 *     or Box<Error> on the Rust side). With ctx == NULL it returns the calling thread's last context-less error.
 *   - "host" entry points take HOST buffers (the reference hands out &Vec<f64>, so results must live in host f64
 *     memory); the library does H2D / D2H itself and is stream-synchronised on return.
 *   - "_dev" entry points take DEVICE pointers on the ctx's device and are asynchronous on ss_ctx_stream(ctx); they
 *     exist so a caller (bench.py, a multi-GPU driver) can keep data resident in HBM and time kernels with events.
 *   - an ss_ctx is bound to one device and one stream and is NOT thread-safe; handles created from a ctx
 *     (ss_dict, ss_queries) must be destroyed before it.
 *   - there is no CPU fallback anywhere: without a CUDA device ss_ctx_create fails with SS_ERR_CUDA.
 */
#ifndef SOUNDSYM_B200_H
#define SOUNDSYM_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum ss_status {
    SS_OK = 0,
    SS_ERR_INVALID = -1,     /* bad argument (NULL, ncoeffs out of range, offsets not monotone, k out of range ...) */
    SS_ERR_CUDA = -2,        /* CUDA runtime error; text in ss_last_error */
    SS_ERR_NOMEM = -3,       /* device or host allocation failed */
    SS_ERR_NOT_TRAINED = -4, /* model == NULL: CosError("Must first train model"), src/lib.rs:140-142 */
    SS_ERR_EMPTY_DICT = -5,  /* match against an empty dictionary (the reference indexes sounds[0] and panics, src/sound.rs:369) */
    SS_ERR_TOO_FEW_ROWS = -6 /* Standardizer needs >= 2 rows (rusty-machine returns Err; src/lib.rs:57-58 unwraps) */
} ss_status;

/* constants of the reference, src/lib.rs:22-25 */
#define SS_NCOEFFS 12
#define SS_NCLUSTERS 26
#define SS_HOP 256
#define SS_BIN 1024
#define SS_F_LO 100.0  /* src/sound.rs:218 */
#define SS_F_HI 8000.0 /* src/sound.rs:218 */
#define SS_MAX_NCOEFFS 13
#define SS_MAX_TOPK 8

typedef enum ss_match_mode {
    SS_COSINE_REF = 0, /* the reference's matcher: cosine_sim + at_distance, src/sound.rs:23-38, 351-370 (bit-exact f64) */
    SS_DTW = 1,        /* north-star extension (no reference counterpart): DTW, spec in oracle/ASSUMPTIONS.h A8 */
    SS_DTW_TARGET = 2  /* at_distance with the DTW distance: the k sounds whose SS_DTW distance is closest to a target (A13) */
} ss_match_mode;

typedef struct ss_ctx ss_ctx;         /* device + stream + workspace */
typedef struct ss_dict ss_dict;       /* a dictionary (or one shard of it) resident in HBM */
typedef struct ss_queries ss_queries; /* a prepared, HBM-resident batch of query segments */

/* GaussianMixtureModel as train_model returns it (src/lib.rs:44-54): row-major host arrays. */
typedef struct ss_gmm {
    int ncomp;             /* NCLUSTERS = 26 */
    int ncoeffs;           /* NCOEFFS = 12 */
    const double* means;   /* ncomp x ncoeffs */
    const double* covs;    /* ncomp x ncoeffs x ncoeffs */
    const double* weights; /* ncomp */
} ss_gmm;

/* ---- context ---------------------------------------------------------------------------------------------------- */
int ss_ctx_create(int device, ss_ctx** out);
void ss_ctx_destroy(ss_ctx* ctx);
const char* ss_last_error(const ss_ctx* ctx);
void* ss_ctx_stream(ss_ctx* ctx);   /* the cudaStream_t all work of this ctx is ordered on */
int ss_ctx_sync(ss_ctx* ctx);       /* cudaStreamSynchronize */
int ss_ctx_device(const ss_ctx* ctx);
/* number of this library's kernels launched through ctx since creation (bench.py reports it as gpu_launches) */
uint64_t ss_ctx_launch_count(const ss_ctx* ctx);
const char* ss_version(void);

/* ---- Sound: MFCC subsystem ------------------------------------------------------------------------------------------
 * ss_frame_count   framing rule of sample::window::Windower as used at src/sound.rs:228-229 (full frames only).
 * ss_decode_pcm    Sound::from_path's sample conversion, src/sound.rs:118-120: s / (i32::MAX >> (32 - bits)).
 * ss_sound_analyze Sound::from_samples, src/sound.rs:92-112 = analyze_mfccs (:215-242) + analyze_max_power (:244-256)
 *                  + analyze_mean_mfccs (:271-286) with one upload of the samples. Any output pointer may be NULL.
 *                  out_mfcc capacity >= frames * ncoeffs. Sound::push_samples (:145-164) calls this on
 *                  samples[initial_frames*HOP ..] and appends.
 * ss_mfcc / ss_max_power   the two analyses on their own.
 */
int ss_frame_count(size_t n, size_t* out_frames);
int ss_decode_pcm(ss_ctx* ctx, const int32_t* pcm, size_t n, int bits_per_sample, double* out_samples);
int ss_sound_analyze(ss_ctx* ctx, const double* samples, size_t n, double sample_rate, int ncoeffs, double* out_mfcc,
                     size_t* out_frames, double* out_max_power, double* out_mean_mfccs);
/* ss_sound_analyze_pcm   Sound::from_path in one call (SURVEY.md §8f item 2): integer PCM in (bits 16 -> an int16_t buffer,
 *                        24 / 32 -> an int32_t buffer), so the host->device copy is 2 or 4 bytes per sample instead of 8;
 *                        the s / (i32::MAX >> (32 - bits)) conversion (src/sound.rs:118-120) runs on the device, then the
 *                        three analyses. out_samples (n doubles, the Sound's `samples` Vec) may be NULL. */
int ss_sound_analyze_pcm(ss_ctx* ctx, const void* pcm, size_t n, int bits_per_sample, double sample_rate, int ncoeffs,
                         double* out_samples, double* out_mfcc, size_t* out_frames, double* out_max_power, double* out_mean_mfccs);
/* ss_sound_analyze_batch   SoundDictionary::from_path (src/sound.rs:304-320: one Sound::from_path per .wav of a directory)
 *                          as ONE upload and one MFCC launch (SURVEY.md §8f item 4). `samples` holds nsounds sounds back to
 *                          back, sound i = samples[sample_offsets[i] .. sample_offsets[i+1]) (offsets[0] = 0), all at the
 *                          same sample_rate. Every sound is framed on its own (no frame straddles two sounds):
 *                          out_frame_offsets (nsounds + 1) gives each sound's row range in out_mfcc (sum of the per-sound
 *                          frame counts x ncoeffs doubles); out_max_power (nsounds) and out_mean_mfccs (nsounds x ncoeffs,
 *                          NaN row for a sound without a full frame) as Sound::from_samples computes them. The three
 *                          outputs may be NULL. Values equal ss_sound_analyze on each sound alone. */
int ss_sound_analyze_batch(ss_ctx* ctx, const double* samples, const uint64_t* sample_offsets, size_t nsounds, double sample_rate,
                           int ncoeffs, double* out_mfcc, uint64_t* out_frame_offsets, double* out_max_power, double* out_mean_mfccs);
int ss_mfcc(ss_ctx* ctx, const double* samples, size_t n, double sample_rate, int ncoeffs, double* out_mfcc,
            size_t* out_frames);
int ss_max_power(ss_ctx* ctx, const double* samples, size_t n, double* out);
/* device-resident form: d_samples (f64, n) -> d_out_mfcc (f64, frames x ncoeffs); asynchronous on the ctx stream */
int ss_mfcc_dev(ss_ctx* ctx, const double* d_samples, size_t n, double sample_rate, int ncoeffs, double* d_out_mfcc);

/* ---- Partitioner: segmentation subsystem ------------------------------------------------------------------------------
 * ss_symbols      discretize_with_model (src/lib.rs:56-60) + the symbolisation loop (src/lib.rs:123-131, max_index
 *                 src/sound.rs:486-495): standardise THIS input's MFCC rows, GMM posteriors, argmax -> 'A' + idx.
 *                 model == NULL -> SS_ERR_NOT_TRAINED. out_posteriors (frames x ncomp) may be NULL.
 * ss_vote_split   voting_experts::cast_votes + split_string (src/lib.rs:135-136) + the length map (src/lib.rs:137):
 *                 out_votes (n+1 counters, may be NULL), out_seg_lens in SAMPLES (chunk symbols x SS_HOP; capacity n).
 * ss_partition    Partitioner::partition_other (src/lib.rs:112-144) = the two above.
 */
int ss_symbols(ss_ctx* ctx, const double* mfcc, size_t frames, const ss_gmm* model, uint8_t* out_symbols,
               double* out_posteriors);
/* ss_gmm_train   train_model (src/lib.rs:44-54): Standardizer on the input, then `iters` EM rounds for `ncomp`
 *                full-covariance Gaussians with CovOption::Regularized(reg) (reference: ncomp 26, iters 5, reg 0.1).
 *                Initial means are `ncomp` distinct rows drawn with a seeded mt19937_64 (the reference draws from
 *                thread_rng, so its model differs from run to run; parity is defined GIVEN a model). On a collapsed
 *                component / singular covariance returns SS_ERR_INVALID — retry with another seed, as the reference's
 *                `while let Err` loop does. Outputs: means ncomp x ncoeffs, covs ncomp x ncoeffs x ncoeffs, weights ncomp. */
int ss_gmm_train(ss_ctx* ctx, const double* mfcc, size_t frames, int ncoeffs, int ncomp, int iters, double reg, uint64_t seed,
                 double* out_means, double* out_covs, double* out_weights);
int ss_vote_split(ss_ctx* ctx, const uint8_t* symbols, size_t n, int depth, int threshold, uint32_t* out_votes,
                  uint64_t* out_seg_lens, size_t* out_nseg);
int ss_partition(ss_ctx* ctx, const double* mfcc, size_t frames, const ss_gmm* model, int depth, int threshold,
                 uint64_t* out_seg_lens, size_t* out_nseg);

/* ---- SoundDictionary / SoundSequence: matcher subsystem ---------------------------------------------------------------
 * ss_dict_create   SoundDictionary::from_segments / add_segments (src/sound.rs:323-343) seen from the matcher: segment d
 *                  owns MFCC frames [frame_offsets[d], frame_offsets[d+1]) of mfcc_flat (frames x ncoeffs, row-major).
 *                  index_base is added to every index this shard reports, so that a dictionary partitioned across GPUs
 *                  (one ss_dict per rank) reports GLOBAL indices.
 * ss_dict_match    SoundDictionary::at_distance (src/sound.rs:351-370) for a batch of queries; targets == NULL means
 *                  1.0 = match_sound (src/sound.rs:346-348). SS_COSINE_REF: k must be 1, out_dist = |sim - target|
 *                  (2.0 and index index_base if nothing is < 2.0, as the reference's fold). SS_DTW: the k best
 *                  (distance, index) ascending, ties to the lowest index; unfilled slots (inf, 0xFFFFFFFF); targets are
 *                  ignored. SS_DTW_TARGET (spec A13, DESIGN.md §3.1h): with D the SS_DTW distance of the pair (its recurrence,
 *                  normalisation, band and NaN rule) and t the query's target, the key is e = fabs(D - t) in f64; the k best
 *                  (e, index) ascending, ties to the lowest index, out_dist = e (as SS_COSINE_REF's |sim - target|), unfilled
 *                  slots (inf, 0xFFFFFFFF), k in 1..SS_MAX_TOPK. targets == NULL means t = 0 for every query, and then the
 *                  results equal SS_DTW's bit for bit. A non-finite target -> SS_ERR_INVALID (the _dev entry points take
 *                  finite targets as a precondition). The ss_dict_last_* readers describe the match as for SS_DTW; the
 *                  ss_dict_set_scan preference does not apply (the match always starts at the fp32 CUDA-core scan).
 *                  out_idx / out_dist: nq x k.
 * ss_queries_*     the same in two steps with the queries kept in HBM (bench.py's kernel-only number; multi-GPU).
 * ss_topk_merge_dev merges `nlists` per-shard results (as gathered from all ranks, list-major [nlists][nq][k]) into the
 *                  global top-k by (distance, index) lexicographic order — the first-minimum rule of the reference's
 *                  strict-'<' scan (src/sound.rs:361-366) carried across shards.
 */
int ss_dict_create(ss_ctx* ctx, const double* mfcc_flat, const uint64_t* frame_offsets, size_t nseg, int ncoeffs,
                   uint32_t index_base, ss_dict** out);
void ss_dict_destroy(ss_dict* dict);
size_t ss_dict_len(const ss_dict* dict);
int ss_dict_match(ss_dict* dict, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int mode,
                  const double* targets, int k, uint32_t* out_idx, double* out_dist);

int ss_queries_create(ss_ctx* ctx, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int ncoeffs,
                      ss_queries** out);
void ss_queries_destroy(ss_queries* q);
/* asynchronous on the ctx stream: the whole match (layout kernel, scan, merge, f64 refine) is enqueued without a host round
 * trip; d_out_idx (u32, nq x k) and d_out_dist (f64, nq x k) are DEVICE pointers. SS_DTW: whether some query needs a
 * fallback stage (fp32 scan / exhaustive f64) is only known once the refine has run, so the results in d_out_* are final after
 * ss_dict_match_finish(dict) - which waits for that one event and, in the rare case, runs the fallback for the queries
 * concerned. The ss_dict_last_* readers, the next match on the same dictionary and ss_dict_match_sharded* call it
 * themselves; `q` must stay alive until then, and so must SS_DTW_TARGET's d_targets (nq finite f64, or NULL). */
int ss_dict_match_dev(ss_dict* dict, ss_queries* q, int mode, const double* d_targets, int k, uint32_t* d_out_idx,
                      double* d_out_dist);
int ss_dict_match_finish(ss_dict* dict);
/* SoundSequence::from_distances (src/sound.rs:405-417) for SS_COSINE_REF, on the device: step t matches the previous
 * step's dictionary segment (step 0: the start query) at target distances[t]. Host buffers, one blocking point.
 * Every step's (out_idx[t], out_dist[t]) equals ss_dict_match(dict, query, 1, SS_COSINE_REF, &distances[t], 1, ...) bit for
 * bit, indices include index_base. A pending SS_DTW match completes first; the ss_dict_last_* readers still describe the
 * last MATCH (a walk changes none of them). nsteps == 0 returns SS_OK and launches nothing. */
int ss_dict_walk(ss_dict* dict, const double* start_mfcc, size_t start_frames, const double* distances, size_t nsteps,
                 uint32_t* out_idx, double* out_dist);
/* the same on device pointers, asynchronous on the ctx stream (nsteps + 1 kernel launches, no host synchronisation);
 * `start` holds exactly one query */
int ss_dict_walk_dev(ss_dict* dict, ss_queries* start, const double* d_distances, size_t nsteps, uint32_t* d_out_idx,
                     double* d_out_dist);
/* SoundSequence::from_distances for SS_DTW_TARGET (DESIGN.md §3.1i), on the device: step t's (out_idx[t], out_dist[t]) equals
 * ss_dict_match(dict, query_t, 1, SS_DTW_TARGET, &distances[t], 1, ...) bit for bit (A13: e = fabs(D - t) under the dictionary's
 * band, indices include index_base); query_0 is the start sound, query_{t+1} the segment out_idx[t] - index_base. A step with
 * no result (every e NaN or +inf) writes (0xFFFFFFFF, +inf), and every later step, which runs from an empty query, does too.
 * distances == NULL means t = 0 at every step: SS_DTW's nq = 1 chain. A non-finite target -> SS_ERR_INVALID. Checks and ordering
 * as ss_dict_walk: a pending SS_DTW match completes first, the ss_dict_last_* readers are untouched, ss_dict_set_scan does not
 * apply (every step is exact f64 DTW against every segment). nsteps == 0 returns SS_OK and launches nothing. Host buffers, one
 * blocking point. */
int ss_dict_walk_dtw(ss_dict* dict, const double* start_mfcc, size_t start_frames, const double* distances, size_t nsteps,
                     uint32_t* out_idx, double* out_dist);
/* the same on device pointers, asynchronous on the ctx stream: exactly nsteps kernel launches, no host synchronisation besides
 * completing a pending SS_DTW match; `start` holds exactly one query; d_distances (nsteps finite f64, or NULL) */
int ss_dict_walk_dtw_dev(ss_dict* dict, ss_queries* start, const double* d_distances, size_t nsteps, uint32_t* d_out_idx,
                         double* d_out_dist);
/* DTW warping path of query p against dictionary segment seg_idx[p] (an index as ss_dict_match
 * reports it, index_base included; 0xFFFFFFFF -> empty path, inf). out_path: (i, j) uint32 pairs, compacted; path p is
 * out_path[out_path_offsets[p] .. out_path_offsets[p+1]) (nq + 1 offsets, in pairs). out_dist[p] is bit-equal to ss_dict_match's
 * SS_DTW distance; an empty side or a distance that is not finite gives an empty path and inf. The path runs from (0, 0) to
 * (Lq-1, Ld-1); backtracking through the DTW matrix D, each step takes the smallest D of diag (i-1, j-1), up (i-1, j), left
 * (i, j-1), ties in that order, NaN as +inf (DESIGN.md §3.1e). path_capacity is in cells:
 * at least the sum over the pairs with both sides non-empty of (Lq + Ld - 1); less, or an index out of range, returns
 * SS_ERR_INVALID. Works whatever mode the dictionary was last matched in. A pending SS_DTW match completes first; the
 * ss_dict_last_* readers still describe the last MATCH. Host buffers, stream-synchronised on return. */
int ss_dict_align(ss_dict* dict, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, const uint32_t* seg_idx,
                  uint32_t* out_path, size_t path_capacity, uint64_t* out_path_offsets, double* out_dist);
/* the same on device pointers, asynchronous on the ctx stream (no host synchronisation besides completing a pending SS_DTW match),
 * so that it can take ss_dict_match_dev's d_out_idx (k = 1) as d_seg_idx directly. path_capacity >= the sum over non-empty queries of
 * (Lq + Ld_max - 1), Ld_max = the longest segment (checked on the host); an index out of range, which only the device sees, gives an
 * empty path and NaN. Launches: 3 + one per wave of pairs with a side longer than 32 frames (waves are sized on the host from the
 * query lengths and Ld_max, so the count is known before the call); nq == 0 launches nothing. */
int ss_dict_align_dev(ss_dict* dict, ss_queries* q, const uint32_t* d_seg_idx, uint32_t* d_out_path, size_t path_capacity,
                      uint64_t* d_out_path_offsets, double* d_out_dist);
/* ss_dict_locate   subsequence DTW (no reference counterpart; spec A12, DESIGN.md §3.1g): WHERE inside a dictionary segment each query
 *              fits best, the query free to start and end at any frame of it. For a query of Lq frames and a segment of Ld frames,
 *              c(i, j) is A8's local cost (same operations, same order) and
 *                  S(0, j) = c(0, j);   S(i, j) = c(i, j) + fmin(fmin(S(i-1, j), S(i, j-1)), S(i-1, j-1))   (i >= 1)
 *              with a missing neighbour (j = 0) +inf and NaN counting as +inf. The start column st(0, j) = j travels along the
 *              neighbour the min chose (ss_dict_align's rule: diag if it equals the min, else up if it does, else left). The end e
 *              is the smallest j whose S(Lq-1, j) is the minimum of the finite values of row Lq-1; the pair's hit is
 *              (cost = S(Lq-1, e), start = st(Lq-1, e), end = e), cost UNNORMALISED; no finite value, empty query or empty
 *              segment: no hit. One hit per (query, segment); the k best across segments by (cost, index) ascending,
 *              indices + index_base; unfilled slots (idx, start, end, cost) = (0xFFFFFFFF, 0xFFFFFFFF, 0xFFFFFFFF, +inf).
 *              cost / (Lq + end - start + 1) is ss_dict_match's SS_DTW distance of the query against frames start..end
 *              of the segment bit for bit, and ss_dict_align's path on that span is the backtrack of S from (Lq-1, end): the span
 *              can feed ss_dict_align and ss_resynth_warped unchanged (dictionary samples offset by start * SS_HOP).
 *              out_*: nq x k; start / end are frame indices within the segment, end inclusive; any output other than out_idx may
 *              be NULL. The Sakoe-Chiba band does not apply. k outside 1..SS_MAX_TOPK or a NULL input -> SS_ERR_INVALID; an
 *              empty dictionary -> SS_ERR_EMPTY_DICT. A pending SS_DTW match completes first; the ss_dict_last_* readers still
 *              describe the last MATCH. Host buffers, stream-synchronised on return. */
int ss_dict_locate(ss_dict* dict, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int k, uint32_t* out_idx,
                   uint32_t* out_start, uint32_t* out_end, double* out_cost);
/* the same on device pointers, asynchronous on the ctx stream (no host synchronisation besides completing a pending SS_DTW match).
 * Launches: 3 per batch of B = max(1, min(nq, floor(2^24 / nseg))) queries, i.e. 3 ceil(nq / B); nq == 0 launches nothing. */
int ss_dict_locate_dev(ss_dict* dict, ss_queries* q, int k, uint32_t* d_out_idx, uint32_t* d_out_start, uint32_t* d_out_end,
                       double* d_out_cost);
int ss_topk_merge_dev(ss_ctx* ctx, const uint32_t* d_idx, const double* d_dist, int nlists, size_t nq, int k,
                      uint32_t* d_out_idx, double* d_out_dist);
/* drops the cached device layouts of a query batch so that the next match rebuilds them (bench.py calls this every
 * step so that the layout kernels are inside the timed region). Stream-ordered, no synchronisation. The length-sorted
 * grouping of the batch depends on the offsets only and stays (it is part of ss_queries_create). */
int ss_queries_invalidate(ss_queries* q);
/* device time of the dominant kernel (DTW scan / cosine scan) of the last ss_dict_match*(…), measured with CUDA events
 * on the ctx stream; synchronises the stream. Returns a negative value if no match has run. */
double ss_dict_last_scan_ms(ss_dict* dict);
/* which kernel scanned the dictionary in the last match (its first stage): 1 = packed-half tensor-core scan (k_dtw_scan_h2), 2 = fp32-DP
 * tensor-core scan (k_dtw_scan_tc), 3 = fp32 CUDA-core scan (k_dtw_scan: a segment or query longer than 32 frames), 4 = cosine-ref */
int ss_dict_last_scan_kind(const ss_dict* dict);
/* DP cells / similarity products the last ss_dict_match*(…) evaluated (sum over pairs of Lq*Ld, resp. of min(Kq,Kd)) */
uint64_t ss_dict_last_work(const ss_dict* dict);
/* SS_DTW only: number of queries of the last match whose exact top-k could not be certified from the fp32 scan's
 * candidate list (see DESIGN.md "filter and refine"); 0 means every reported index is the f64 argmin. */
uint64_t ss_dict_last_uncertified(const ss_dict* dict);
/* SS_DTW only: number of queries of the last match that the tensor-core (fp16) scan could not certify and that were
 * therefore re-run through the fp32 scan before the result was returned. */
uint64_t ss_dict_last_tc_fallback(const ss_dict* dict);
/* SS_DTW only: number of queries of the last match that neither scan could certify (e.g. many near-identical dictionary
 * entries) and that were therefore matched by exhaustive f64 DTW against every segment. */
uint64_t ss_dict_last_exhaustive(const ss_dict* dict);

/* ---- the matcher across the GPUs of one box (SURVEY.md §8b / §8e) ------------------------------------------------------------
 * The dictionary is partitioned into contiguous shards balanced by frames (ss_shard_bounds), one ss_dict per GPU created with
 * index_base = the shard's first global index. A match then runs on every GPU against its shard; the query frames cross PCIe
 * once (1 / nranks per GPU) and are all-gathered over NVLink; the per-shard top-k lists are exchanged with ONE ncclAllGather
 * and merged on every rank by (distance, index) - the first-minimum rule of the reference's strict-'<' scan
 * (src/sound.rs:361-366) across shards, so the result equals the single-GPU result bit for bit.
 *
 * Two front ends:
 *   single process   ss_dict_create_sharded(ctxs, nctx, ...) / ss_sharded_dict_match(...): same arguments as ss_dict_create /
 *                    ss_dict_match; the library owns the shards, an NCCL communicator per GPU (ncclCommInitAll) and one
 *                    worker thread per GPU. This is what SoundDictionary::match_sound / at_distance (src/sound.rs:346-370)
 *                    bind to when more than one GPU is given.
 *   one rank per process (torchrun, MPI): ss_comm_unique_id on rank 0, ship the SS_COMM_ID_BYTES to the other ranks by any
 *                    means, ss_comm_create on every rank, then the rank-local calls ss_queries_create_sharded /
 *                    ss_dict_match_sharded[_dev] with this rank's shard - collective: every rank must make the same call.
 * NCCL is bound at run time (dlopen of libnccl.so.2); without it these calls return SS_ERR_CUDA and nothing else is affected. */
#define SS_COMM_ID_BYTES 128
typedef struct ss_comm ss_comm;                 /* this rank's end of a communicator: one ctx (GPU), rank, nranks */
typedef struct ss_sharded_dict ss_sharded_dict; /* a dictionary partitioned across the GPUs of one process */

int ss_shard_bounds(const uint64_t* frame_offsets, size_t nseg, int nshards, uint64_t* out_cuts /* nshards + 1 */);
int ss_comm_unique_id(void* out_id /* SS_COMM_ID_BYTES */);
int ss_comm_create(ss_ctx* ctx, int nranks, int rank, const void* id, ss_comm** out);
int ss_comm_create_all(ss_ctx* const* ctxs, int nctx, ss_comm** out /* nctx entries */);
void ss_comm_destroy(ss_comm* comm);
int ss_comm_rank(const ss_comm* comm);
int ss_comm_nranks(const ss_comm* comm);
/* the query batch resident on this rank's GPU, its frames uploaded 1 / nranks per rank and all-gathered over NVLink */
int ss_queries_create_sharded(ss_comm* comm, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int ncoeffs,
                              ss_queries** out);
/* local match against `shard`, exchange, merge: d_out_* (device) hold the GLOBAL top-k on every rank. Stream-ordered, but the
 * host waits for the shard's fallback decision (ss_dict_match_finish) before it enqueues the exchange. */
int ss_dict_match_sharded_dev(ss_dict* shard, ss_comm* comm, ss_queries* q, int mode, const double* d_targets, int k,
                              uint32_t* d_out_idx, double* d_out_dist);
/* the same with HOST buffers in and out (ss_dict_match's contract) */
int ss_dict_match_sharded(ss_dict* shard, ss_comm* comm, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int mode,
                          const double* targets, int k, uint32_t* out_idx, double* out_dist);
/* SoundDictionary::from_segments / add_segments + match_sound / at_distance over several GPUs of ONE process */
int ss_dict_create_sharded(ss_ctx* const* ctxs, int nctx, const double* mfcc_flat, const uint64_t* frame_offsets, size_t nseg,
                           int ncoeffs, ss_sharded_dict** out);
int ss_sharded_dict_match(ss_sharded_dict* dict, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int mode,
                          const double* targets, int k, uint32_t* out_idx, double* out_dist);
void ss_sharded_dict_destroy(ss_sharded_dict* dict);
size_t ss_sharded_dict_len(const ss_sharded_dict* dict);
int ss_sharded_dict_nshards(const ss_sharded_dict* dict);

/* ss_dict_debug_tc_scan   measurement hook for the SS_DTW filter stage (no reference counterpart; tests/test_parity_large_gpu.py):
 *              the RAW distance the tensor-core scan (fp16 products, fp32 accumulation in TMEM, fp32 DP) assigns to EVERY
 *              (query, segment) pair - out_scan[nq x nseg], NaN where a side is empty - together with the mean frame
 *              (out_mu, 16 doubles, the first ncoeffs used) both sides were centred on and the power-of-two scale s of the
 *              norm columns, so that a host can rebuild the fp16 operands exactly and measure |scan - DTW(rounded frames)|
 *              against the slack the certification assumes (DESIGN.md §3.1a). Runs the production scan kernel with one extra
 *              store per pair compiled in. SS_ERR_INVALID when these inputs would take the fp32 scan instead (a segment or
 *              query longer than 32 frames, values outside the fp16 range). */
int ss_dict_debug_tc_scan(ss_dict* dict, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, float* out_scan,
                          double* out_mu, float* out_scale);
/* the same for the packed-half scan (fp16 products with an F16 accumulator, DP in half2: the default first stage); out_s = its
 * power-of-two cost scale S (the operands are A = S [-2 a~, s, s, rd(|a~|^2 / s)], the scan value is D16 / (S (Lq + Ld))) */
int ss_dict_debug_h2_scan(ss_dict* dict, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, float* out_scan,
                          double* out_mu, float* out_scale, float* out_s);
/* test / A-B hook: which filter stage an SS_DTW match STARTS with when all of them apply. 0 (default) = packed-half tensor-core
 * scan, 1 = fp32-DP tensor-core scan, 2 = fp32 CUDA-core scan, 3 = packed-half scan WITHOUT its second chance (the pass over the
 * per-slice candidate lists that certifies most of what the merged list could not), so that tests can drive the later stages.
 * The results are identical by construction (every stage is followed by the f64 refine + certification); only the speed differs. */
int ss_dict_set_scan(ss_dict* dict, int first_stage);

/* Sakoe-Chiba band of the SS_DTW distance (DESIGN.md §3.1f), per dictionary. radius 0 (the default) = no band: every result is
 * bit-identical to a dictionary that never set one. For radius r >= 1, cell (i, j) of a pair of Lq x Ld frames is inside the band iff
 *     |i (Ld - 1) - j (Lq - 1)| <= r max(Lq - 1, Ld - 1)       (64-bit integers)
 * - |i - j| <= r for equal lengths; otherwise the band follows the line from (0, 0) to (Lq-1, Ld-1), r counted in frames of the
 * longer side. A cell outside the band has D = +inf and is never a predecessor; inside it the recurrence, the normalisation
 * D(Lq-1, Ld-1) / (Lq + Ld), the (distance, index) order and the NaN rule are unchanged. The end cell is always reachable, and
 * r >= min(Lq-1, Ld-1) covers the whole matrix. The band applies to SS_DTW matches (ss_dict_match, _dev, _sharded*) and to
 * ss_dict_align[_dev]; SS_COSINE_REF, ss_dict_walk and the ss_dict_debug_* hooks ignore it. A pending SS_DTW match completes
 * first, with the radius it started with. NULL -> SS_ERR_INVALID. With one rank per process every rank sets the radius of its own
 * shard, and all ranks must set the same radius. */
int ss_dict_set_dtw_band(ss_dict* dict, uint32_t radius);
uint32_t ss_dict_dtw_band(const ss_dict* dict); /* 0 for NULL */
/* the same on every shard of a single-process sharded dictionary */
int ss_sharded_dict_set_dtw_band(ss_sharded_dict* dict, uint32_t radius);

/* ss_resynth   SoundSequence::clone_from_dictionary sample assembly (src/sound.rs:451-472) + to_sound (:475-483):
 *              for target segment t copy min(len) samples of dictionary sound match_idx[t] and zero-pad to
 *              target_lens[t]; segments are concatenated into out_samples (capacity sum(target_lens)). */
int ss_resynth(ss_ctx* ctx, const double* dict_samples, const uint64_t* dict_sample_offsets, size_t ndict,
               const uint32_t* match_idx, const uint64_t* target_lens, size_t nseg, double* out_samples);
/* ss_resynth_warped   ss_resynth along the DTW warping path of each match (no reference counterpart; spec A11, DESIGN.md §3.5), so
 *              that every matched sound follows its target segment's timing instead of being zero-padded or cut. paths /
 *              path_offsets are what ss_dict_align writes for the same segments and indices: (i, j) uint32 pairs, path t =
 *              paths[2 path_offsets[t] .. 2 path_offsets[t+1]) (nseg + 1 offsets in pairs, path_offsets[0] = 0). With H = SS_HOP,
 *              L = target_lens[t], m = match_idx[t] and X(p) = sample p of dictionary sound m (0.0 at or past its end):
 *              - output block b (samples n = b H + r, 0 <= r < min(H, L - b H)) plays source frame j(b): the j of the first cell
 *                of row b; for b >= Lq = 1 + the last cell's i, j(b) = j(Lq-1) + (b - Lq + 1); an empty path gives j(b) = b;
 *              - with s_b = j(b) H (64-bit): out = X(s_b + r) if b = 0 or s_b = s_{b-1} + H, else the one-hop crossfade
 *                X(s_{b-1} + H + r) (H - r) / H + X(s_b + r) r / H (exact dyadic weights; two products and a sum, each
 *                rounded to nearest, no FMA).
 *              A diagonal or empty path gives ss_resynth's samples bit for bit. Segments are concatenated into out_samples
 *              (capacity sum(target_lens)). Host buffers, stream-synchronised on return; one kernel launch, none when
 *              sum(target_lens) = 0. SS_ERR_INVALID (with a message) for a NULL buffer (paths may be NULL when every path is
 *              empty), path offsets not monotone or not starting at 0, a non-empty path not starting at (0, 0), a step other
 *              than (1, 0), (0, 1), (1, 1), or match_idx[t] >= ndict; nseg == 0 returns SS_OK and launches nothing; ndict == 0
 *              gives SS_ERR_EMPTY_DICT. */
int ss_resynth_warped(ss_ctx* ctx, const double* dict_samples, const uint64_t* dict_sample_offsets, size_t ndict,
                      const uint32_t* match_idx, const uint32_t* paths, const uint64_t* path_offsets, const uint64_t* target_lens,
                      size_t nseg, double* out_samples);

/* cosine_sim_angular over consecutive mean-MFCC rows, SoundSequence::new (src/sound.rs:392-396, 62-69):
 * out_dist[i] = acos(clamp(cosine_sim(mean[i], mean[i+1]))) / pi with the reference's x < -1 -> 1 rule; nrows-1 outputs */
int ss_sequence_distances(ss_ctx* ctx, const double* mean_mfccs, size_t nrows, int ncoeffs, double* out_dist);

#ifdef __cplusplus
}
#endif
#endif /* SOUNDSYM_B200_H */
