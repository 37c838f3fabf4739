// capi.cu — the extern "C" boundary declared in include/soundsym_b200.h: context, error strings, handle lifetimes and
// the host-buffer wrappers (H2D, kernels, D2H, stream-synchronised on return). No compute happens on the host.
#include <cstring>
#include <limits>

#include "match.cuh"
#include "sound.cuh"

namespace ss {

static thread_local std::string g_noctx_error;

int set_error(ss_ctx* ctx, int code, const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf;
    else g_noctx_error = buf;
    return code;
}

static int check_offsets(ss_ctx* ctx, const uint64_t* off, size_t n, const char* what) {
    if (!off) return set_error(ctx, SS_ERR_INVALID, "%s: offsets are NULL", what);
    for (size_t i = 0; i < n; i++)
        if (off[i + 1] < off[i]) return set_error(ctx, SS_ERR_INVALID, "%s: offsets not monotone at %zu", what, i);
    return SS_OK;
}

// host-side bookkeeping of a (re)filled batch: offsets rebased to 0, lengths, cached layouts dropped
int queries_prepare(ss_queries* q, const uint64_t* q_frame_offsets, size_t nq) {
    q->nq = nq;
    q->nonempty = 0;
    q->max_len = 0;
    q->lane_built = false;
    q->cos_built = false;
    q->tc_built = false;
    q->h2_built = false;
    q->tc_grouped = false;
    q->h_off.resize(nq + 1);
    const uint64_t base = nq ? q_frame_offsets[0] : 0;
    q->h_off[0] = 0;
    for (size_t i = 0; i < nq; i++) {
        q->h_off[i + 1] = q_frame_offsets[i + 1] - base;
        q->nonempty += q_frame_offsets[i + 1] > q_frame_offsets[i];
        q->max_len = std::max<uint32_t>(q->max_len, (uint32_t)std::min<uint64_t>(0xFFFFFFFFull, q_frame_offsets[i + 1] - q_frame_offsets[i]));
    }
    q->total_frames = q->h_off[nq];
    return SS_OK;
}

// (re)fills a query batch in place: device buffers are grow-only, so a reused handle does no cudaMalloc / cudaFree
int queries_fill(ss_queries* q, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq) {
    ss_ctx* ctx = q->ctx;
    SS_TRY(queries_prepare(q, q_frame_offsets, nq));
    const uint64_t base = nq ? q_frame_offsets[0] : 0;
    // the frames start crossing PCIe first; the length-sorted grouping of the batch (host work) overlaps that copy
    SS_TRY(upload(ctx, q->d_mfcc, q_mfcc ? q_mfcc + base * q->c : nullptr, (size_t)q->total_frames * q->c));
    SS_TRY(upload(ctx, q->d_off, q->h_off.data(), nq + 1));
    SS_TRY(dtw_tc_queries_group(q));
    return SS_OK;
}

int queries_check(ss_ctx* ctx, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int ncoeffs) {
    if (ncoeffs < 1 || ncoeffs > SS_MAX_NCOEFFS) return set_error(ctx, SS_ERR_INVALID, "ncoeffs must be in 1..%d (got %d)", SS_MAX_NCOEFFS, ncoeffs);
    if (nq > 0x7FFFFFF0ull) return set_error(ctx, SS_ERR_INVALID, "too many queries");
    SS_TRY(check_offsets(ctx, q_frame_offsets, nq, "queries"));
    if (nq && q_frame_offsets[nq] > q_frame_offsets[0] && !q_mfcc) return set_error(ctx, SS_ERR_INVALID, "q_mfcc is NULL");
    return SS_OK;
}

// SS_DTW_TARGET's host-buffer targets: every one finite (the _dev entry points take that as a precondition)
int targets_check(ss_ctx* ctx, int mode, const double* targets, size_t nq) {
    if (mode != SS_DTW_TARGET || !targets) return SS_OK;
    for (size_t i = 0; i < nq; i++)
        if (!std::isfinite(targets[i])) return set_error(ctx, SS_ERR_INVALID, "targets[%zu] = %g is not finite", i, targets[i]);
    return SS_OK;
}

}  // namespace ss

using namespace ss;

extern "C" {

const char* ss_version(void) { return "soundsym_b200 0.1 (sm_100a)"; }

int ss_ctx_create(int device, ss_ctx** out) {
    if (!out) return set_error(nullptr, SS_ERR_INVALID, "ss_ctx_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return set_error(nullptr, SS_ERR_CUDA, "no CUDA device (%s); this library has no CPU fallback",
                         e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= ndev) return set_error(nullptr, SS_ERR_INVALID, "device %d out of range (0..%d)", device, ndev - 1);
    ss_ctx* ctx = new (std::nothrow) ss_ctx();
    if (!ctx) return set_error(nullptr, SS_ERR_NOMEM, "out of host memory");
    ctx->device = device;
    if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking)) != cudaSuccess) {
        set_error(nullptr, SS_ERR_CUDA, "device %d: %s", device, cudaGetErrorString(e));
        delete ctx;
        return SS_ERR_CUDA;
    }
    cudaDeviceGetAttribute(&ctx->sm_count, cudaDevAttrMultiProcessorCount, device);
    int major = 0;
    cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device);
    if (major != 10) {
        set_error(nullptr, SS_ERR_CUDA, "device %d has compute capability %d.x; this library is built for sm_100a only", device, major);
        cudaStreamDestroy(ctx->stream);
        delete ctx;
        return SS_ERR_CUDA;
    }
    *out = ctx;
    return SS_OK;
}

void ss_ctx_destroy(ss_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    if (ctx->sound_state && ctx->sound_state_free) ctx->sound_state_free(ctx->sound_state);
    if (ctx->seg_state && ctx->seg_state_free) ctx->seg_state_free(ctx->seg_state);
    for (void* b : ctx->pinned_free) cudaFreeHost(b);
    cudaStreamDestroy(ctx->stream);
    delete ctx;
}

const char* ss_last_error(const ss_ctx* ctx) { return ctx ? ctx->err.c_str() : g_noctx_error.c_str(); }
void* ss_ctx_stream(ss_ctx* ctx) { return ctx ? (void*)ctx->stream : nullptr; }
int ss_ctx_device(const ss_ctx* ctx) { return ctx ? ctx->device : -1; }
uint64_t ss_ctx_launch_count(const ss_ctx* ctx) { return ctx ? ctx->launches : 0; }
int ss_ctx_sync(ss_ctx* ctx) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SS_OK;
}

int ss_frame_count(size_t n, size_t* out_frames) {
    if (!out_frames) return set_error(nullptr, SS_ERR_INVALID, "out_frames is NULL");
    *out_frames = n >= SS_BIN ? (n - SS_BIN) / SS_HOP + 1 : 0;
    return SS_OK;
}

// ---- dictionary / queries ----------------------------------------------------------------------------------------
int ss_dict_create(ss_ctx* ctx, const double* mfcc_flat, const uint64_t* frame_offsets, size_t nseg, int ncoeffs,
                   uint32_t index_base, ss_dict** out) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (!out) return set_error(ctx, SS_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (ncoeffs < 1 || ncoeffs > SS_MAX_NCOEFFS) return set_error(ctx, SS_ERR_INVALID, "ncoeffs must be in 1..%d (got %d)", SS_MAX_NCOEFFS, ncoeffs);
    if (nseg > 0xFFFFFFF0ull) return set_error(ctx, SS_ERR_INVALID, "too many segments");
    SS_TRY(check_offsets(ctx, frame_offsets, nseg, "ss_dict_create"));
    if (nseg && frame_offsets[nseg] > frame_offsets[0] && !mfcc_flat) return set_error(ctx, SS_ERR_INVALID, "mfcc_flat is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    ss_dict* d = new (std::nothrow) ss_dict();
    if (!d) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
    d->ctx = ctx;
    d->nseg = nseg;
    d->c = ncoeffs;
    d->index_base = index_base;
    d->h_off.resize(nseg + 1);
    const uint64_t base = nseg ? frame_offsets[0] : 0;
    d->h_off[0] = 0;
    for (size_t i = 0; i < nseg; i++) {
        d->h_off[i + 1] = frame_offsets[i + 1] - base;
        d->max_len = std::max<uint32_t>(d->max_len, (uint32_t)std::min<uint64_t>(0xFFFFFFFFull, frame_offsets[i + 1] - frame_offsets[i]));
    }
    d->total_frames = d->h_off[nseg];
    int rc = upload(ctx, d->d_mfcc, mfcc_flat ? mfcc_flat + base * ncoeffs : nullptr, (size_t)d->total_frames * ncoeffs);
    if (rc == SS_OK) rc = upload(ctx, d->d_off, d->h_off.data(), nseg + 1);
    if (rc == SS_OK) rc = cosine_dict_build(d);
    if (rc == SS_OK) rc = dtw_dict_build(d);
    if (rc == SS_OK) rc = dtw_tc_dict_build(d);
    if (rc == SS_OK) rc = dtw_h2_dict_build(d);
    if (rc == SS_OK && cudaStreamSynchronize(ctx->stream) != cudaSuccess) rc = set_error(ctx, SS_ERR_CUDA, "dictionary build failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc != SS_OK) {
        delete d;
        return rc;
    }
    *out = d;
    return SS_OK;
}

void ss_dict_destroy(ss_dict* d) {
    if (!d) return;
    cudaSetDevice(d->ctx->device);
    cudaStreamSynchronize(d->ctx->stream);
    CacheFrees cache;  // nothing can still touch the buffers: they go to the device cache, not back to the driver
    delete d;
}
size_t ss_dict_len(const ss_dict* d) { return d ? d->nseg : 0; }
uint64_t ss_dict_last_work(const ss_dict* d) { return d ? d->last_work : 0; }
int ss_dict_last_scan_kind(const ss_dict* d) { return d ? d->last_scan_kind : 0; }

int ss_dict_match_finish(ss_dict* d) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    SS_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    return dtw_match_finish(d);
}
// the counters of the last match are only final once its fallback decision has been taken
static bool finished(const ss_dict* dc) {
    ss_dict* d = const_cast<ss_dict*>(dc);
    if (!d) return false;
    cudaSetDevice(d->ctx->device);
    return dtw_match_finish(d) == SS_OK;
}
uint64_t ss_dict_last_tc_fallback(const ss_dict* d) { return finished(d) ? d->last_tc_fallback : ~0ull; }
uint64_t ss_dict_last_exhaustive(const ss_dict* d) { return finished(d) ? d->last_exhaustive : ~0ull; }
uint64_t ss_dict_last_uncertified(const ss_dict* d) { return finished(d) ? d->last_uncertified : ~0ull; }

int ss_queries_create(ss_ctx* ctx, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int ncoeffs, ss_queries** out) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (!out) return set_error(ctx, SS_ERR_INVALID, "out is NULL");
    *out = nullptr;
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, ncoeffs));
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    ss_queries* q = new (std::nothrow) ss_queries();
    if (!q) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
    q->ctx = ctx;
    q->c = ncoeffs;
    const int rc = queries_fill(q, q_mfcc, q_frame_offsets, nq);
    if (rc != SS_OK) {
        delete q;
        return rc;
    }
    *out = q;
    return SS_OK;
}

int ss_queries_invalidate(ss_queries* q) {
    if (!q) return set_error(nullptr, SS_ERR_INVALID, "queries is NULL");
    // stream-ordered: the next match rebuilds the layouts behind whatever still reads the old ones; no synchronisation
    q->lane_built = false;
    q->cos_built = false;
    q->tc_built = false;
    q->h2_built = false;
    return SS_OK;
}

double ss_dict_last_scan_ms(ss_dict* d) {
    if (!d || !d->scan_timed) return -1.0;
    cudaSetDevice(d->ctx->device);
    if (cudaEventSynchronize(d->ev_scan1) != cudaSuccess) return -1.0;
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, d->ev_scan0, d->ev_scan1) != cudaSuccess) return -1.0;
    return (double)ms;
}

void ss_queries_destroy(ss_queries* q) {
    if (!q) return;
    cudaSetDevice(q->ctx->device);
    cudaStreamSynchronize(q->ctx->stream);
    CacheFrees cache;
    delete q;
}

int ss_dict_match_dev(ss_dict* d, ss_queries* q, int mode, const double* d_targets, int k, uint32_t* d_out_idx, double* d_out_dist) {
    if (!d || !q) return set_error(d ? d->ctx : nullptr, SS_ERR_INVALID, "dict / queries is NULL");
    ss_ctx* ctx = d->ctx;
    if (q->ctx != ctx) return set_error(ctx, SS_ERR_INVALID, "dict and queries belong to different contexts");
    if (q->c != d->c) return set_error(ctx, SS_ERR_INVALID, "ncoeffs mismatch: dict %d, queries %d", d->c, q->c);
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "match against an empty dictionary");
    if (q->nq && (!d_out_idx || !d_out_dist)) return set_error(ctx, SS_ERR_INVALID, "output pointers are NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    if (mode == SS_COSINE_REF) {
        if (k != 1) return set_error(ctx, SS_ERR_INVALID, "SS_COSINE_REF returns one match per query (k must be 1, got %d)", k);
        SS_TRY(dtw_match_finish(d));  // a pending SS_DTW match shares the dictionary's workspaces
        d->last_scan_kind = 4;
        return cosine_match_dev(d, q, d_targets, d_out_idx, d_out_dist);
    }
    if (mode == SS_DTW) return dtw_match_dev(d, q, k, d_out_idx, d_out_dist);
    if (mode == SS_DTW_TARGET) return dtw_match_dev(d, q, k, d_out_idx, d_out_dist, /*target=*/true, d_targets);
    return set_error(ctx, SS_ERR_INVALID, "unknown match mode %d", mode);
}

int ss_dict_match(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int mode, const double* targets,
                  int k, uint32_t* out_idx, double* out_dist) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "match against an empty dictionary");
    if (k < 1 || k > SS_MAX_TOPK) return set_error(ctx, SS_ERR_INVALID, "k must be in 1..%d (got %d)", SS_MAX_TOPK, k);
    if (nq && (!out_idx || !out_dist)) return set_error(ctx, SS_ERR_INVALID, "output pointers are NULL");
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, d->c));
    SS_TRY(targets_check(ctx, mode, targets, nq));
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!d->scratch_q) {
        d->scratch_q = new (std::nothrow) ss_queries();
        if (!d->scratch_q) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
        d->scratch_q->ctx = ctx;
        d->scratch_q->c = d->c;
    }
    ss_queries* q = d->scratch_q;
    auto body = [&]() -> int {
        SS_TRY(dtw_match_finish(d));  // a pending asynchronous match still owns the workspaces
        TraceTimer tt(ctx);
        SS_TRY(queries_fill(q, q_mfcc, q_frame_offsets, nq));
        tt.lap("ss_dict_match: queries_fill");
        SS_CUDA(ctx, d->d_res_idx.reserve(nq * (size_t)k));
        SS_CUDA(ctx, d->d_res_dist.reserve(nq * (size_t)k));
        const bool use_targets = targets && (mode == SS_COSINE_REF || mode == SS_DTW_TARGET);
        if (use_targets) SS_TRY(upload(ctx, d->d_res_targets, targets, nq));
        SS_TRY(ss_dict_match_dev(d, q, mode, use_targets ? d->d_res_targets.p : nullptr, k, d->d_res_idx.p, d->d_res_dist.p));
        tt.lap("ss_dict_match: first stage");
        // ONE blocking point per call: the result copies (into the caller's pageable or pinned buffers) queue behind the
        // match; the uncertified count reaches pinned memory ahead of them, so the fallback decision costs no extra round
        // trip. Only if a fallback stage had to run are the results copied again.
        for (int pass = 0; pass < 2; pass++) {
            if (nq) {
                SS_CUDA(ctx, cudaMemcpyAsync(out_idx, d->d_res_idx.p, nq * (size_t)k * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
                SS_CUDA(ctx, cudaMemcpyAsync(out_dist, d->d_res_dist.p, nq * (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            }
            SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            if (pass || mode == SS_COSINE_REF) break;
            SS_TRY(dtw_match_finish(d));
            if (!d->last_tc_fallback && !d->last_exhaustive) break;
        }
        return SS_OK;
    };
    const int rc = body();
    if (rc != SS_OK) cudaStreamSynchronize(ctx->stream);
    return rc;
}

// SoundSequence::from_distances for SS_COSINE_REF. Like the cosine match, the walk first completes a pending asynchronous
// SS_DTW match; it has its own workspaces and leaves the ss_dict_last_* counters as the last match left them.
int ss_dict_walk_dev(ss_dict* d, ss_queries* start, const double* d_distances, size_t nsteps, uint32_t* d_out_idx, double* d_out_dist) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (nsteps && (!d_distances || !d_out_idx || !d_out_dist)) return set_error(ctx, SS_ERR_INVALID, "distance / output pointers are NULL");
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "walk over an empty dictionary");
    if (!start) return set_error(ctx, SS_ERR_INVALID, "start is NULL");
    if (start->ctx != ctx) return set_error(ctx, SS_ERR_INVALID, "dict and start belong to different contexts");
    if (start->c != d->c) return set_error(ctx, SS_ERR_INVALID, "ncoeffs mismatch: dict %d, start %d", d->c, start->c);
    if (start->nq != 1) return set_error(ctx, SS_ERR_INVALID, "start must hold exactly one query (got %zu)", start->nq);
    if (nsteps > 0xFFFFFFFFull) return set_error(ctx, SS_ERR_INVALID, "too many steps");
    if (!nsteps) return SS_OK;
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SS_TRY(dtw_match_finish(d));  // a pending SS_DTW match completes first, as before a cosine match
    return cosine_walk_dev(d, start->d_mfcc.p, start->d_off.p, d_distances, nsteps, d_out_idx, d_out_dist);
}

int ss_dict_walk(ss_dict* d, const double* start_mfcc, size_t start_frames, const double* distances, size_t nsteps, uint32_t* out_idx,
                 double* out_dist) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (nsteps && (!distances || !out_idx || !out_dist)) return set_error(ctx, SS_ERR_INVALID, "distance / output pointers are NULL");
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "walk over an empty dictionary");
    if (start_frames && !start_mfcc) return set_error(ctx, SS_ERR_INVALID, "start_mfcc is NULL");
    if (start_frames > 0x7FFFFFFFull / (uint64_t)d->c) return set_error(ctx, SS_ERR_INVALID, "start sound too long");
    if (nsteps > 0xFFFFFFFFull) return set_error(ctx, SS_ERR_INVALID, "too many steps");
    if (!nsteps) return SS_OK;
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    auto body = [&]() -> int {
        SS_TRY(dtw_match_finish(d));
        d->h_walk_off[0] = 0;
        d->h_walk_off[1] = start_frames;
        SS_TRY(upload(ctx, d->d_walk_start, start_mfcc, start_frames * (size_t)d->c));
        SS_TRY(upload(ctx, d->d_walk_off, d->h_walk_off, 2));
        SS_TRY(upload(ctx, d->d_walk_targets, distances, nsteps));
        SS_CUDA(ctx, d->d_walk_idx.reserve(nsteps));
        SS_CUDA(ctx, d->d_walk_dist.reserve(nsteps));
        SS_TRY(cosine_walk_dev(d, d->d_walk_start.p, d->d_walk_off.p, d->d_walk_targets.p, nsteps, d->d_walk_idx.p, d->d_walk_dist.p));
        // ONE blocking point per call
        SS_CUDA(ctx, cudaMemcpyAsync(out_idx, d->d_walk_idx.p, nsteps * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaMemcpyAsync(out_dist, d->d_walk_dist.p, nsteps * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return SS_OK;
    };
    const int rc = body();
    if (rc != SS_OK) cudaStreamSynchronize(ctx->stream);
    return rc;
}

// SoundSequence::from_distances for SS_DTW_TARGET (DESIGN.md §3.1i), with ss_dict_walk's checks and ordering. The walk is exact
// f64 DTW against every segment, so ss_dict_set_scan does not apply; the band does.
int ss_dict_walk_dtw_dev(ss_dict* d, ss_queries* start, const double* d_distances, size_t nsteps, uint32_t* d_out_idx, double* d_out_dist) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (nsteps && (!d_out_idx || !d_out_dist)) return set_error(ctx, SS_ERR_INVALID, "output pointers are NULL");
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "walk over an empty dictionary");
    if (!start) return set_error(ctx, SS_ERR_INVALID, "start is NULL");
    if (start->ctx != ctx) return set_error(ctx, SS_ERR_INVALID, "dict and start belong to different contexts");
    if (start->c != d->c) return set_error(ctx, SS_ERR_INVALID, "ncoeffs mismatch: dict %d, start %d", d->c, start->c);
    if (start->nq != 1) return set_error(ctx, SS_ERR_INVALID, "start must hold exactly one query (got %zu)", start->nq);
    if (nsteps > 0xFFFFFFFFull) return set_error(ctx, SS_ERR_INVALID, "too many steps");
    if (!nsteps) return SS_OK;
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SS_TRY(dtw_match_finish(d));  // a pending SS_DTW match completes first, as before a cosine walk
    return dtw_walk_dev(d, start->d_mfcc.p, start->d_off.p, start->h_off[1], d_distances, nsteps, d_out_idx, d_out_dist);
}

int ss_dict_walk_dtw(ss_dict* d, const double* start_mfcc, size_t start_frames, const double* distances, size_t nsteps, uint32_t* out_idx,
                     double* out_dist) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (nsteps && (!out_idx || !out_dist)) return set_error(ctx, SS_ERR_INVALID, "output pointers are NULL");
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "walk over an empty dictionary");
    if (start_frames && !start_mfcc) return set_error(ctx, SS_ERR_INVALID, "start_mfcc is NULL");
    if (start_frames > 0x7FFFFFFFull / (uint64_t)d->c) return set_error(ctx, SS_ERR_INVALID, "start sound too long");
    if (nsteps > 0xFFFFFFFFull) return set_error(ctx, SS_ERR_INVALID, "too many steps");
    SS_TRY(targets_check(ctx, SS_DTW_TARGET, distances, nsteps));
    if (!nsteps) return SS_OK;
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    auto body = [&]() -> int {
        SS_TRY(dtw_match_finish(d));
        d->h_walk_off[0] = 0;
        d->h_walk_off[1] = start_frames;
        SS_TRY(upload(ctx, d->d_walk_start, start_mfcc, start_frames * (size_t)d->c));
        SS_TRY(upload(ctx, d->d_walk_off, d->h_walk_off, 2));
        if (distances) SS_TRY(upload(ctx, d->d_walk_targets, distances, nsteps));
        SS_CUDA(ctx, d->d_walk_idx.reserve(nsteps));
        SS_CUDA(ctx, d->d_walk_dist.reserve(nsteps));
        SS_TRY(dtw_walk_dev(d, d->d_walk_start.p, d->d_walk_off.p, start_frames, distances ? d->d_walk_targets.p : nullptr, nsteps, d->d_walk_idx.p,
                            d->d_walk_dist.p));
        // ONE blocking point per call
        SS_CUDA(ctx, cudaMemcpyAsync(out_idx, d->d_walk_idx.p, nsteps * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaMemcpyAsync(out_dist, d->d_walk_dist.p, nsteps * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return SS_OK;
    };
    const int rc = body();
    if (rc != SS_OK) cudaStreamSynchronize(ctx->stream);
    return rc;
}

// DTW warping paths (DESIGN.md §3.1e). Alignment takes indices, not a matcher: it works whatever mode the dictionary was last
// matched in. Like a walk it first completes a pending SS_DTW match, has its own workspaces and leaves the ss_dict_last_*
// counters as the last match left them.
static size_t align_capacity_dev(const ss_dict* d, const uint64_t* h_qoff, size_t nq) {
    const uint64_t wpad = std::max<uint32_t>(d->max_len, 1) - 1;
    size_t cells = 0;
    for (size_t p = 0; p < nq; p++)
        if (h_qoff[p + 1] > h_qoff[p]) cells += h_qoff[p + 1] - h_qoff[p] + wpad;
    return cells;
}

int ss_dict_align_dev(ss_dict* d, ss_queries* q, const uint32_t* d_seg_idx, uint32_t* d_out_path, size_t path_capacity,
                      uint64_t* d_out_path_offsets, double* d_out_dist) {
    if (!d || !q) return set_error(d ? d->ctx : nullptr, SS_ERR_INVALID, "dict / queries is NULL");
    ss_ctx* ctx = d->ctx;
    if (q->ctx != ctx) return set_error(ctx, SS_ERR_INVALID, "dict and queries belong to different contexts");
    if (q->c != d->c) return set_error(ctx, SS_ERR_INVALID, "ncoeffs mismatch: dict %d, queries %d", d->c, q->c);
    if (!d_out_path_offsets) return set_error(ctx, SS_ERR_INVALID, "d_out_path_offsets is NULL");
    if (q->nq && (!d_seg_idx || !d_out_dist)) return set_error(ctx, SS_ERR_INVALID, "index / distance pointers are NULL");
    const size_t need = align_capacity_dev(d, q->h_off.data(), q->nq);
    if (path_capacity < need)
        return set_error(ctx, SS_ERR_INVALID, "path_capacity %zu < %zu cells (sum of Lq + Ld_max - 1 over non-empty queries)", path_capacity, need);
    if (need && !d_out_path) return set_error(ctx, SS_ERR_INVALID, "d_out_path is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SS_TRY(dtw_match_finish(d));  // a pending SS_DTW match completes first (its d_out_idx may be this call's d_seg_idx)
    return dtw_align_dev(d, q->d_mfcc.p, q->d_off.p, q->h_off.data(), q->nq, d_seg_idx, d_out_path, d_out_path_offsets, d_out_dist);
}

int ss_dict_align(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, const uint32_t* seg_idx, uint32_t* out_path,
                  size_t path_capacity, uint64_t* out_path_offsets, double* out_dist) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (!out_path_offsets) return set_error(ctx, SS_ERR_INVALID, "out_path_offsets is NULL");
    if (nq && (!seg_idx || !out_dist)) return set_error(ctx, SS_ERR_INVALID, "index / distance pointers are NULL");
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, d->c));
    std::vector<uint64_t> off(nq + 1, 0);
    size_t need = 0;
    for (size_t p = 0; p < nq; p++) {
        off[p + 1] = q_frame_offsets[p + 1] - q_frame_offsets[0];
        if (seg_idx[p] == 0xFFFFFFFFu) continue;
        const uint32_t s = seg_idx[p] - d->index_base;
        if (seg_idx[p] < d->index_base || s >= d->nseg)
            return set_error(ctx, SS_ERR_INVALID, "seg_idx[%zu] = %u is outside [%u, %u)", p, seg_idx[p], d->index_base,
                             (uint32_t)(d->index_base + d->nseg));
        const uint64_t lq = off[p + 1] - off[p], ld = d->h_off[s + 1] - d->h_off[s];
        if (lq && ld) need += lq + ld - 1;
    }
    if (path_capacity < need)
        return set_error(ctx, SS_ERR_INVALID, "path_capacity %zu < %zu cells (sum of Lq + Ld - 1 over the pairs)", path_capacity, need);
    if (need && !out_path) return set_error(ctx, SS_ERR_INVALID, "out_path is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    auto body = [&]() -> int {
        SS_TRY(dtw_match_finish(d));
        SS_TRY(upload(ctx, d->d_align_q, q_mfcc ? q_mfcc + q_frame_offsets[0] * d->c : nullptr, (size_t)off[nq] * d->c));
        SS_TRY(upload(ctx, d->d_align_qoff, off.data(), nq + 1));
        SS_TRY(upload(ctx, d->d_align_seg, seg_idx, nq));
        SS_CUDA(ctx, d->d_align_path.reserve(2 * align_capacity_dev(d, off.data(), nq)));
        SS_CUDA(ctx, d->d_align_off.reserve(nq + 1));
        SS_CUDA(ctx, d->d_align_dist.reserve(nq));
        SS_TRY(dtw_align_dev(d, d->d_align_q.p, d->d_align_qoff.p, off.data(), nq, d->d_align_seg.p, d->d_align_path.p, d->d_align_off.p,
                             d->d_align_dist.p));
        SS_CUDA(ctx, cudaMemcpyAsync(out_path_offsets, d->d_align_off.p, (nq + 1) * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
        if (nq) SS_CUDA(ctx, cudaMemcpyAsync(out_dist, d->d_align_dist.p, nq * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const uint64_t cells = out_path_offsets[nq];  // <= need: every path is at most Lq + Ld - 1 cells
        if (cells) {
            SS_CUDA(ctx, cudaMemcpyAsync(out_path, d->d_align_path.p, cells * 2 * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
        return SS_OK;
    };
    const int rc = body();
    if (rc != SS_OK) cudaStreamSynchronize(ctx->stream);
    return rc;
}

// Subsequence DTW (A12, DESIGN.md §3.1g). Like an alignment it takes no matcher state: a pending SS_DTW match completes first,
// and the ss_dict_last_* counters stay as the last match left them. The band does not apply.
int ss_dict_locate_dev(ss_dict* d, ss_queries* q, int k, uint32_t* d_out_idx, uint32_t* d_out_start, uint32_t* d_out_end, double* d_out_cost) {
    if (!d || !q) return set_error(d ? d->ctx : nullptr, SS_ERR_INVALID, "dict / queries is NULL");
    ss_ctx* ctx = d->ctx;
    if (q->ctx != ctx) return set_error(ctx, SS_ERR_INVALID, "dict and queries belong to different contexts");
    if (q->c != d->c) return set_error(ctx, SS_ERR_INVALID, "ncoeffs mismatch: dict %d, queries %d", d->c, q->c);
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "locate in an empty dictionary");
    if (k < 1 || k > SS_MAX_TOPK) return set_error(ctx, SS_ERR_INVALID, "k must be in 1..%d (got %d)", SS_MAX_TOPK, k);
    if (q->nq && !d_out_idx) return set_error(ctx, SS_ERR_INVALID, "d_out_idx is NULL");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    SS_TRY(dtw_match_finish(d));  // a pending SS_DTW match shares the exhaustive stage's tables
    return dtw_locate_dev(d, q, k, d_out_idx, d_out_start, d_out_end, d_out_cost);
}

int ss_dict_locate(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int k, uint32_t* out_idx, uint32_t* out_start,
                   uint32_t* out_end, double* out_cost) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "locate in an empty dictionary");
    if (k < 1 || k > SS_MAX_TOPK) return set_error(ctx, SS_ERR_INVALID, "k must be in 1..%d (got %d)", SS_MAX_TOPK, k);
    if (nq && !out_idx) return set_error(ctx, SS_ERR_INVALID, "out_idx is NULL");
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, d->c));
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!d->scratch_q) {
        d->scratch_q = new (std::nothrow) ss_queries();
        if (!d->scratch_q) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
        d->scratch_q->ctx = ctx;
        d->scratch_q->c = d->c;
    }
    ss_queries* q = d->scratch_q;
    auto body = [&]() -> int {
        SS_TRY(dtw_match_finish(d));
        SS_TRY(queries_fill(q, q_mfcc, q_frame_offsets, nq));
        const size_t n = nq * (size_t)k;
        SS_CUDA(ctx, d->d_locate_idx.reserve(n));
        if (out_start) SS_CUDA(ctx, d->d_locate_start.reserve(n));
        if (out_end) SS_CUDA(ctx, d->d_locate_end.reserve(n));
        if (out_cost) SS_CUDA(ctx, d->d_locate_cost.reserve(n));
        SS_TRY(dtw_locate_dev(d, q, k, d->d_locate_idx.p, out_start ? d->d_locate_start.p : nullptr, out_end ? d->d_locate_end.p : nullptr,
                              out_cost ? d->d_locate_cost.p : nullptr));
        if (n) {  // ONE blocking point per call
            SS_CUDA(ctx, cudaMemcpyAsync(out_idx, d->d_locate_idx.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            if (out_start) SS_CUDA(ctx, cudaMemcpyAsync(out_start, d->d_locate_start.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            if (out_end) SS_CUDA(ctx, cudaMemcpyAsync(out_end, d->d_locate_end.p, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            if (out_cost) SS_CUDA(ctx, cudaMemcpyAsync(out_cost, d->d_locate_cost.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        }
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return SS_OK;
    };
    const int rc = body();
    if (rc != SS_OK) cudaStreamSynchronize(ctx->stream);
    return rc;
}

int ss_dict_set_scan(ss_dict* d, int first_stage) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    if (first_stage < 0 || first_stage > 3) return set_error(d->ctx, SS_ERR_INVALID, "first_stage must be 0, 1, 2 or 3");
    SS_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    SS_TRY(dtw_match_finish(d));
    d->scan_pref = first_stage;
    return SS_OK;
}

// Sakoe-Chiba band of the exact DTW (A10, DESIGN.md §3.1f). A pending SS_DTW match completes first, under the radius it
// started with: its first stage already ran with that radius.
int ss_dict_set_dtw_band(ss_dict* d, uint32_t radius) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    SS_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    SS_TRY(dtw_match_finish(d));
    d->dtw_band = radius;
    return SS_OK;
}

uint32_t ss_dict_dtw_band(const ss_dict* d) { return d ? d->dtw_band : 0; }

static int debug_scan(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, float* out_scan, double* out_mu,
                      float* out_scale, float* out_s);

int ss_dict_debug_tc_scan(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, float* out_scan, double* out_mu,
                          float* out_scale) {
    return debug_scan(d, q_mfcc, q_frame_offsets, nq, out_scan, out_mu, out_scale, nullptr);
}
int ss_dict_debug_h2_scan(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, float* out_scan, double* out_mu,
                          float* out_scale, float* out_s) {
    if (!out_s) return set_error(d ? d->ctx : nullptr, SS_ERR_INVALID, "out_s is NULL");
    return debug_scan(d, q_mfcc, q_frame_offsets, nq, out_scan, out_mu, out_scale, out_s);
}

// out_s == NULL: the fp32-DP tensor-core scan; else the packed-half scan (and its cost scale S)
static int debug_scan(ss_dict* d, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, float* out_scan, double* out_mu,
                      float* out_scale, float* out_s) {
    if (!d) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    ss_ctx* ctx = d->ctx;
    if (!out_scan || !out_mu || !out_scale) return set_error(ctx, SS_ERR_INVALID, "output pointers are NULL");
    if (d->nseg == 0) return set_error(ctx, SS_ERR_EMPTY_DICT, "empty dictionary");
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, d->c));
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    ss_queries q;
    q.ctx = ctx;
    q.c = d->c;
    SS_TRY(queries_fill(&q, q_mfcc, q_frame_offsets, nq));
    const size_t nslots = (nq + 127) / 128 * 128, nseg = d->nseg;
    DevBuf<float> d_out;
    SS_CUDA(ctx, d_out.reserve(nslots * nseg));
    SS_CUDA(ctx, cudaMemsetAsync(d_out.p, 0xFF, nslots * nseg * sizeof(float), ctx->stream));  // NaN = not evaluated
    std::vector<uint32_t> slot_qid;
    SS_TRY(dtw_match_finish(d));
    int rc = out_s ? dtw_h2_debug_scan(d, &q, d_out.p, &slot_qid, out_mu, out_scale, out_s) : dtw_tc_debug_scan(d, &q, d_out.p, &slot_qid, out_mu, out_scale);
    if (rc != SS_OK) {
        cudaStreamSynchronize(ctx->stream);
        return rc;
    }
    for (size_t i = 0; i < nq * nseg; i++) out_scan[i] = std::numeric_limits<float>::quiet_NaN();
    for (size_t s = 0; s < slot_qid.size(); s++) {  // scan rows are in length-sorted slot order: back to query order
        const uint32_t qid = slot_qid[s];
        if (qid == 0xFFFFFFFFu) continue;
        SS_CUDA(ctx, cudaMemcpyAsync(out_scan + (size_t)qid * nseg, d_out.p + s * nseg, nseg * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    }
    SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return SS_OK;
}

int ss_topk_merge_dev(ss_ctx* ctx, const uint32_t* d_idx, const double* d_dist, int nlists, size_t nq, int k, uint32_t* d_out_idx,
                      double* d_out_dist) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (nq && (!d_idx || !d_dist || !d_out_idx || !d_out_dist)) return set_error(ctx, SS_ERR_INVALID, "NULL pointer");
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    return topk_merge_dev(ctx, d_idx, d_dist, nlists, nq, k, d_out_idx, d_out_dist);
}

}  // extern "C"
