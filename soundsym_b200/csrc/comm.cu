// comm.cu — the matcher across the GPUs of one box, INSIDE the library (SURVEY.md §8b / §8e): the dictionary is partitioned
// into contiguous shards (one ss_dict per GPU, global index bases), the query frames cross PCIe once (1/N per GPU) and are
// all-gathered over NVLink, every GPU matches the whole batch against its shard, and the per-shard top-k lists are exchanged
// with ONE ncclAllGather of a contiguous (distance, index) block per rank and merged on every rank by (distance, index) -
// the reference's first-minimum rule (src/sound.rs:361-366) carried across shards.
//
// Two front ends over the same rank-local code:
//   ss_comm_create        one rank per process (torchrun / MPI style; the caller ships the 128-byte id to the other ranks)
//   ss_dict_create_sharded / ss_sharded_dict_match   one process, one worker thread per GPU (ncclCommInitAll) - what a
//                         Rust SoundDictionary bound to this library calls: same signature as the single-GPU match.
// NCCL is bound at run time with dlopen (the copy already mapped in the process, else $SS_NCCL_LIB - the Python loader points
// it at the one PyTorch ships - else the system libnccl.so.2): the library has no link-time dependency on it and single-GPU
// users never load it.
#include <dlfcn.h>
#include <nccl.h>  // types and prototypes only; every call goes through the table below

#include <algorithm>
#include <condition_variable>
#include <mutex>
#include <thread>

#include "match.cuh"

namespace ss {

struct NcclApi {
    decltype(&ncclGetUniqueId) GetUniqueId;
    decltype(&ncclCommInitRank) CommInitRank;
    decltype(&ncclCommInitAll) CommInitAll;
    decltype(&ncclCommDestroy) CommDestroy;
    decltype(&ncclAllGather) AllGather;
    decltype(&ncclGetErrorString) GetErrorString;
};

static const NcclApi* nccl_api(std::string* err) {
    static std::mutex mu;
    static NcclApi api;
    static bool ok = false, tried = false;
    static std::string why;
    std::lock_guard<std::mutex> lock(mu);
    if (!tried) {
        tried = true;
        // 1. a copy that is already mapped (PyTorch's bundled one, if torch was imported first); 2. $SS_NCCL_LIB (the Python
        // loader points it at the bundled copy, so that a later `import torch` finds the NCCL it was built against under the
        // same soname); 3. the system library
        void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);
        if (!h) {
            const char* env = getenv("SS_NCCL_LIB");
            if (env && *env) h = dlopen(env, RTLD_NOW | RTLD_LOCAL);
        }
        for (const char* name : {"libnccl.so.2", "libnccl.so"}) {
            if (h) break;
            h = dlopen(name, RTLD_NOW | RTLD_LOCAL);
        }
        if (!h) {
            why = std::string("cannot load NCCL: ") + (dlerror() ? dlerror() : "libnccl.so.2 not found");
        } else {
            bool all = true;
            auto sym = [&](const char* n) {
                void* p = dlsym(h, n);
                if (!p) all = false, why = std::string("NCCL symbol missing: ") + n;
                return p;
            };
            api.GetUniqueId = reinterpret_cast<decltype(api.GetUniqueId)>(sym("ncclGetUniqueId"));
            api.CommInitRank = reinterpret_cast<decltype(api.CommInitRank)>(sym("ncclCommInitRank"));
            api.CommInitAll = reinterpret_cast<decltype(api.CommInitAll)>(sym("ncclCommInitAll"));
            api.CommDestroy = reinterpret_cast<decltype(api.CommDestroy)>(sym("ncclCommDestroy"));
            api.AllGather = reinterpret_cast<decltype(api.AllGather)>(sym("ncclAllGather"));
            api.GetErrorString = reinterpret_cast<decltype(api.GetErrorString)>(sym("ncclGetErrorString"));
            ok = all;
        }
    }
    if (!ok && err) *err = why;
    return ok ? &api : nullptr;
}

#define SS_NCCL(ctx, api, expr)                                                                                          \
    do {                                                                                                                 \
        ncclResult_t _r = (expr);                                                                                        \
        if (_r != ncclSuccess)                                                                                           \
            return ss::set_error((ctx), SS_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, (api)->GetErrorString(_r), __FILE__, __LINE__); \
    } while (0)

}  // namespace ss

struct ss_comm {
    ss_ctx* ctx = nullptr;
    ncclComm_t comm = nullptr;
    int nranks = 1, rank = 0;
    ss::DevBuf<unsigned char> d_gather;   // [nranks] x {dist f64 [nq x k], idx u32 [nq x k]}
    ss::DevBuf<uint32_t> d_out_idx;       // host-buffer entry point: merged results before they leave the device
    ss::DevBuf<double> d_out_dist, d_targets;
    ss_queries* scratch_q = nullptr;
    ~ss_comm() { delete scratch_q; }
};

namespace ss {

// list-major exchange block -> merged top-k by (distance, index); block l = {dist f64 [nq x k], idx u32 [nq x k]} at l * stride
__global__ void k_topk_merge_blocks(const unsigned char* __restrict__ blocks, size_t stride, int nlists, size_t nq, int k,
                                    uint32_t* __restrict__ out_idx, double* __restrict__ out_dist) {
    const size_t qi = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (qi >= nq) return;
    double dv[SS_MAX_TOPK];
    uint32_t iv[SS_MAX_TOPK];
    int n = 0;
    for (int l = 0; l < nlists; l++) {
        const double* dist = reinterpret_cast<const double*>(blocks + (size_t)l * stride);
        const uint32_t* idx = reinterpret_cast<const uint32_t*>(blocks + (size_t)l * stride + nq * (size_t)k * sizeof(double));
        for (int s = 0; s < k; s++) {
            const double dd = dist[qi * k + s];
            const uint32_t ii = idx[qi * k + s];
            if (ii != 0xFFFFFFFFu && dd == dd) topk_push(dv, iv, n, k, dd, ii);  // as k_topk_merge (exact.cu)
        }
    }
    topk_store(dv, iv, n, k, 0, out_idx + qi * k, out_dist + qi * k);
}

static size_t exchange_stride(size_t nq, int k) { return (nq * (size_t)k * 12 + 255) / 256 * 256; }

// fills a query batch with 1/nranks of the frames copied from the host by THIS rank and the rest all-gathered over NVLink
static int queries_fill_sharded(ss_comm* cm, ss_queries* q, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq) {
    ss_ctx* ctx = cm->ctx;
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) return set_error(ctx, SS_ERR_CUDA, "%s", why.c_str());
    SS_TRY(queries_prepare(q, q_frame_offsets, nq));
    const uint64_t base = nq ? q_frame_offsets[0] : 0;
    const size_t total = (size_t)q->total_frames * q->c;
    const size_t chunk = ((total + cm->nranks - 1) / cm->nranks + 1) & ~(size_t)1;  // doubles per rank
    SS_CUDA(ctx, q->d_mfcc.reserve(std::max<size_t>(chunk * cm->nranks, 1)));
    const size_t b = std::min(total, chunk * cm->rank), e = std::min(total, b + chunk);
    if (e > b)
        SS_CUDA(ctx, cudaMemcpyAsync(q->d_mfcc.p + b, q_mfcc + base * q->c + b, (e - b) * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    SS_TRY(upload(ctx, q->d_off, q->h_off.data(), nq + 1));
    SS_TRY(dtw_tc_queries_group(q));  // host work, overlaps the copies
    if (chunk) SS_NCCL(ctx, api, api->AllGather(q->d_mfcc.p + chunk * cm->rank, q->d_mfcc.p, chunk, ncclDouble, cm->comm, ctx->stream));
    return SS_OK;
}

static int match_sharded_dev(ss_dict* d, ss_comm* cm, ss_queries* q, int mode, const double* d_targets, int k, uint32_t* d_out_idx,
                             double* d_out_dist) {
    ss_ctx* ctx = d->ctx;
    if (cm->ctx != ctx || q->ctx != ctx) return set_error(ctx, SS_ERR_INVALID, "shard, communicator and queries must share one context");
    if (k < 1 || k > SS_MAX_TOPK) return set_error(ctx, SS_ERR_INVALID, "k must be in 1..%d (got %d)", SS_MAX_TOPK, k);
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) return set_error(ctx, SS_ERR_CUDA, "%s", why.c_str());
    const size_t nq = q->nq, stride = exchange_stride(nq, k);
    SS_CUDA(ctx, cm->d_gather.reserve(std::max<size_t>(stride * cm->nranks, 256)));
    unsigned char* mine = cm->d_gather.p + stride * cm->rank;
    double* l_dist = reinterpret_cast<double*>(mine);
    uint32_t* l_idx = reinterpret_cast<uint32_t*>(mine + nq * (size_t)k * sizeof(double));
    if (d->nseg == 0) {
        // an empty shard (more GPUs than segments) contributes nothing: (inf, 0xFFFFFFFF) everywhere
        if (nq) SS_TRY(fill_result(ctx, l_idx, l_dist, nq * (size_t)k));
    } else {
        SS_TRY(ss_dict_match_dev(d, q, mode, d_targets, k, l_idx, l_dist));
        SS_TRY(dtw_match_finish(d));  // the shard's results are final (fallback stages done) before they are exchanged
    }
    if (nq) {
        SS_NCCL(ctx, api, api->AllGather(mine, cm->d_gather.p, stride, ncclChar, cm->comm, ctx->stream));
        k_topk_merge_blocks<<<ceil_div((long long)nq, 128), 128, 0, ctx->stream>>>(cm->d_gather.p, stride, cm->nranks, nq, k, d_out_idx, d_out_dist);
        SS_LAUNCHED(ctx);
    }
    return SS_OK;
}

}  // namespace ss

using namespace ss;

// ---- one process, one worker thread per GPU ---------------------------------------------------------------------------
struct ss_sharded_dict {
    int n = 0;
    size_t nseg = 0;
    int c = 0;
    std::vector<ss_ctx*> ctxs;
    std::vector<ss_dict*> shards;
    std::vector<ss_comm*> comms;
    // persistent workers: one per GPU, parked on a condition variable between calls
    struct Job {
        const double* q_mfcc;
        const uint64_t* q_off;
        size_t nq;
        int mode;
        const double* targets;
        int k;
        uint32_t* out_idx;
        double* out_dist;
    } job{};
    std::vector<std::thread> workers;
    std::mutex mu;
    std::condition_variable cv_go, cv_done;
    uint64_t generation = 0;
    int remaining = 0;
    bool stop = false;
    std::vector<int> rc;
    std::vector<std::vector<uint32_t>> sink_idx;   // non-root workers' host results (discarded: every rank holds the merged top-k)
    std::vector<std::vector<double>> sink_dist;

    void worker(int r) {
        uint64_t seen = 0;
        cudaSetDevice(ctxs[r]->device);
        for (;;) {
            Job j;
            {
                std::unique_lock<std::mutex> lock(mu);
                cv_go.wait(lock, [&] { return stop || generation != seen; });
                if (stop) return;
                seen = generation;
                j = job;
            }
            uint32_t* oi = j.out_idx;
            double* od = j.out_dist;
            if (r != 0) {
                sink_idx[r].resize(j.nq * (size_t)j.k);
                sink_dist[r].resize(j.nq * (size_t)j.k);
                oi = sink_idx[r].data(), od = sink_dist[r].data();
            }
            const int rcode = ss_dict_match_sharded(shards[r], comms[r], j.q_mfcc, j.q_off, j.nq, j.mode, j.targets, j.k, oi, od);
            {
                std::lock_guard<std::mutex> lock(mu);
                rc[r] = rcode;
                if (--remaining == 0) cv_done.notify_all();
            }
        }
    }
};

extern "C" {

int ss_comm_unique_id(void* out_id) {
    if (!out_id) return set_error(nullptr, SS_ERR_INVALID, "out_id is NULL");
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) return set_error(nullptr, SS_ERR_CUDA, "%s", why.c_str());
    ncclUniqueId id;
    SS_NCCL(nullptr, api, api->GetUniqueId(&id));
    static_assert(sizeof(id) == SS_COMM_ID_BYTES, "ncclUniqueId size");
    memcpy(out_id, &id, sizeof(id));
    return SS_OK;
}

int ss_comm_create(ss_ctx* ctx, int nranks, int rank, const void* id, ss_comm** out) {
    if (!ctx) return set_error(nullptr, SS_ERR_INVALID, "ctx is NULL");
    if (!out || !id) return set_error(ctx, SS_ERR_INVALID, "out / id is NULL");
    *out = nullptr;
    if (nranks < 1 || rank < 0 || rank >= nranks) return set_error(ctx, SS_ERR_INVALID, "rank %d of %d", rank, nranks);
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) return set_error(ctx, SS_ERR_CUDA, "%s", why.c_str());
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    ss_comm* cm = new (std::nothrow) ss_comm();
    if (!cm) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
    cm->ctx = ctx;
    cm->nranks = nranks;
    cm->rank = rank;
    ncclUniqueId uid;
    memcpy(&uid, id, sizeof(uid));
    ncclResult_t r = api->CommInitRank(&cm->comm, nranks, uid, rank);
    if (r != ncclSuccess) {
        delete cm;
        return set_error(ctx, SS_ERR_CUDA, "ncclCommInitRank failed: %s", api->GetErrorString(r));
    }
    *out = cm;
    return SS_OK;
}

int ss_comm_create_all(ss_ctx* const* ctxs, int nctx, ss_comm** out) {
    if (!ctxs || !out || nctx < 1) return set_error(nullptr, SS_ERR_INVALID, "ss_comm_create_all: bad arguments");
    for (int i = 0; i < nctx; i++) out[i] = nullptr;
    std::string why;
    const NcclApi* api = nccl_api(&why);
    if (!api) return set_error(ctxs[0], SS_ERR_CUDA, "%s", why.c_str());
    std::vector<int> devs(nctx);
    for (int i = 0; i < nctx; i++) {
        if (!ctxs[i]) return set_error(nullptr, SS_ERR_INVALID, "ctxs[%d] is NULL", i);
        devs[i] = ctxs[i]->device;
        for (int j = 0; j < i; j++)
            if (devs[j] == devs[i]) return set_error(ctxs[0], SS_ERR_INVALID, "contexts %d and %d share device %d: one shard per GPU", j, i, devs[i]);
    }
    std::vector<ncclComm_t> comms(nctx);
    SS_NCCL(ctxs[0], api, api->CommInitAll(comms.data(), nctx, devs.data()));
    for (int i = 0; i < nctx; i++) {
        ss_comm* cm = new (std::nothrow) ss_comm();
        if (!cm) return set_error(ctxs[0], SS_ERR_NOMEM, "out of host memory");
        cm->ctx = ctxs[i];
        cm->comm = comms[i];
        cm->nranks = nctx;
        cm->rank = i;
        out[i] = cm;
    }
    return SS_OK;
}

void ss_comm_destroy(ss_comm* cm) {
    if (!cm) return;
    cudaSetDevice(cm->ctx->device);
    cudaStreamSynchronize(cm->ctx->stream);
    const NcclApi* api = nccl_api(nullptr);
    if (api && cm->comm) api->CommDestroy(cm->comm);
    delete cm;
}
int ss_comm_rank(const ss_comm* cm) { return cm ? cm->rank : -1; }
int ss_comm_nranks(const ss_comm* cm) { return cm ? cm->nranks : 0; }

int ss_shard_bounds(const uint64_t* frame_offsets, size_t nseg, int nshards, uint64_t* out_cuts) {
    if (!frame_offsets || !out_cuts || nshards < 1) return set_error(nullptr, SS_ERR_INVALID, "ss_shard_bounds: bad arguments");
    const uint64_t base = frame_offsets[0], total = frame_offsets[nseg] - base;
    out_cuts[0] = 0;
    for (int r = 1; r < nshards; r++) {
        // first segment whose start offset reaches r / nshards of the frames (lower_bound), never before the previous cut
        const uint64_t want = base + total * (uint64_t)r / (uint64_t)nshards;
        const uint64_t* p = std::lower_bound(frame_offsets, frame_offsets + nseg + 1, want);
        out_cuts[r] = std::max<uint64_t>(out_cuts[r - 1], std::min<uint64_t>((uint64_t)(p - frame_offsets), nseg));
    }
    out_cuts[nshards] = nseg;
    return SS_OK;
}

int ss_queries_create_sharded(ss_comm* cm, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int ncoeffs, ss_queries** out) {
    if (!cm) return set_error(nullptr, SS_ERR_INVALID, "comm is NULL");
    ss_ctx* ctx = cm->ctx;
    if (!out) return set_error(ctx, SS_ERR_INVALID, "out is NULL");
    *out = nullptr;
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, ncoeffs));
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    ss_queries* q = new (std::nothrow) ss_queries();
    if (!q) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
    q->ctx = ctx;
    q->c = ncoeffs;
    const int rc = queries_fill_sharded(cm, q, q_mfcc, q_frame_offsets, nq);
    if (rc != SS_OK) {
        cudaStreamSynchronize(ctx->stream);
        delete q;
        return rc;
    }
    *out = q;
    return SS_OK;
}

int ss_dict_match_sharded_dev(ss_dict* d, ss_comm* cm, ss_queries* q, int mode, const double* d_targets, int k, uint32_t* d_out_idx,
                              double* d_out_dist) {
    if (!d || !cm || !q) return set_error(d ? d->ctx : nullptr, SS_ERR_INVALID, "shard / comm / queries is NULL");
    if (q->nq && (!d_out_idx || !d_out_dist)) return set_error(d->ctx, SS_ERR_INVALID, "output pointers are NULL");
    SS_CUDA(d->ctx, cudaSetDevice(d->ctx->device));
    return match_sharded_dev(d, cm, q, mode, d_targets, k, d_out_idx, d_out_dist);
}

int ss_dict_match_sharded(ss_dict* d, ss_comm* cm, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int mode,
                          const double* targets, int k, uint32_t* out_idx, double* out_dist) {
    if (!d || !cm) return set_error(d ? d->ctx : nullptr, SS_ERR_INVALID, "shard / comm is NULL");
    ss_ctx* ctx = d->ctx;
    if (k < 1 || k > SS_MAX_TOPK) return set_error(ctx, SS_ERR_INVALID, "k must be in 1..%d (got %d)", SS_MAX_TOPK, k);
    if (mode == SS_COSINE_REF && k != 1) return set_error(ctx, SS_ERR_INVALID, "SS_COSINE_REF returns one match per query (k must be 1, got %d)", k);
    if (nq && (!out_idx || !out_dist)) return set_error(ctx, SS_ERR_INVALID, "output pointers are NULL");
    SS_TRY(queries_check(ctx, q_mfcc, q_frame_offsets, nq, d->c));
    SS_TRY(targets_check(ctx, mode, targets, nq));
    SS_CUDA(ctx, cudaSetDevice(ctx->device));
    if (!cm->scratch_q) {
        cm->scratch_q = new (std::nothrow) ss_queries();
        if (!cm->scratch_q) return set_error(ctx, SS_ERR_NOMEM, "out of host memory");
        cm->scratch_q->ctx = ctx;
        cm->scratch_q->c = d->c;
    }
    ss_queries* q = cm->scratch_q;
    auto body = [&]() -> int {
        SS_TRY(dtw_match_finish(d));
        SS_TRY(queries_fill_sharded(cm, q, q_mfcc, q_frame_offsets, nq));
        SS_CUDA(ctx, cm->d_out_idx.reserve(std::max<size_t>(nq * (size_t)k, 1)));
        SS_CUDA(ctx, cm->d_out_dist.reserve(std::max<size_t>(nq * (size_t)k, 1)));
        const bool use_targets = targets && (mode == SS_COSINE_REF || mode == SS_DTW_TARGET);
        if (use_targets) SS_TRY(upload(ctx, cm->d_targets, targets, nq));
        SS_TRY(match_sharded_dev(d, cm, q, mode, use_targets ? cm->d_targets.p : nullptr, k, cm->d_out_idx.p, cm->d_out_dist.p));
        if (nq) {
            SS_CUDA(ctx, cudaMemcpyAsync(out_idx, cm->d_out_idx.p, nq * (size_t)k * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
            SS_CUDA(ctx, cudaMemcpyAsync(out_dist, cm->d_out_dist.p, nq * (size_t)k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        }
        SS_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        return SS_OK;
    };
    const int rc = body();
    if (rc != SS_OK) cudaStreamSynchronize(ctx->stream);
    return rc;
}

int ss_dict_create_sharded(ss_ctx* const* ctxs, int nctx, const double* mfcc_flat, const uint64_t* frame_offsets, size_t nseg, int ncoeffs,
                           ss_sharded_dict** out) {
    if (!ctxs || nctx < 1 || !ctxs[0]) return set_error(nullptr, SS_ERR_INVALID, "ss_dict_create_sharded: no contexts");
    if (!out) return set_error(ctxs[0], SS_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (!frame_offsets) return set_error(ctxs[0], SS_ERR_INVALID, "frame_offsets is NULL");
    ss_sharded_dict* sd = new (std::nothrow) ss_sharded_dict();
    if (!sd) return set_error(ctxs[0], SS_ERR_NOMEM, "out of host memory");
    sd->n = nctx;
    sd->nseg = nseg;
    sd->c = ncoeffs;
    sd->ctxs.assign(ctxs, ctxs + nctx);
    sd->shards.assign(nctx, nullptr);
    sd->comms.assign(nctx, nullptr);
    sd->rc.assign(nctx, SS_OK);
    sd->sink_idx.resize(nctx);
    sd->sink_dist.resize(nctx);
    std::vector<uint64_t> cuts(nctx + 1);
    int rc = ss_shard_bounds(frame_offsets, nseg, nctx, cuts.data());
    for (int r = 0; r < nctx && rc == SS_OK; r++) {
        rc = ss_dict_create(ctxs[r], mfcc_flat, frame_offsets + cuts[r], (size_t)(cuts[r + 1] - cuts[r]), ncoeffs, (uint32_t)cuts[r], &sd->shards[r]);
        if (rc != SS_OK) set_error(ctxs[0], rc, "shard %d: %s", r, ss_last_error(ctxs[r]));
    }
    if (rc == SS_OK) rc = ss_comm_create_all(ctxs, nctx, sd->comms.data());
    if (rc != SS_OK) {
        ss_sharded_dict_destroy(sd);
        return rc;
    }
    for (int r = 0; r < nctx; r++) sd->workers.emplace_back([sd, r] { sd->worker(r); });
    *out = sd;
    return SS_OK;
}

void ss_sharded_dict_destroy(ss_sharded_dict* sd) {
    if (!sd) return;
    {
        std::lock_guard<std::mutex> lock(sd->mu);
        sd->stop = true;
    }
    sd->cv_go.notify_all();
    for (auto& t : sd->workers) t.join();
    for (ss_comm* c : sd->comms) ss_comm_destroy(c);
    for (ss_dict* d : sd->shards) ss_dict_destroy(d);
    delete sd;
}

size_t ss_sharded_dict_len(const ss_sharded_dict* sd) { return sd ? sd->nseg : 0; }

int ss_sharded_dict_set_dtw_band(ss_sharded_dict* sd, uint32_t radius) {
    if (!sd) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    for (ss_dict* d : sd->shards) SS_TRY(ss_dict_set_dtw_band(d, radius));
    return SS_OK;
}
int ss_sharded_dict_nshards(const ss_sharded_dict* sd) { return sd ? sd->n : 0; }

int ss_sharded_dict_match(ss_sharded_dict* sd, const double* q_mfcc, const uint64_t* q_frame_offsets, size_t nq, int mode, const double* targets,
                          int k, uint32_t* out_idx, double* out_dist) {
    if (!sd) return set_error(nullptr, SS_ERR_INVALID, "dict is NULL");
    if (sd->nseg == 0) return set_error(sd->ctxs[0], SS_ERR_EMPTY_DICT, "match against an empty dictionary");
    {
        std::lock_guard<std::mutex> lock(sd->mu);
        sd->job = {q_mfcc, q_frame_offsets, nq, mode, targets, k, out_idx, out_dist};
        sd->remaining = sd->n;
        sd->generation++;
    }
    sd->cv_go.notify_all();
    {
        std::unique_lock<std::mutex> lock(sd->mu);
        sd->cv_done.wait(lock, [&] { return sd->remaining == 0; });
    }
    for (int r = 0; r < sd->n; r++)
        if (sd->rc[r] != SS_OK) return set_error(sd->ctxs[0], sd->rc[r], "shard %d: %s", r, ss_last_error(sd->ctxs[r]));
    return SS_OK;
}

}  // extern "C"
