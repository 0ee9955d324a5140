// libvpca C ABI (include/vpca.h): context management, host<->device staging and the call sequence
// encode -> Gram -> (cross-GPU reduce) -> symmetrize -> centering -> eigensolve.
// Mirrors the method set of the reference's VariantsPcaDriver
// (src/main/scala/com/google/cloud/genomics/spark/examples/VariantsPca.scala:81-286); see vpca.h for the mapping.
//
// Threading model (the reference runs the bodies of `mapPartitions` concurrently, one task thread per core,
// VariantsPca.scala:184-189): host-input calls (accumulate_calls / _u16 / _bits / _bed / dense-from-host) take one
// of `staging_lanes` LANES -- a private stream pair, double-buffered staging and a private Gram schedule -- and hold
// the context mutex only for bookkeeping, never across a copy, a kernel or a stream synchronisation.  So the H2D copy
// and encode of one task overlap the Gram kernel of another; a partition's staging Gram (slot) is private to the
// task that owns the partition id, and `commit` folds it into the Gram with integer adds on the context's stream.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cmath>
#include <condition_variable>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <map>
#include <mutex>
#include <string>
#include <vector>

#include "vpca_internal.h"

using namespace vpca;

namespace {
thread_local std::string tls_error;
thread_local const vpca_ctx* tls_error_ctx = nullptr;
thread_local std::string tls_error_copy;
}   // namespace

struct vpca_ctx {
    vpca_config cfg{};
    int n = 0;
    int elem_bits = 8;   // 8 = int8, 16 = bf16, 4 = packed e2m1
    int max_mult = 2;
    int num_pc = 2;
    cudaStream_t stream = nullptr;
    bool own_stream = false;
    int32_t* d_S = nullptr;
    bool own_S = false;
    int band_row0 = 0, band_rows = 0;   // rows of the Gram this context stores (band_rows == n: all of them)
    // projecting context (vpca_create_projecting): n_proj samples beyond the n fitted ones.  The Gram buffer is
    // (n + n_proj) x n, pitch n: rows [0, n) the fitted Gram, rows [n, n + n_proj) the cross block.  Input sample s is
    // row d_rows[s] of the genotype tiles (d_rows == nullptr: identity).
    int n_proj = 0;
    int32_t* d_rows = nullptr;
    int proj_k = 0;                // k of the last vpca_compute_pca (0: none since the Gram last changed)
    double* d_proj = nullptr;      // projection scratch + result (eig_project)
    int rows() const { return n + n_proj; }                                        // rows of X
    size_t gram_cells() const { return (size_t)(band_rows + n_proj) * (size_t)n; }   // int32 cells of d_S
    // scoring context (vpca_create_scoring): no Gram; the n samples are scored against a saved model that lives on the
    // device.  An accumulator holds (T, r) of the model's k columns: n x k doubles, then n int64 (model.cu).
    bool scoring = false;
    int model_k = 0, model_nfit = 0;
    int64_t model_nv = 0;
    double* d_model_L = nullptr;      // model_nv x model_k
    int32_t* d_model_n = nullptr;     // model_nv
    double* d_model_terms = nullptr;  // lambda[k] | a[k] | b[k] | matrix mean
    double* d_direct = nullptr;       // accumulator of direct input (partition_id < 0), in call order
    int64_t direct_matched = 0;
    std::mutex direct_mu;             // direct scoring calls add into d_direct one at a time
    struct Scored {
        double* d_acc = nullptr;
        int64_t matched = 0;
    };
    std::map<int64_t, Scored> scored;   // committed partitions in ascending id
    char* d_scratch = nullptr;          // model passes on the context's stream (panels routes, vpca_score_project)
    int64_t cap_scratch = 0;
    size_t slot_bytes() const {
        return scoring ? (size_t)n * (model_k + 1) * sizeof(double) : (size_t)rows() * n * sizeof(int32_t);
    }
    bool finalized = false;
    bool pca_done = false;
    GramPlan plan;        // schedule state of the launches on `stream` (device-resident input)
    EigWork eig;
    bool eig_ready = false;
    JoinWork join;        // multi-dataset keying (join.cu); one join at a time (join_mu)
    std::mutex join_mu;

    struct Slot {
        int64_t pid = -1;
        int32_t* d_S = nullptr;
        bool used = false;
        bool busy = false;             // a call of the owning task is in flight
        bool fresh = false;            // still to be zeroed by its first batch
        int64_t nv = 0;
        int64_t matched = 0;           // scoring: variants with a model row
        cudaEvent_t ev_free = nullptr; // recorded after the commit that last read the slot
    };
    std::vector<Slot> slots;

    // One lane = everything a host-input call needs to run without the other lanes: streams, double-buffered CSR /
    // dense staging, error flags and its own Gram schedule (the speed-weighted stream-K shares must not change under
    // a running kernel, so they are per stream).
    struct Lane {
        cudaStream_t stream = nullptr, copy_stream = nullptr;
        int64_t* d_off[2] = {nullptr, nullptr};
        int32_t* d_idx[2] = {nullptr, nullptr};
        void* d_x[2] = {nullptr, nullptr};
        cudaEvent_t ev_copy[2] = {nullptr, nullptr};
        cudaEvent_t ev_done[2] = {nullptr, nullptr};
        cudaEvent_t ev_order = nullptr, ev_t0 = nullptr, ev_t1 = nullptr;
        int* d_flags = nullptr;
        int* h_flags = nullptr;
        GramPlan plan;
        char* d_scratch = nullptr;   // loadings output / scoring model rows and partials (grow-only)
        int64_t cap_scratch = 0;
        bool ready = false, busy = false;
    };
    std::vector<Lane> lanes;
    int64_t chunk_variants = 0, chunk_nnz = 0;
    int64_t panel = 8192;   // cells per panel row of the internal dense staging tiles (VPCA_PANEL)

    cudaEvent_t ev_t0 = nullptr, ev_t1 = nullptr, ev_e0 = nullptr, ev_e1 = nullptr;
    bool gram_timed = false, eig_timed = false;

    int64_t total_variants = 0;      // committed + direct
    int64_t inflight_variants = 0;   // staged in slots, not yet committed
    vpca_stats st{};
    std::atomic<int64_t> c_launches{0}, c_gram{0}, c_h2d{0}, c_d2h{0};
    std::atomic<float> lane_gram_ms{0.f};
    std::mutex mu;
    std::condition_variable cv;
    std::mutex err_mu;
    std::string err;
};

namespace {

int fail(vpca_ctx* ctx, int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    tls_error = buf;
    tls_error_ctx = ctx;
    if (ctx) {
        std::lock_guard<std::mutex> lk(ctx->err_mu);
        ctx->err = buf;
    }
    return code;
}

#define CUDA_OK(ctx, call)                                                                                      \
    do {                                                                                                        \
        cudaError_t _e = (call);                                                                                \
        if (_e != cudaSuccess)                                                                                  \
            return fail(ctx, VPCA_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(_e), __FILE__,   \
                        __LINE__);                                                                              \
    } while (0)

// Entry points of the Gram on a scoring context (vpca_create_scoring), which has none.
#define REFUSE_ON_SCORING(ctx)                                                                                  \
    do {                                                                                                        \
        if ((ctx)->scoring)                                                                                     \
            return fail(ctx, VPCA_ERR_UNSUPPORTED, "%s: a scoring context has no Gram", __func__);              \
    } while (0)

template <typename T>
static cudaError_t grow_buffer(T** p, int64_t* cap, int64_t need) {
    if (need <= *cap && *p != nullptr) return cudaSuccess;
    cudaFree(*p);
    *p = nullptr;
    *cap = 0;
    const int64_t c = need + need / 4 + 1024;
    cudaError_t e = cudaMalloc(p, (size_t)c * sizeof(T));
    if (e == cudaSuccess) *cap = c;
    return e;
}

// every similarity count is at most (#variants) * max_mult^2 and must stay a Java Int (VariantsPca.scala:185).
// `extra` = variants about to be added on top of everything committed AND everything staged in uncommitted partitions.
int check_overflow(vpca_ctx* ctx, int64_t extra) {
    const long double worst =
        (long double)(ctx->total_variants + ctx->inflight_variants + extra) * ctx->max_mult * ctx->max_mult;
    if (worst > 2147483647.0L)
        return fail(ctx, VPCA_ERR_OVERFLOW, "%lld variants x multiplicity %d^2 could overflow an int32 similarity count",
                    (long long)(ctx->total_variants + ctx->inflight_variants + extra), ctx->max_mult);
    return VPCA_OK;
}

void free_lane(vpca_ctx::Lane& L) {
    if (L.stream) cudaStreamSynchronize(L.stream);
    if (L.copy_stream) cudaStreamSynchronize(L.copy_stream);
    for (int b = 0; b < 2; ++b) {
        cudaFree(L.d_off[b]);
        cudaFree(L.d_idx[b]);
        cudaFree(L.d_x[b]);
        if (L.ev_copy[b]) cudaEventDestroy(L.ev_copy[b]);
        if (L.ev_done[b]) cudaEventDestroy(L.ev_done[b]);
        L.d_off[b] = nullptr;
        L.d_idx[b] = nullptr;
        L.d_x[b] = nullptr;
        L.ev_copy[b] = L.ev_done[b] = nullptr;
    }
    for (cudaEvent_t* ev : {&L.ev_order, &L.ev_t0, &L.ev_t1})
        if (*ev) {
            cudaEventDestroy(*ev);
            *ev = nullptr;
        }
    cudaFree(L.d_flags);
    L.d_flags = nullptr;
    cudaFree(L.d_scratch);
    L.d_scratch = nullptr;
    L.cap_scratch = 0;
    if (L.h_flags) cudaFreeHost(L.h_flags);
    L.h_flags = nullptr;
    gram_plan_free(L.plan);
    if (L.copy_stream) cudaStreamDestroy(L.copy_stream);
    if (L.stream) cudaStreamDestroy(L.stream);
    L.copy_stream = L.stream = nullptr;
    L.ready = false;
}

void copy_peers(const GramPlan& from, GramPlan& to) {
    to.own_lo = from.own_lo;
    to.own_hi = from.own_hi;
    to.num_peers = from.num_peers;
    to.peer_rank = from.peer_rank;
    to.peer_mode = from.peer_mode;
    for (int d = 0; d < 16; ++d) {
        to.peer_S[d] = from.peer_S[d];
        to.peer_flags[d] = from.peer_flags[d];
        to.own_end[d] = from.own_end[d];
    }
}

void sync_peers_to_lanes(vpca_ctx* ctx) {
    for (auto& L : ctx->lanes) copy_peers(ctx->plan, L.plan);
}

void staging_geometry(vpca_ctx* ctx) {
    if (ctx->chunk_variants != 0) return;
    const int n = ctx->rows(), bits = ctx->elem_bits;
    int64_t cv = ctx->cfg.chunk_variants;
    if (cv <= 0) {
        cv = (256ll << 20) * 8 / ((int64_t)n * bits);
        cv = std::max<int64_t>(1024, std::min<int64_t>(cv, 1 << 20));
    }
    if (const char* pe = getenv("VPCA_PANEL")) {
        const int64_t pv = atoll(pe);
        if (pv >= 128 && pv % 128 == 0) ctx->panel = pv;
    }
    cv = std::max<int64_t>(ctx->panel, (cv / ctx->panel) * ctx->panel);   // whole panels
    int64_t cz = ctx->cfg.chunk_nnz;
    if (cz <= 0) cz = 64ll << 20;
    cz = std::max<int64_t>(cz, 1024);
    ctx->chunk_variants = cv;
    ctx->chunk_nnz = cz;
}

// Allocates the lane's streams and staging buffers on first use; on any failure everything is released again, so a
// later call retries from scratch instead of running on half a lane.
int ensure_lane(vpca_ctx* ctx, vpca_ctx::Lane& L) {
    if (L.ready) return VPCA_OK;
    const int n = ctx->rows(), bits = ctx->elem_bits;
    const int64_t cv = ctx->chunk_variants, cz = ctx->chunk_nnz;
    cudaError_t e = cudaStreamCreateWithFlags(&L.stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&L.copy_stream, cudaStreamNonBlocking);
    for (int b = 0; b < 2 && e == cudaSuccess; ++b) {
        e = cudaMalloc(&L.d_off[b], (size_t)(cv + 1) * sizeof(int64_t));
        if (e == cudaSuccess) e = cudaMalloc(&L.d_idx[b], (size_t)cz * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&L.d_x[b], (size_t)n * (size_t)cv * bits / 8);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&L.ev_copy[b], cudaEventDisableTiming);
        if (e == cudaSuccess) e = cudaEventCreateWithFlags(&L.ev_done[b], cudaEventDisableTiming);
    }
    if (e == cudaSuccess) e = cudaEventCreateWithFlags(&L.ev_order, cudaEventDisableTiming);
    if (e == cudaSuccess) e = cudaEventCreate(&L.ev_t0);
    if (e == cudaSuccess) e = cudaEventCreate(&L.ev_t1);
    if (e == cudaSuccess) e = cudaMalloc(&L.d_flags, sizeof(int));
    if (e == cudaSuccess) e = cudaHostAlloc(&L.h_flags, sizeof(int), cudaHostAllocPortable);
    if (e != cudaSuccess) {
        free_lane(L);
        return fail(ctx, e == cudaErrorMemoryAllocation ? VPCA_ERR_NOMEM : VPCA_ERR_CUDA, "staging lane: %s",
                    cudaGetErrorString(e));
    }
    copy_peers(ctx->plan, L.plan);
    L.ready = true;
    return VPCA_OK;
}

// A free lane, blocking while all are taken.  Also orders the lane's stream after everything enqueued on the context's
// stream so far (a preceding vpca_reset / vpca_load_partial_gram).
struct LaneGuard {
    vpca_ctx* ctx;
    vpca_ctx::Lane* lane = nullptr;
    int rc = VPCA_OK;
    explicit LaneGuard(vpca_ctx* c) : ctx(c) {
        std::unique_lock<std::mutex> lk(ctx->mu);
        staging_geometry(ctx);
        ctx->cv.wait(lk, [&] {
            for (auto& L : ctx->lanes)
                if (!L.busy) return true;
            return false;
        });
        for (auto& L : ctx->lanes)
            if (!L.busy) {
                lane = &L;
                break;
            }
        lane->busy = true;
        rc = ensure_lane(ctx, *lane);
        if (rc == VPCA_OK) {
            cudaError_t e = cudaEventRecord(lane->ev_order, ctx->stream);
            if (e == cudaSuccess) e = cudaStreamWaitEvent(lane->stream, lane->ev_order, 0);
            if (e != cudaSuccess) rc = fail(ctx, VPCA_ERR_CUDA, "lane ordering: %s", cudaGetErrorString(e));
        }
    }
    ~LaneGuard() {
        {
            std::lock_guard<std::mutex> lk(ctx->mu);
            lane->busy = false;
        }
        ctx->cv.notify_one();
    }
};

int launch_gram(vpca_ctx* ctx, GramPlan& plan, cudaStream_t stream, cudaEvent_t t0, cudaEvent_t t1, const void* d_x,
                int64_t nv, int64_t ld, int64_t panel, int32_t* d_target) {
    // fp32 TMEM accumulation (bf16 / e2m1) is exact only below 2^24: bound the variants one launch may fold.
    // vpca_create guarantees that the bound is at least one panel.
    int64_t limit = nv;
    if (ctx->elem_bits != 8) {
        limit = (int64_t)(16777216ll / ((int64_t)ctx->max_mult * ctx->max_mult));
        const int64_t q = panel > 0 ? panel : 128;
        limit = (limit / q) * q;
        if (limit <= 0)
            return fail(ctx, VPCA_ERR_UNSUPPORTED, "max_multiplicity %d leaves no exact fp32 accumulation window for panels of "
                        "%lld variants", ctx->max_mult, (long long)q);
    }
    for (int64_t v0 = 0; v0 < nv; v0 += limit) {
        const int64_t cnt = std::min<int64_t>(limit, nv - v0);
        std::string msg;
        cudaEventRecord(t0, stream);
        // sub-launches start on a panel boundary (panel layout) or at column v0 (row-major)
        const size_t byte_off = panel > 0 ? (size_t)(v0 / panel) * (size_t)ctx->rows() * (size_t)panel * ctx->elem_bits / 8
                                          : (size_t)v0 * ctx->elem_bits / 8;
        cudaError_t e = gram_accumulate(plan, static_cast<const char*>(d_x) + byte_off, ctx->elem_bits, ctx->n, ctx->rows(),
                                        cnt, ld, panel, d_target, stream, &msg);
        cudaEventRecord(t1, stream);
        if (e != cudaSuccess)
            return fail(ctx, VPCA_ERR_CUDA, "Gram launch failed: %s %s", cudaGetErrorString(e), msg.c_str());
        ctx->c_gram += 1;
        ctx->c_launches += 1;
    }
    return VPCA_OK;
}

// Caller holds ctx->mu.
vpca_ctx::Slot* find_slot(vpca_ctx* ctx, int64_t pid, bool create, int* rc) {
    *rc = VPCA_OK;
    for (auto& s : ctx->slots)
        if (s.used && s.pid == pid) return &s;
    if (!create) return nullptr;
    for (auto& s : ctx->slots)
        if (!s.used) {
            if (s.d_S == nullptr) {
                cudaError_t e = cudaMalloc(&s.d_S, ctx->slot_bytes());
                if (e == cudaSuccess) e = cudaEventCreateWithFlags(&s.ev_free, cudaEventDisableTiming);
                if (e != cudaSuccess) {
                    cudaFree(s.d_S);
                    s.d_S = nullptr;
                    *rc = fail(ctx, VPCA_ERR_NOMEM, "cudaMalloc of a partition Gram failed: %s", cudaGetErrorString(e));
                    return nullptr;
                }
            }
            s.used = true;
            s.fresh = true;
            s.busy = false;
            s.pid = pid;
            s.nv = 0;
            s.matched = 0;
            return &s;
        }
    *rc = fail(ctx, VPCA_ERR_STATE, "more than %d partitions in flight; commit or abort one first",
               (int)ctx->slots.size());
    return nullptr;
}

// Bookkeeping that brackets every host-input accumulate call.  begin(): state + overflow checks, slot lookup.
// end(): counters, slot release; a failed batch poisons its partition (the staging Gram may be partially updated).
struct CallScope {
    vpca_ctx* ctx;
    int64_t pid, nv;
    int64_t matched = 0;   // scoring: variants of the call with a model row
    vpca_ctx::Slot* slot = nullptr;
    int32_t* target = nullptr;   // Gram / staging Gram; on a scoring context the (T, r) accumulator
    bool fresh = false;
    int begin() {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
        int rc = ctx->scoring ? VPCA_OK : check_overflow(ctx, nv);   // scores accumulate in FP64 and int64
        if (rc != VPCA_OK) return rc;
        target = ctx->scoring ? reinterpret_cast<int32_t*>(ctx->d_direct) : ctx->d_S;
        if (pid >= 0) {
            slot = find_slot(ctx, pid, true, &rc);
            if (slot == nullptr) return rc;
            if (slot->busy) {
                slot = nullptr;
                return fail(ctx, VPCA_ERR_STATE, "partition %lld is being written by another thread (spark.speculation "
                            "must stay off)", (long long)pid);
            }
            slot->busy = true;
            fresh = slot->fresh;
            slot->fresh = false;
            target = slot->d_S;
            ctx->inflight_variants += nv;   // reserved now, so that concurrent tasks cannot jointly pass the bound
        } else if (ctx->band_rows != ctx->n) {
            return fail(ctx, VPCA_ERR_STATE, "a band-only Gram takes device-resident input (vpca_accumulate_panels / "
                        "vpca_accumulate_dense with on_device = 1)");
        }
        return VPCA_OK;
    }
    int end(int rc) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (slot != nullptr) {
            slot->busy = false;
            if (rc == VPCA_OK) {
                slot->nv += nv;
                slot->matched += matched;
            } else {
                ctx->inflight_variants -= nv + slot->nv;
                ctx->st.variants_accumulated -= slot->nv;
                slot->used = false;
            }
        } else if (rc == VPCA_OK) {
            ctx->total_variants += nv;
            ctx->direct_matched += matched;
        } else if (rc == VPCA_ERR_INDEX_OUT_OF_RANGE || rc == VPCA_ERR_OVERFLOW) {
            std::lock_guard<std::mutex> lk2(ctx->err_mu);
            ctx->err += " [direct accumulation: the Gram may hold a partial batch, call vpca_reset]";
            tls_error = ctx->err;
        }
        if (rc == VPCA_OK) ctx->st.variants_accumulated += nv;
        return rc;
    }
};

// First batch of a partition: zero its staging Gram on the lane's stream, after the commit that last read it.
int prepare_slot(vpca_ctx* ctx, vpca_ctx::Lane& L, CallScope& sc) {
    if (sc.slot == nullptr || !sc.fresh) return VPCA_OK;
    CUDA_OK(ctx, cudaStreamWaitEvent(L.stream, sc.slot->ev_free, 0));
    CUDA_OK(ctx, cudaMemsetAsync(sc.slot->d_S, 0, ctx->slot_bytes(), L.stream));
    return VPCA_OK;
}

void lane_gram_time(vpca_ctx* ctx, vpca_ctx::Lane& L) {
    float ms = 0.f;
    if (cudaEventElapsedTime(&ms, L.ev_t0, L.ev_t1) == cudaSuccess) {
        ctx->lane_gram_ms.store(ms);
        std::lock_guard<std::mutex> lk(ctx->mu);
        ctx->gram_timed = false;
        ctx->st.gram_cta_group = L.plan.cta_group;
        ctx->st.gram_resident = L.plan.last_resident;
    }
}

// What a chunk loop (process_calls, packed_chunks, the panels routes) does with each encoded chunk: the Gram launch,
// the loadings of a saved model, or the scoring of a study against one (model.cu).
struct ChunkSink {
    enum Kind { GRAM, LOADINGS, SCORE } kind = GRAM;
    int32_t* gram = nullptr;               // GRAM: the Gram or staging Gram the launch adds into
    int k = 0;                             // LOADINGS / SCORE: columns
    double* d_L = nullptr;                 // LOADINGS: device output of one chunk (nvc x k) ...
    int32_t* d_cnt = nullptr;              // ... and its carriers
    double* h_L = nullptr;                 // LOADINGS: host output of the call (nv x k) ...
    int32_t* h_cnt = nullptr;              // ... and its carriers
    const int32_t* d_mrows = nullptr;      // SCORE: model row of every variant of the call (device)
    double* d_part = nullptr;              // SCORE: scratch of model_score
    double* d_acc = nullptr;               // SCORE: the accumulator the chunk adds into
    bool launched = false;                 // set once a Gram launch ran (lane timing)
};

// Consume variants [v, v + nvc) of the call, encoded in panel layout at d_x, on `stream`.
int consume_chunk(vpca_ctx* ctx, GramPlan& plan, cudaStream_t stream, cudaEvent_t t0, cudaEvent_t t1, ChunkSink& sink,
                  const void* d_x, int64_t v, int64_t nvc, int64_t panel) {
    switch (sink.kind) {
    case ChunkSink::GRAM: {
        const int rc = launch_gram(ctx, plan, stream, t0, t1, d_x, nvc, panel, panel, sink.gram);
        if (rc == VPCA_OK) sink.launched = true;
        return rc;
    }
    case ChunkSink::LOADINGS:
        CUDA_OK(ctx, model_loadings(d_x, ctx->elem_bits, nvc, panel, ctx->rows(), ctx->n, ctx->eig.d_evecs, sink.k, sink.d_L,
                                    sink.d_cnt, stream));
        CUDA_OK(ctx, cudaMemcpyAsync(sink.h_L + (size_t)v * sink.k, sink.d_L, (size_t)nvc * sink.k * sizeof(double),
                                     cudaMemcpyDeviceToHost, stream));
        CUDA_OK(ctx, cudaMemcpyAsync(sink.h_cnt + v, sink.d_cnt, (size_t)nvc * sizeof(int32_t), cudaMemcpyDeviceToHost, stream));
        ctx->c_launches += (sink.k + 7) / 8;
        ctx->c_d2h += nvc * (sink.k * 8 + 4);
        return VPCA_OK;
    case ChunkSink::SCORE:
        CUDA_OK(ctx, model_score(d_x, ctx->elem_bits, nvc, panel, ctx->rows(), sink.d_mrows + v, ctx->d_model_L, ctx->d_model_n,
                                 sink.k, sink.d_part, sink.d_acc, stream));
        ctx->c_launches += (sink.k + 7) / 8 + 1;
        return VPCA_OK;
    }
    return fail(ctx, VPCA_ERR_BAD_ARG, "internal: unknown chunk consumer");
}

// CSR rows -> encode -> sink, on lane L.  out_tile != nullptr: copy the encoded tile back instead.
int process_calls(vpca_ctx* ctx, vpca_ctx::Lane& L, const int64_t* offsets, const void* sample_idx, int idx_bytes,
                  int64_t nv, ChunkSink* sink, void* out_tile, int64_t out_ld) {
    const int bits = ctx->elem_bits;
    // validate the whole offsets array before anything is sized from it
    if (offsets[0] < 0) return fail(ctx, VPCA_ERR_BAD_ARG, "offsets[0] must be >= 0");
    for (int64_t q = 0; q < nv; ++q)
        if (offsets[q + 1] < offsets[q]) return fail(ctx, VPCA_ERR_BAD_ARG, "offsets must be non-decreasing (row %lld)", (long long)q);
    *L.h_flags = 0;
    CUDA_OK(ctx, cudaMemsetAsync(L.d_flags, 0, sizeof(int), L.stream));
    int64_t v = 0;
    int chunk = 0;
    while (v < nv) {
        // largest run of rows that fits both the variant and the index budget
        int64_t vend = std::min(nv, v + ctx->chunk_variants);
        if (offsets[vend] - offsets[v] > ctx->chunk_nnz) {
            const int64_t* hi = std::upper_bound(offsets + v, offsets + vend + 1, offsets[v] + ctx->chunk_nnz);
            vend = (hi - offsets) - 1;
            if (bits == 4 && vend - v >= 128) vend = v + ((vend - v) / 128) * 128;   // keep packed rows byte aligned
            if (vend <= v)
                return fail(ctx, VPCA_ERR_BAD_ARG, "row %lld has %lld entries, more than chunk_nnz=%lld", (long long)v,
                            (long long)(offsets[v + 1] - offsets[v]), (long long)ctx->chunk_nnz);
        }
        const int64_t nvc = vend - v, nnz = offsets[vend] - offsets[v];
        if (nnz > ctx->chunk_nnz || nvc > ctx->chunk_variants)
            return fail(ctx, VPCA_ERR_BAD_ARG, "internal: chunk of %lld rows / %lld entries exceeds the staging buffers",
                        (long long)nvc, (long long)nnz);
        const int b = chunk & 1;
        // the copy stream may overwrite buffer b only after the kernels that read it have run
        CUDA_OK(ctx, cudaStreamWaitEvent(L.copy_stream, L.ev_done[b], 0));
        CUDA_OK(ctx, cudaMemcpyAsync(L.d_off[b], offsets + v, (size_t)(nvc + 1) * sizeof(int64_t), cudaMemcpyHostToDevice,
                                     L.copy_stream));
        if (nnz > 0)
            CUDA_OK(ctx, cudaMemcpyAsync(L.d_idx[b], static_cast<const char*>(sample_idx) + (size_t)offsets[v] * idx_bytes,
                                         (size_t)nnz * idx_bytes, cudaMemcpyHostToDevice, L.copy_stream));
        CUDA_OK(ctx, cudaEventRecord(L.ev_copy[b], L.copy_stream));
        ctx->c_h2d += (nvc + 1) * 8 + nnz * idx_bytes;
        CUDA_OK(ctx, cudaStreamWaitEvent(L.stream, L.ev_copy[b], 0));
        const int64_t P = ctx->panel;
        CUDA_OK(ctx, encode_calls(L.d_off[b], offsets[v], L.d_idx[b], idx_bytes, nvc, ctx->rows(), bits, ctx->max_mult, L.d_x[b],
                                  P, P, ctx->d_rows, L.d_flags, L.stream));
        ctx->c_launches += 2;
        if (out_tile != nullptr) {
            // panel layout -> the caller's row-major tile, one 2-D copy per panel (chunk boundaries are multiples of
            // 128 variants, so 4-bit rows split on byte boundaries)
            for (int64_t pv = 0; pv < nvc; pv += P) {
                const int64_t wv = std::min(P, nvc - pv);
                CUDA_OK(ctx, cudaMemcpy2DAsync(static_cast<char*>(out_tile) + (size_t)(v + pv) * bits / 8,
                                               (size_t)out_ld * bits / 8,
                                               static_cast<const char*>(L.d_x[b]) + (size_t)(pv / P) * ctx->rows() * P * bits / 8,
                                               (size_t)P * bits / 8, (size_t)(wv * bits + 7) / 8, (size_t)ctx->rows(),
                                               cudaMemcpyDeviceToHost, L.stream));
            }
            ctx->c_d2h += (nvc * bits + 7) / 8 * (int64_t)ctx->rows();
        } else {
            int rc = consume_chunk(ctx, L.plan, L.stream, L.ev_t0, L.ev_t1, *sink, L.d_x[b], v, nvc, P);
            if (rc != VPCA_OK) return rc;
        }
        CUDA_OK(ctx, cudaEventRecord(L.ev_done[b], L.stream));
        v = vend;
        ++chunk;
    }
    CUDA_OK(ctx, cudaMemcpyAsync(L.h_flags, L.d_flags, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
    // the caller's buffers are read asynchronously: do not return before every copy has completed
    CUDA_OK(ctx, cudaStreamSynchronize(L.stream));
    if (sink != nullptr && sink->launched) lane_gram_time(ctx, L);
    if (*L.h_flags & 1)
        return fail(ctx, VPCA_ERR_INDEX_OUT_OF_RANGE, "sample index outside [0, %d) (the reference throws at "
                    "VariantsPca.scala:59/:188)", ctx->rows());
    if (*L.h_flags & 2)
        return fail(ctx, VPCA_ERR_OVERFLOW, "a sample is listed more than max_multiplicity=%d times in one row",
                    ctx->max_mult);
    return VPCA_OK;
}


}  // namespace

extern "C" {

int vpca_version(void) { return VPCA_VERSION_MAJOR * 1000 + VPCA_VERSION_MINOR; }

const char* vpca_last_error(const vpca_ctx* ctx) {
    // a thread that just failed on `ctx` reads its own message, whatever other threads have done to the context since
    if (ctx == nullptr || tls_error_ctx == ctx) return tls_error.c_str();
    vpca_ctx* c = const_cast<vpca_ctx*>(ctx);
    std::lock_guard<std::mutex> lk(c->err_mu);
    tls_error_copy = c->err;
    return tls_error_copy.c_str();
}

static int create_impl(const vpca_config* cfg, int n_proj, const int32_t* sample_rows, const vpca_model* model,
                       vpca_ctx** out) {
    if (out == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "out is NULL");
    *out = nullptr;
    if (cfg == nullptr || cfg->struct_size != sizeof(vpca_config))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "cfg is NULL or struct_size != sizeof(vpca_config) (%zu)",
                    sizeof(vpca_config));
    if (cfg->n_samples < 2) return fail(nullptr, VPCA_ERR_BAD_ARG, "n_samples must be >= 2");
    if (cfg->dtype != VPCA_DTYPE_I8 && cfg->dtype != VPCA_DTYPE_BF16 && cfg->dtype != VPCA_DTYPE_E2M1)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "unknown dtype %d", cfg->dtype);
    if (cfg->staging_lanes < 0 || cfg->staging_lanes > 16)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "staging_lanes must be in [0, 16]");
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(nullptr, VPCA_ERR_CUDA, "no CUDA device: %s (libvpca has no CPU fallback)", cudaGetErrorString(e));
    if (cfg->device < 0 || cfg->device >= ndev) return fail(nullptr, VPCA_ERR_BAD_ARG, "device %d of %d", cfg->device, ndev);
    CUDA_OK(nullptr, cudaSetDevice(cfg->device));
    cudaDeviceProp prop;
    CUDA_OK(nullptr, cudaGetDeviceProperties(&prop, cfg->device));
    if (prop.major != 10)
        return fail(nullptr, VPCA_ERR_UNSUPPORTED, "device %d is sm_%d%d; libvpca is built for sm_100a (B200) only",
                    cfg->device, prop.major, prop.minor);
    vpca_ctx* ctx = new (std::nothrow) vpca_ctx();
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_NOMEM, "out of host memory");
    ctx->cfg = *cfg;
    ctx->n = cfg->n_samples;
    ctx->n_proj = n_proj;
    ctx->elem_bits = cfg->dtype == VPCA_DTYPE_I8 ? 8 : (cfg->dtype == VPCA_DTYPE_BF16 ? 16 : 4);
    ctx->max_mult = cfg->max_multiplicity > 0 ? cfg->max_multiplicity : 2;
    ctx->num_pc = cfg->num_pc > 0 ? cfg->num_pc : 2;
    if (ctx->elem_bits == 4 && ctx->max_mult > 2) {
        delete ctx;
        return fail(nullptr, VPCA_ERR_BAD_ARG, "VPCA_DTYPE_E2M1 represents multiplicities 0, 1, 2 only (max_multiplicity <= 2)");
    }
    if (ctx->elem_bits != 8 && 16777216ll / ((int64_t)ctx->max_mult * ctx->max_mult) < 8192) {
        // fp32 tensor accumulation is exact below 2^24 only: a launch folds at least one panel (8192 variants), so the
        // largest count of one panel, 8192 * max_mult^2, must stay below that (bf16: max_multiplicity <= 45)
        const int mm = ctx->max_mult;
        delete ctx;
        return fail(nullptr, VPCA_ERR_BAD_ARG, "max_multiplicity %d is too large for exact fp32 accumulation of bf16 cells "
                    "(<= 45); use VPCA_DTYPE_I8", mm);
    }
    const bool band = cfg->gram_band_rows > 0;
    if (band && (cfg->d_gram != nullptr || cfg->gram_band_row0 < 0 || cfg->gram_band_row0 + cfg->gram_band_rows > ctx->n)) {
        delete ctx;
        return fail(nullptr, VPCA_ERR_BAD_ARG, "gram_band_row0/rows must lie in [0, n_samples] and need a library-owned Gram");
    }
    ctx->band_row0 = band ? cfg->gram_band_row0 : 0;
    ctx->band_rows = band ? cfg->gram_band_rows : ctx->n;
    if (band) {   // without peers the Gram kernel computes exactly these rows (owner-computes), with peers it flushes to owners
        ctx->plan.own_lo = ctx->band_row0;
        ctx->plan.own_hi = ctx->band_row0 + ctx->band_rows;
    }
    if (cfg->stream != nullptr) {
        ctx->stream = static_cast<cudaStream_t>(cfg->stream);
    } else {
        e = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        ctx->own_stream = true;
    }
    const size_t gram_cells = model != nullptr ? 0 : ctx->gram_cells();
    if (model != nullptr) {
        // scoring context: the model goes to the device, and one accumulator for direct input; no Gram
        ctx->scoring = true;
        ctx->model_k = model->k;
        ctx->model_nfit = model->n_fitted;
        ctx->model_nv = model->n_variants;
        const size_t V = (size_t)std::max<int64_t>(1, model->n_variants), k = (size_t)model->k;
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_model_L, V * k * sizeof(double));
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_model_n, V * sizeof(int32_t));
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_model_terms, (3 * k + 1) * sizeof(double));
        if (e == cudaSuccess) e = cudaMalloc(&ctx->d_direct, ctx->slot_bytes());
        if (e == cudaSuccess && model->n_variants > 0) {
            e = cudaMemcpy(ctx->d_model_L, model->loadings, (size_t)model->n_variants * k * sizeof(double), cudaMemcpyHostToDevice);
            if (e == cudaSuccess)
                e = cudaMemcpy(ctx->d_model_n, model->carriers, (size_t)model->n_variants * sizeof(int32_t), cudaMemcpyHostToDevice);
        }
        if (e == cudaSuccess) {
            std::vector<double> terms(3 * k + 1);
            for (size_t c = 0; c < k; ++c) {
                terms[c] = model->eigenvalues[c];
                terms[k + c] = model->col_sums[c];
                terms[2 * k + c] = model->rowsum_dots[c];
            }
            terms[3 * k] = model->matrix_mean;
            e = cudaMemcpy(ctx->d_model_terms, terms.data(), terms.size() * sizeof(double), cudaMemcpyHostToDevice);
        }
        if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_direct, 0, ctx->slot_bytes(), ctx->stream);
    } else if (e == cudaSuccess) {
        if (cfg->d_gram != nullptr) {
            ctx->d_S = static_cast<int32_t*>(cfg->d_gram);
        } else {
            e = cudaMalloc(&ctx->d_S, (gram_cells + 64) * sizeof(int32_t));   // + barrier flags of the peer-reduce mode
            ctx->own_S = true;
            if (e == cudaSuccess) e = cudaMemsetAsync(ctx->d_S + gram_cells, 0, 64 * sizeof(int32_t), ctx->stream);
        }
    }
    if (e == cudaSuccess && model == nullptr) e = cudaMemsetAsync(ctx->d_S, 0, gram_cells * sizeof(int32_t), ctx->stream);
    if (e == cudaSuccess && sample_rows != nullptr) {
        e = cudaMalloc(&ctx->d_rows, (size_t)ctx->rows() * sizeof(int32_t));
        if (e == cudaSuccess)
            e = cudaMemcpy(ctx->d_rows, sample_rows, (size_t)ctx->rows() * sizeof(int32_t), cudaMemcpyHostToDevice);
    }
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_t0);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_t1);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_e0);
    if (e == cudaSuccess) e = cudaEventCreate(&ctx->ev_e1);
    if (e != cudaSuccess) {
        const int rc = fail(nullptr, e == cudaErrorMemoryAllocation ? VPCA_ERR_NOMEM : VPCA_ERR_CUDA, "vpca_create: %s",
                            cudaGetErrorString(e));
        vpca_destroy(ctx);
        return rc;
    }
    const int nslots = cfg->partitions_in_flight > 0 ? cfg->partitions_in_flight : 4;
    ctx->slots.resize(nslots);
    ctx->lanes.resize(cfg->staging_lanes > 0 ? cfg->staging_lanes : 2);
    *out = ctx;
    return VPCA_OK;
}

int vpca_create(const vpca_config* cfg, vpca_ctx** out) { return create_impl(cfg, 0, nullptr, nullptr, out); }

int vpca_create_projecting(const vpca_config* cfg, const vpca_projection* proj, vpca_ctx** out) {
    if (out != nullptr) *out = nullptr;
    if (proj == nullptr || proj->struct_size != sizeof(vpca_projection))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "proj is NULL or struct_size != sizeof(vpca_projection) (%zu)",
                    sizeof(vpca_projection));
    if (cfg == nullptr || cfg->struct_size != sizeof(vpca_config))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "cfg is NULL or struct_size != sizeof(vpca_config) (%zu)", sizeof(vpca_config));
    const int m = proj->n_projected;
    if (m < 0 || (int64_t)cfg->n_samples + m > 0x7fffffff)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "n_projected must be >= 0 and n_samples + n_projected < 2^31");
    const int total = cfg->n_samples + m;
    bool identity = true;
    if (proj->sample_rows != nullptr && cfg->n_samples >= 0) {
        std::vector<char> seen((size_t)total, 0);
        for (int s = 0; s < total; ++s) {
            const int32_t r = proj->sample_rows[s];
            if (r < 0 || r >= total || seen[(size_t)r])
                return fail(nullptr, VPCA_ERR_BAD_ARG, "sample_rows is not a permutation of [0, %d): entry %d is %d", total, s, r);
            seen[(size_t)r] = 1;
            identity = identity && r == s;
        }
    }
    if (m > 0) {
        // Out of scope for projection: fused peer reductions (refused by vpca_gram_set_peers*), row bands and the exact
        // block cover (the cross block needs the rectangle tiling)
        if (cfg->gram_band_rows > 0)
            return fail(nullptr, VPCA_ERR_UNSUPPORTED, "a projecting context stores the whole fitted Gram (no gram_band_rows)");
        const char* ex = getenv("VPCA_EXACT_COVER");
        if (ex != nullptr && atoi(ex) != 0)
            return fail(nullptr, VPCA_ERR_UNSUPPORTED, "VPCA_EXACT_COVER=1 has no tiling of the cross block");
    }
    return create_impl(cfg, m, identity ? nullptr : proj->sample_rows, nullptr, out);
}

int vpca_destroy(vpca_ctx* ctx) {
    if (ctx == nullptr) return VPCA_OK;
    cudaSetDevice(ctx->cfg.device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (auto& L : ctx->lanes) free_lane(L);
    for (auto& s : ctx->slots) {
        cudaFree(s.d_S);
        if (s.ev_free) cudaEventDestroy(s.ev_free);
    }
    if (ctx->plan.peers_ipc)
        for (int d = 0; d < ctx->plan.num_peers; ++d)
            if (d != ctx->plan.peer_rank && ctx->plan.peer_S[d] != nullptr) cudaIpcCloseMemHandle(ctx->plan.peer_base[d]);
    if (ctx->own_S) cudaFree(ctx->d_S);
    cudaFree(ctx->d_rows);
    cudaFree(ctx->d_proj);
    cudaFree(ctx->d_model_L);
    cudaFree(ctx->d_model_n);
    cudaFree(ctx->d_model_terms);
    cudaFree(ctx->d_direct);
    cudaFree(ctx->d_scratch);
    for (auto& kv : ctx->scored) cudaFree(kv.second.d_acc);
    if (ctx->eig_ready) eig_free(ctx->eig);
    join_free(ctx->join);
    gram_plan_free(ctx->plan);
    for (cudaEvent_t ev : {ctx->ev_t0, ctx->ev_t1, ctx->ev_e0, ctx->ev_e1})
        if (ev) cudaEventDestroy(ev);
    if (ctx->own_stream && ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return VPCA_OK;
}

int vpca_synchronize(vpca_ctx* ctx) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return VPCA_OK;
}

int vpca_reset(vpca_ctx* ctx) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> jl(ctx->join_mu);   // lock order everywhere: join_mu, then mu
    std::lock_guard<std::mutex> lk(ctx->mu);
    for (auto& L : ctx->lanes)
        if (L.busy) return fail(ctx, VPCA_ERR_STATE, "vpca_reset while an accumulate call is in flight");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (ctx->scoring) {
        CUDA_OK(ctx, cudaMemsetAsync(ctx->d_direct, 0, ctx->slot_bytes(), ctx->stream));
        CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));   // no commit still reads a partial that is freed below
        for (auto& kv : ctx->scored) cudaFree(kv.second.d_acc);
        ctx->scored.clear();
        ctx->direct_matched = 0;
    } else {
        CUDA_OK(ctx, cudaMemsetAsync(ctx->d_S, 0, ctx->gram_cells() * sizeof(int32_t), ctx->stream));
    }
    for (auto& s : ctx->slots) s.used = false;
    ctx->finalized = false;
    ctx->pca_done = false;
    ctx->proj_k = 0;
    ctx->total_variants = 0;
    ctx->inflight_variants = 0;
    ctx->st.variants_accumulated = 0;
    ctx->join.out_rows = -1;   // joined rows of an earlier analysis do not outlive a reset (join_mu is held, see above)
    return VPCA_OK;
}

int vpca_encode_calls(vpca_ctx* ctx, const int64_t* offsets, const int32_t* sample_idx, int64_t nv, void* out,
                      int64_t ld) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    if (offsets == nullptr || out == nullptr || nv < 0 || ld < nv || (nv > 0 && sample_idx == nullptr && offsets[nv] > offsets[0]))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_encode_calls: bad argument");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    LaneGuard lg(ctx);
    if (lg.rc != VPCA_OK) return lg.rc;
    return process_calls(ctx, *lg.lane, offsets, sample_idx, 4, nv, nullptr, out, ld);
}

static int accumulate_calls_impl(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const void* sample_idx,
                                 int idx_bytes, int64_t nv) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    if (offsets == nullptr || nv < 0 || (nv > 0 && sample_idx == nullptr && offsets[nv] > offsets[0]))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_accumulate_calls: bad argument");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
        return VPCA_OK;
    }
    CallScope sc{ctx, partition_id, nv};
    int rc = sc.begin();
    if (rc != VPCA_OK) return rc;
    {
        LaneGuard lg(ctx);
        rc = lg.rc;
        if (rc == VPCA_OK) rc = prepare_slot(ctx, *lg.lane, sc);
        ChunkSink sink;
        sink.gram = sc.target;
        if (rc == VPCA_OK) rc = process_calls(ctx, *lg.lane, offsets, sample_idx, idx_bytes, nv, &sink, nullptr, 0);
    }
    return sc.end(rc);
}

int vpca_accumulate_calls(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const int32_t* sample_idx,
                          int64_t nv) {
    return accumulate_calls_impl(ctx, partition_id, offsets, sample_idx, 4, nv);
}

int vpca_accumulate_calls_u16(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const uint16_t* sample_idx,
                              int64_t nv) {
    if (ctx != nullptr && ctx->rows() > 65536)
        return fail(ctx, VPCA_ERR_BAD_ARG, "16-bit sample indices need n_samples (+ n_projected) <= 65536");
    return accumulate_calls_impl(ctx, partition_id, offsets, sample_idx, 2, nv);
}

// Packed rows -> encode -> sink, on lane L.  code 0: bitmap rows; 1 / 2: PLINK .bed rows counting A1 / A2 (encode.cu).
static int packed_chunks(vpca_ctx* ctx, vpca_ctx::Lane& L, const uint8_t* bits, int64_t nv, int64_t stride_bytes, int code,
                         ChunkSink& sink) {
    // bits beyond sample n-1 in the last byte of a row would be read as carriers of non-existent samples: the kernel
    // masks them (smp >= n), nothing to validate on the host.
    const int64_t P = ctx->panel;
    const int64_t cap_rows = std::min<int64_t>(ctx->chunk_variants, (ctx->chunk_nnz * (int64_t)sizeof(int32_t)) / stride_bytes);
    if (cap_rows < 32) return fail(ctx, VPCA_ERR_BAD_ARG, "stride_bytes too large for the staging buffer");
    const int64_t whole = std::max<int64_t>(P, (cap_rows / P) * P);
    const int64_t step = whole <= cap_rows ? whole : (cap_rows / 32) * 32;
    int chunk = 0;
    for (int64_t v = 0; v < nv; v += step, ++chunk) {
        const int64_t nvc = std::min(step, nv - v);
        const int b = chunk & 1;
        CUDA_OK(ctx, cudaStreamWaitEvent(L.copy_stream, L.ev_done[b], 0));
        CUDA_OK(ctx, cudaMemcpyAsync(L.d_idx[b], bits + (size_t)v * stride_bytes, (size_t)nvc * stride_bytes,
                                     cudaMemcpyHostToDevice, L.copy_stream));
        CUDA_OK(ctx, cudaEventRecord(L.ev_copy[b], L.copy_stream));
        ctx->c_h2d += nvc * stride_bytes;
        CUDA_OK(ctx, cudaStreamWaitEvent(L.stream, L.ev_copy[b], 0));
        CUDA_OK(ctx, encode_bits(reinterpret_cast<const uint8_t*>(L.d_idx[b]), stride_bytes, nvc, ctx->rows(), ctx->elem_bits,
                                 L.d_x[b], P, P, code, ctx->d_rows, L.stream));
        ctx->c_launches += 1;
        const int r = consume_chunk(ctx, L.plan, L.stream, L.ev_t0, L.ev_t1, sink, L.d_x[b], v, nvc, P);
        if (r != VPCA_OK) return r;
        CUDA_OK(ctx, cudaEventRecord(L.ev_done[b], L.stream));
    }
    CUDA_OK(ctx, cudaStreamSynchronize(L.stream));   // the caller's buffer is free to reuse on return
    return VPCA_OK;
}

static int packed_args(vpca_ctx* ctx, const uint8_t* bits, int64_t nv, int64_t stride_bytes, int code) {
    const int64_t min_stride = code == 0 ? (ctx->rows() + 7) / 8 : (ctx->rows() + 3) / 4;
    if (nv < 0 || (nv > 0 && bits == nullptr) || stride_bytes < min_stride)
        return fail(ctx, VPCA_ERR_BAD_ARG, "packed rows: stride_bytes must be >= ceil(n_samples / %d)", code == 0 ? 8 : 4);
    return VPCA_OK;
}

static int accumulate_packed(vpca_ctx* ctx, int64_t partition_id, const uint8_t* bits, int64_t nv, int64_t stride_bytes,
                             int code) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    int rc = packed_args(ctx, bits, nv, stride_bytes, code);
    if (rc != VPCA_OK) return rc;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
        return VPCA_OK;
    }
    CallScope sc{ctx, partition_id, nv};
    rc = sc.begin();
    if (rc != VPCA_OK) return rc;
    {
        LaneGuard lg(ctx);
        rc = lg.rc;
        if (rc == VPCA_OK) rc = prepare_slot(ctx, *lg.lane, sc);
        ChunkSink sink;
        sink.gram = sc.target;
        if (rc == VPCA_OK) rc = packed_chunks(ctx, *lg.lane, bits, nv, stride_bytes, code, sink);
        if (rc == VPCA_OK) lane_gram_time(ctx, *lg.lane);
    }
    return sc.end(rc);
}

int vpca_accumulate_bits(vpca_ctx* ctx, int64_t partition_id, const uint8_t* bits, int64_t nv, int64_t stride_bytes) {
    return accumulate_packed(ctx, partition_id, bits, nv, stride_bytes, 0);
}

int vpca_accumulate_bed(vpca_ctx* ctx, int64_t partition_id, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                        int32_t counted_allele) {
    if (counted_allele != 1 && counted_allele != 2)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_accumulate_bed: counted_allele must be 1 (A1) or 2 (A2)");
    return accumulate_packed(ctx, partition_id, rows, nv, stride_bytes, counted_allele);
}

// ---- multi-dataset keying (join.cu) -----------------------------------------------------------------------------
int vpca_hash_keys(vpca_ctx* ctx, const uint8_t* payload, const int64_t* key_offsets, int64_t nkeys, uint64_t* out) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    if (nkeys < 0 || key_offsets == nullptr || (nkeys > 0 && out == nullptr))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_hash_keys: bad argument");
    if (nkeys == 0) return VPCA_OK;
    for (int64_t q = 0; q < nkeys; ++q)
        if (key_offsets[q + 1] < key_offsets[q] || key_offsets[0] < 0)
            return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_hash_keys: key_offsets must be non-negative and non-decreasing (key %lld)", (long long)q);
    const int64_t bytes = key_offsets[nkeys] - key_offsets[0];
    if (bytes > 0 && payload == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_hash_keys: payload is NULL");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    uint8_t* d_pay = nullptr;
    int64_t* d_koff = nullptr;
    uint64_t* d_out = nullptr;
    cudaError_t e = cudaMalloc(&d_pay, (size_t)bytes + 16);
    if (e == cudaSuccess) e = cudaMalloc(&d_koff, (size_t)(nkeys + 1) * 8);
    if (e == cudaSuccess) e = cudaMalloc(&d_out, (size_t)nkeys * 16);
    if (e == cudaSuccess && bytes > 0)
        e = cudaMemcpyAsync(d_pay, payload + key_offsets[0], (size_t)bytes, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d_koff, key_offsets, (size_t)(nkeys + 1) * 8, cudaMemcpyHostToDevice, ctx->stream);
    // the device copy starts at the first key: shift the base pointer instead of rebasing the offsets
    if (e == cudaSuccess) e = hash_keys(d_pay - key_offsets[0], d_koff, nkeys, d_out, ctx->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(out, d_out, (size_t)nkeys * 16, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(d_pay);
    cudaFree(d_koff);
    cudaFree(d_out);
    if (e != cudaSuccess) return fail(ctx, VPCA_ERR_CUDA, "vpca_hash_keys: %s", cudaGetErrorString(e));
    ctx->c_launches += 1;
    ctx->c_h2d += bytes + (nkeys + 1) * 8;
    ctx->c_d2h += nkeys * 16;
    return VPCA_OK;
}

int vpca_join_rows(vpca_ctx* ctx, int32_t mode, int32_t variant_set_count, int64_t n_left, const uint8_t* key_payload,
                   const int64_t* key_offsets, const int64_t* offsets, const int32_t* sample_idx, int64_t nrows,
                   int64_t* out_rows, int64_t* out_nnz) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    if ((mode != VPCA_JOIN && mode != VPCA_MERGE) || nrows < 0 || nrows > 0x7ffffff0ll || key_offsets == nullptr ||
        offsets == nullptr || out_rows == nullptr || out_nnz == nullptr)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_join_rows: bad argument");
    if (mode == VPCA_JOIN && (n_left < 0 || n_left > nrows))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_join_rows: n_left must be in [0, nrows]");
    if (mode == VPCA_MERGE && variant_set_count < 1)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_join_rows: variant_set_count must be >= 1");
    if (key_offsets[0] < 0 || offsets[0] < 0) return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_join_rows: negative offset");
    for (int64_t q = 0; q < nrows; ++q)
        if (key_offsets[q + 1] < key_offsets[q] || offsets[q + 1] < offsets[q])
            return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_join_rows: offsets must be non-decreasing (row %lld)", (long long)q);
    const int64_t kbytes = key_offsets[nrows] - key_offsets[0], nnz = offsets[nrows] - offsets[0];
    if ((kbytes > 0 && key_payload == nullptr) || (nnz > 0 && sample_idx == nullptr))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_join_rows: NULL payload");
    std::lock_guard<std::mutex> jl(ctx->join_mu);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    JoinWork& w = ctx->join;
    w.out_rows = -1;
    CUDA_OK(ctx, grow_buffer(&w.d_payload, &w.cap_payload, kbytes + 16));
    if (nrows + 1 > w.cap_in_rows || w.d_key_off == nullptr || w.d_off == nullptr) {
        cudaFree(w.d_key_off);
        cudaFree(w.d_off);
        w.d_key_off = w.d_off = nullptr;
        w.cap_in_rows = 0;
        const int64_t c = nrows + nrows / 4 + 1024;
        CUDA_OK(ctx, cudaMalloc(&w.d_key_off, (size_t)c * 8));
        CUDA_OK(ctx, cudaMalloc(&w.d_off, (size_t)c * 8));
        w.cap_in_rows = c;
    }
    CUDA_OK(ctx, grow_buffer(&w.d_idx, &w.cap_in_nnz, nnz + 1));
    if (kbytes > 0)
        CUDA_OK(ctx, cudaMemcpyAsync(w.d_payload, key_payload + key_offsets[0], (size_t)kbytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_OK(ctx, cudaMemcpyAsync(w.d_key_off, key_offsets, (size_t)(nrows + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_OK(ctx, cudaMemcpyAsync(w.d_off, offsets, (size_t)(nrows + 1) * 8, cudaMemcpyHostToDevice, ctx->stream));
    if (nnz > 0)
        CUDA_OK(ctx, cudaMemcpyAsync(w.d_idx, sample_idx + offsets[0], (size_t)nnz * 4, cudaMemcpyHostToDevice, ctx->stream));
    ctx->c_h2d += kbytes + 2 * (nrows + 1) * 8 + nnz * 4;
    int64_t launches = 0, rows = 0, calls = 0;
    // the device copies start at the first key / first call: shift the base pointers instead of rebasing the offsets
    cudaError_t e = join_rows(w, mode, variant_set_count, n_left, w.d_payload - key_offsets[0], w.d_key_off, w.d_off,
                              w.d_idx - offsets[0], nrows, ctx->stream, &rows, &calls, &launches);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);   // the caller's buffers were read asynchronously
    ctx->c_launches += launches;
    if (e != cudaSuccess)
        return fail(ctx, e == cudaErrorMemoryAllocation ? VPCA_ERR_NOMEM : VPCA_ERR_CUDA, "vpca_join_rows: %s", cudaGetErrorString(e));
    w.out_rows = rows;
    w.out_nnz = calls;
    *out_rows = rows;
    *out_nnz = calls;
    return VPCA_OK;
}

int vpca_join_fetch(vpca_ctx* ctx, int64_t* out_offsets, int32_t* out_idx) {
    if (ctx == nullptr || out_offsets == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    std::lock_guard<std::mutex> jl(ctx->join_mu);
    JoinWork& w = ctx->join;
    if (w.out_rows < 0) return fail(ctx, VPCA_ERR_STATE, "no joined rows: call vpca_join_rows first");
    if (w.out_nnz > 0 && out_idx == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "out_idx is NULL");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaMemcpyAsync(out_offsets, w.d_out_off, (size_t)(w.out_rows + 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    if (w.out_nnz > 0)
        CUDA_OK(ctx, cudaMemcpyAsync(out_idx, w.d_out_idx, (size_t)w.out_nnz * 4, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (w.out_rows + 1) * 8 + w.out_nnz * 4;
    return VPCA_OK;
}

int vpca_join_size(vpca_ctx* ctx, int64_t* out_rows, int64_t* out_nnz) {
    if (ctx == nullptr || out_rows == nullptr || out_nnz == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    std::lock_guard<std::mutex> jl(ctx->join_mu);
    if (ctx->join.out_rows < 0) return fail(ctx, VPCA_ERR_STATE, "no joined rows: call vpca_join_rows first");
    *out_rows = ctx->join.out_rows;
    *out_nnz = ctx->join.out_nnz;
    return VPCA_OK;
}

int vpca_accumulate_joined(vpca_ctx* ctx, int64_t partition_id) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> jl(ctx->join_mu);
    JoinWork& w = ctx->join;
    if (w.out_rows < 0) return fail(ctx, VPCA_ERR_STATE, "no joined rows: call vpca_join_rows first");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const int64_t nv = w.out_rows;
    if (nv == 0) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
        return VPCA_OK;
    }
    CallScope sc{ctx, partition_id, nv};
    int rc = sc.begin();
    if (rc != VPCA_OK) return rc;
    auto body = [&](vpca_ctx::Lane& L) -> int {
        int r = prepare_slot(ctx, L, sc);
        if (r != VPCA_OK) return r;
        *L.h_flags = 0;
        CUDA_OK(ctx, cudaMemsetAsync(L.d_flags, 0, sizeof(int), L.stream));
        const int64_t P = ctx->panel;
        int chunk = 0;
        for (int64_t v = 0; v < nv; v += ctx->chunk_variants, ++chunk) {
            const int64_t nvc = std::min(ctx->chunk_variants, nv - v);
            const int b = chunk & 1;
            // the joined CSR is device-resident: rows [v, v + nvc) are encoded straight from it (absolute offsets, base 0)
            CUDA_OK(ctx, encode_calls(w.d_out_off + v, 0, w.d_out_idx, 4, nvc, ctx->rows(), ctx->elem_bits, ctx->max_mult,
                                      L.d_x[b], P, P, ctx->d_rows, L.d_flags, L.stream));
            ctx->c_launches += 2;
            r = launch_gram(ctx, L.plan, L.stream, L.ev_t0, L.ev_t1, L.d_x[b], nvc, P, P, sc.target);
            if (r != VPCA_OK) return r;
        }
        CUDA_OK(ctx, cudaMemcpyAsync(L.h_flags, L.d_flags, sizeof(int), cudaMemcpyDeviceToHost, L.stream));
        CUDA_OK(ctx, cudaStreamSynchronize(L.stream));
        lane_gram_time(ctx, L);
        if (*L.h_flags & 1)
            return fail(ctx, VPCA_ERR_INDEX_OUT_OF_RANGE, "sample index outside [0, %d) (the reference throws at "
                        "VariantsPca.scala:59/:188)", ctx->rows());
        if (*L.h_flags & 2)
            return fail(ctx, VPCA_ERR_OVERFLOW, "a sample is listed more than max_multiplicity=%d times in one joined row "
                        "(a sample present in both datasets counts twice, VariantsPca.scala:127/:187)", ctx->max_mult);
        return VPCA_OK;
    };
    {
        LaneGuard lg(ctx);   // orders the lane after the join kernels on the context's stream
        rc = lg.rc;
        if (rc == VPCA_OK) rc = body(*lg.lane);
    }
    return sc.end(rc);
}

int vpca_commit(vpca_ctx* ctx, int64_t partition_id) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized");
    int rc;
    vpca_ctx::Slot* s = find_slot(ctx, partition_id, false, &rc);
    if (s == nullptr) return VPCA_OK;   // an empty partition never staged anything
    if (s->busy) return fail(ctx, VPCA_ERR_STATE, "partition %lld still has an accumulate call in flight", (long long)partition_id);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (ctx->scoring) {
        // the partial is kept as it is, per partition id: vpca_score_project adds them in ascending id, so the result does
        // not depend on the commit order; a partition committed again replaces its earlier partial (it counts once)
        if (s->nv > 0) {
            vpca_ctx::Scored& dst = ctx->scored[partition_id];
            if (dst.d_acc == nullptr) {
                cudaError_t e = cudaMalloc(&dst.d_acc, ctx->slot_bytes());
                if (e != cudaSuccess) {
                    ctx->scored.erase(partition_id);
                    return fail(ctx, VPCA_ERR_NOMEM, "cudaMalloc of a partition score failed: %s", cudaGetErrorString(e));
                }
            }
            CUDA_OK(ctx, cudaMemcpyAsync(dst.d_acc, s->d_S, ctx->slot_bytes(), cudaMemcpyDeviceToDevice, ctx->stream));
            CUDA_OK(ctx, cudaEventRecord(s->ev_free, ctx->stream));
            dst.matched = s->matched;
        }
        ctx->total_variants += s->nv;
        ctx->inflight_variants -= s->nv;
        s->used = false;
        return VPCA_OK;
    }
    // the partition's variants were reserved against the int32 bound when they were staged (CallScope::begin)
    if (s->nv > 0) {
        // every accumulate call of the partition synchronised its lane before returning: the staging Gram is complete
        if (ctx->plan.num_peers > 1 && ctx->plan.peer_mode == 1)
            CUDA_OK(ctx, gram_add_owners(ctx->plan, s->d_S, ctx->n, ctx->stream));
        else if (ctx->plan.num_peers > 1)
            CUDA_OK(ctx, gram_add_peers(ctx->plan, s->d_S, (int64_t)ctx->n * ctx->n, ctx->stream));
        else
            CUDA_OK(ctx, gram_add(ctx->d_S, s->d_S, (int64_t)ctx->rows() * ctx->n, ctx->stream));
        CUDA_OK(ctx, cudaEventRecord(s->ev_free, ctx->stream));
        ctx->c_launches += 1;
    }
    ctx->total_variants += s->nv;
    ctx->inflight_variants -= s->nv;
    s->used = false;
    return VPCA_OK;
}

int vpca_abort(vpca_ctx* ctx, int64_t partition_id) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    int rc;
    vpca_ctx::Slot* s = find_slot(ctx, partition_id, false, &rc);
    if (s != nullptr) {
        if (s->busy) return fail(ctx, VPCA_ERR_STATE, "partition %lld still has an accumulate call in flight", (long long)partition_id);
        ctx->st.variants_accumulated -= s->nv;
        ctx->inflight_variants -= s->nv;
        s->used = false;
    }
    return VPCA_OK;
}

int vpca_accumulate_dense(vpca_ctx* ctx, const void* x, int64_t nv, int64_t ld, int on_device) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    if (x == nullptr || nv < 0 || ld < nv) return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_accumulate_dense: bad argument");
    const int bits = ctx->elem_bits;
    if (bits == 4 && (ld % 128) != 0)
        return fail(ctx, VPCA_ERR_BAD_ARG, "packed e2m1 tiles need ld %% 128 == 0 (and zero padding up to a multiple of 128 variants)");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (on_device) {
        std::lock_guard<std::mutex> lk(ctx->mu);
        if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
        if (nv == 0) return VPCA_OK;
        int rc = check_overflow(ctx, nv);
        if (rc != VPCA_OK) return rc;
        const int align = bits == 4 ? 31 : 15;
        if ((reinterpret_cast<uintptr_t>(x) & align) != 0 || ((ld * bits / 8) & align) != 0)
            return fail(ctx, VPCA_ERR_BAD_ARG, "device tile must be %d-byte aligned with a %d-byte multiple row pitch",
                        align + 1, align + 1);
        rc = launch_gram(ctx, ctx->plan, ctx->stream, ctx->ev_t0, ctx->ev_t1, x, nv, ld, 0, ctx->d_S);
        if (rc != VPCA_OK) return rc;
        ctx->gram_timed = true;
        ctx->st.gram_cta_group = ctx->plan.cta_group;
        ctx->st.gram_resident = ctx->plan.last_resident;
        ctx->total_variants += nv;
        ctx->st.variants_accumulated += nv;
        return VPCA_OK;
    }
    if (nv == 0) return VPCA_OK;
    CallScope sc{ctx, -1, nv};
    int rc = sc.begin();
    if (rc != VPCA_OK) return rc;
    auto body = [&](vpca_ctx::Lane& L) -> int {
        int chunk = 0;
        for (int64_t v = 0; v < nv; v += ctx->chunk_variants, ++chunk) {
            const int64_t nvc = std::min(ctx->chunk_variants, nv - v);
            const int b = chunk & 1;
            CUDA_OK(ctx, cudaStreamWaitEvent(L.copy_stream, L.ev_done[b], 0));
            // the caller's row-major tile -> panel layout, one 2-D copy per panel; a partial last panel is zeroed first
            const int64_t P = ctx->panel;
            if ((nvc % P) != 0)
                CUDA_OK(ctx, cudaMemsetAsync(static_cast<char*>(L.d_x[b]) + (size_t)(nvc / P) * ctx->rows() * P * bits / 8, 0,
                                             (size_t)ctx->rows() * P * bits / 8, L.copy_stream));
            for (int64_t pv = 0; pv < nvc; pv += P) {
                const int64_t wv = std::min(P, nvc - pv);
                CUDA_OK(ctx, cudaMemcpy2DAsync(static_cast<char*>(L.d_x[b]) + (size_t)(pv / P) * ctx->rows() * P * bits / 8,
                                               (size_t)P * bits / 8, static_cast<const char*>(x) + (size_t)(v + pv) * bits / 8,
                                               (size_t)ld * bits / 8, (size_t)(wv * bits + 7) / 8, (size_t)ctx->rows(),
                                               cudaMemcpyHostToDevice, L.copy_stream));
            }
            CUDA_OK(ctx, cudaEventRecord(L.ev_copy[b], L.copy_stream));
            ctx->c_h2d += (nvc * bits + 7) / 8 * (int64_t)ctx->rows();
            CUDA_OK(ctx, cudaStreamWaitEvent(L.stream, L.ev_copy[b], 0));
            int r = launch_gram(ctx, L.plan, L.stream, L.ev_t0, L.ev_t1, L.d_x[b], nvc, P, P, ctx->d_S);
            if (r != VPCA_OK) return r;
            CUDA_OK(ctx, cudaEventRecord(L.ev_done[b], L.stream));
        }
        CUDA_OK(ctx, cudaStreamSynchronize(L.stream));   // caller's buffer is free to reuse on return
        lane_gram_time(ctx, L);
        return VPCA_OK;
    };
    {
        LaneGuard lg(ctx);
        rc = lg.rc;
        if (rc == VPCA_OK) rc = body(*lg.lane);
    }
    return sc.end(rc);
}

int vpca_accumulate_panels(vpca_ctx* ctx, const void* d_x, int64_t nv, int64_t panel_variants) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (d_x == nullptr || nv < 0 || panel_variants < 128 || (panel_variants % 128) != 0)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_accumulate_panels: panel_variants must be a positive multiple of 128");
    if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
    if ((reinterpret_cast<uintptr_t>(d_x) & 31) != 0) return fail(ctx, VPCA_ERR_BAD_ARG, "panels must be 32-byte aligned");
    // a band-only Gram either has peers in owner-rows mode (every context gets a variant shard and flushes each row to
    // its owner) or no peers at all (owner-computes: every context gets ALL variants and produces only its own rows)
    if (ctx->band_rows != ctx->n && ctx->plan.num_peers > 1 && ctx->plan.peer_mode != 1)
        return fail(ctx, VPCA_ERR_STATE, "a band-only Gram with peers needs VPCA_PEER_OWNER_ROWS");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    int rc = check_overflow(ctx, nv);
    if (rc != VPCA_OK) return rc;
    ChunkSink sink;
    sink.gram = ctx->d_S;
    rc = consume_chunk(ctx, ctx->plan, ctx->stream, ctx->ev_t0, ctx->ev_t1, sink, d_x, 0, nv, panel_variants);
    if (rc != VPCA_OK) return rc;
    ctx->gram_timed = true;
    ctx->st.gram_cta_group = ctx->plan.cta_group;
    ctx->st.gram_resident = ctx->plan.last_resident;
    ctx->total_variants += nv;
    ctx->st.variants_accumulated += nv;
    return VPCA_OK;
}

int vpca_synth_panels_device(vpca_ctx* ctx, uint64_t seed, int64_t v0, int64_t nv, int mode, void* d_x,
                             int64_t panel_variants) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (d_x == nullptr || nv < 0 || v0 < 0 || (mode != 0 && mode != 1) || panel_variants < 128 || (panel_variants % 128) != 0)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_synth_panels_device: bad argument");
    if (mode == 1 && ctx->max_mult < 2) return fail(ctx, VPCA_ERR_BAD_ARG, "dosage mode needs max_multiplicity >= 2");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    cudaError_t e = synth_dense(seed, ctx->rows(), v0, nv, mode, ctx->elem_bits, d_x, panel_variants, panel_variants, ctx->stream);
    if (e != cudaSuccess) return fail(ctx, VPCA_ERR_CUDA, "synthetic generator: %s", cudaGetErrorString(e));
    ctx->c_launches += 2 * ((nv + (1 << 22) - 1) >> 22);
    return VPCA_OK;
}

int vpca_gram_device_ptr(vpca_ctx* ctx, void** d_gram) {
    if (ctx == nullptr || d_gram == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    *d_gram = ctx->d_S;
    return VPCA_OK;
}

int vpca_finalize_gram(vpca_ctx* ctx) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->finalized) return VPCA_OK;
    for (auto& s : ctx->slots)
        if (s.used)
            return fail(ctx, VPCA_ERR_STATE, "partition %lld is neither committed nor aborted", (long long)s.pid);
    for (auto& L : ctx->lanes)
        if (L.busy) return fail(ctx, VPCA_ERR_STATE, "vpca_finalize_gram while an accumulate call is in flight");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (ctx->band_rows == ctx->n) {   // a row band stays a band of the lower triangle: nothing to mirror into
        CUDA_OK(ctx, gram_symmetrize(ctx->d_S, ctx->n, ctx->stream));
        ctx->c_launches += 1;
    }
    ctx->finalized = true;
    ctx->pca_done = false;
    ctx->proj_k = 0;
    return VPCA_OK;
}

static int copy_gram_out(vpca_ctx* ctx, int32_t* out, size_t cells) {
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaMemcpyAsync(out, ctx->d_S, cells * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (int64_t)(cells * sizeof(int32_t));
    return VPCA_OK;
}

int vpca_get_gram(vpca_ctx* ctx, int32_t* out) {
    if (ctx == nullptr || out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "call vpca_finalize_gram first");
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "this context stores a row band: use vpca_get_gram_band");
    return copy_gram_out(ctx, out, (size_t)ctx->n * ctx->n);
}

int vpca_get_gram_band(vpca_ctx* ctx, int32_t row0, int32_t rows, int32_t* out) {
    if (ctx == nullptr || out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (rows <= 0 || row0 < ctx->band_row0 || row0 + rows > ctx->band_row0 + ctx->band_rows)
        return fail(ctx, VPCA_ERR_BAD_ARG, "rows [%d, %d) are outside the band [%d, %d) this context stores", row0, row0 + rows,
                    ctx->band_row0, ctx->band_row0 + ctx->band_rows);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const size_t cells = (size_t)rows * ctx->n;
    CUDA_OK(ctx, cudaMemcpyAsync(out, ctx->d_S + (size_t)(row0 - ctx->band_row0) * ctx->n, cells * sizeof(int32_t),
                                 cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (int64_t)(cells * sizeof(int32_t));
    return VPCA_OK;
}

int vpca_get_partial_gram(vpca_ctx* ctx, int32_t* out, int64_t* variants_in_gram) {
    if (ctx == nullptr || out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized: use vpca_get_gram");
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "this context stores a row band: use vpca_get_gram_band");
    if (variants_in_gram) *variants_in_gram = ctx->total_variants;
    return copy_gram_out(ctx, out, ctx->gram_cells());
}

int vpca_load_partial_gram(vpca_ctx* ctx, const int32_t* gram, int64_t variants_in_gram) {
    if (ctx == nullptr || gram == nullptr || variants_in_gram < 0) return fail(ctx, VPCA_ERR_BAD_ARG, "bad argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized; call vpca_reset first");
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "this context stores a row band");
    for (auto& s : ctx->slots)
        if (s.used) return fail(ctx, VPCA_ERR_STATE, "partition %lld is in flight", (long long)s.pid);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const size_t bytes = ctx->gram_cells() * sizeof(int32_t);
    CUDA_OK(ctx, cudaMemcpyAsync(ctx->d_S, gram, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_h2d += (int64_t)bytes;
    // the restored counts keep counting against the int32 bound (VariantsPca.scala:185)
    ctx->total_variants = variants_in_gram;
    ctx->inflight_variants = 0;
    return check_overflow(ctx, 0);
}

int vpca_set_gram(vpca_ctx* ctx, const int32_t* gram) {
    if (ctx == nullptr || gram == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "this context stores a row band");
    if (ctx->n_proj > 0)
        return fail(ctx, VPCA_ERR_UNSUPPORTED, "a projecting context computes its cross block from genotypes: vpca_set_gram "
                    "would leave it stale");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const size_t bytes = (size_t)ctx->n * ctx->n * sizeof(int32_t);
    CUDA_OK(ctx, cudaMemcpyAsync(ctx->d_S, gram, bytes, cudaMemcpyHostToDevice, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_h2d += (int64_t)bytes;
    for (auto& s : ctx->slots) s.used = false;
    ctx->inflight_variants = 0;
    ctx->finalized = true;
    ctx->pca_done = false;
    return VPCA_OK;
}

int64_t vpca_variant_count(vpca_ctx* ctx) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    return ctx->total_variants;
}

static int run_center(vpca_ctx* ctx, bool materialise) {
    if (!ctx->eig_ready) {
        cudaError_t e = eig_alloc(ctx->eig, ctx->n, std::max(ctx->num_pc, 16));
        if (e != cudaSuccess) {
            eig_free(ctx->eig);
            return fail(ctx, VPCA_ERR_NOMEM, "eigensolver workspace: %s", cudaGetErrorString(e));
        }
        ctx->eig_ready = true;
    }
    CUDA_OK(ctx, center_gram(ctx->eig, ctx->d_S, ctx->stream, materialise));
    ctx->c_launches += materialise ? 3 : 2;
    return VPCA_OK;
}

int vpca_compute_pca(vpca_ctx* ctx, int32_t k, double* vecs, double* evals, int32_t* non_zero_rows) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (vecs == nullptr || k < 1 || k > ctx->n || k > std::max(ctx->num_pc, 16))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_compute_pca: k=%d out of range", k);
    if (!ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "call vpca_finalize_gram first");
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "this context stores a row band of the Gram");
    if (ctx->n > 65535)
        return fail(ctx, VPCA_ERR_UNSUPPORTED, "computePca is limited to 65535 samples, like the reference (MLlib RowMatrix "
                    "behind VariantsPca.scala:226 refuses more columns); the Gram itself has no such limit");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaEventRecord(ctx->ev_e0, ctx->stream));
    int rc = run_center(ctx, false);   // row sums + mean; the solver materialises C only if it needs it
    if (rc != VPCA_OK) return rc;
    {   // VPCA_EIG=direct|lanczos|auto (default auto: Lanczos from 512 samples up, direct reduction as its fallback)
        const char* em = getenv("VPCA_EIG");
        ctx->eig.mode = (em != nullptr && strcmp(em, "direct") == 0) ? 1 : (em != nullptr && strcmp(em, "lanczos") == 0) ? 2 : 0;
    }
    int64_t launches = 0;
    CUDA_OK(ctx, eig_topk(ctx->eig, k, ctx->stream, &launches));
    ctx->c_launches += launches;
    CUDA_OK(ctx, cudaEventRecord(ctx->ev_e1, ctx->stream));
    ctx->st.eig_method = ctx->eig.last_method;
    ctx->st.eig_iterations = ctx->eig.last_iters;
    ctx->eig_timed = true;
    const size_t nb = (size_t)ctx->n * k * sizeof(double);
    CUDA_OK(ctx, cudaMemcpyAsync(vecs, ctx->eig.d_evecs, nb, cudaMemcpyDeviceToHost, ctx->stream));
    if (evals) CUDA_OK(ctx, cudaMemcpyAsync(evals, ctx->eig.d_evals, k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    int nz = 0;
    CUDA_OK(ctx, cudaMemcpyAsync(&nz, ctx->eig.d_nz, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    if (non_zero_rows) *non_zero_rows = nz;
    ctx->c_d2h += (int64_t)nb + (evals ? k * 8 : 0) + 4;
    ctx->pca_done = true;
    ctx->proj_k = k;
    return VPCA_OK;
}

int vpca_get_cross_gram(vpca_ctx* ctx, int32_t* out) {
    if (ctx == nullptr || out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "call vpca_finalize_gram first");
    if (ctx->n_proj == 0) return VPCA_OK;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const size_t cells = (size_t)ctx->n_proj * ctx->n;
    CUDA_OK(ctx, cudaMemcpyAsync(out, ctx->d_S + (size_t)ctx->n * ctx->n, cells * sizeof(int32_t), cudaMemcpyDeviceToHost,
                                 ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (int64_t)(cells * sizeof(int32_t));
    return VPCA_OK;
}

int vpca_project_pca(vpca_ctx* ctx, int32_t k, double* out) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->proj_k == 0) return fail(ctx, VPCA_ERR_STATE, "call vpca_compute_pca first");
    if (k < 1 || k > ctx->proj_k)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_project_pca: k=%d outside [1, %d] (the k of the last vpca_compute_pca)", k,
                    ctx->proj_k);
    if (ctx->n_proj == 0) return VPCA_OK;
    if (out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "out is NULL");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const int m = ctx->n_proj, kmax = std::max(ctx->num_pc, 16);
    const size_t part = (size_t)proj_chunks(ctx->n) * m * kmax;
    if (ctx->d_proj == nullptr) {
        cudaError_t e = cudaMalloc(&ctx->d_proj, ((size_t)m + part + (size_t)m * kmax) * sizeof(double));
        if (e != cudaSuccess) {
            ctx->d_proj = nullptr;
            return fail(ctx, VPCA_ERR_NOMEM, "projection workspace: %s", cudaGetErrorString(e));
        }
    }
    double* d_rowmean = ctx->d_proj;
    double* d_part = d_rowmean + m;
    double* d_y = d_part + part;
    CUDA_OK(ctx, eig_project(ctx->eig, ctx->d_S + (size_t)ctx->n * ctx->n, m, k, d_rowmean, d_part, d_y, ctx->stream));
    ctx->c_launches += 3;
    CUDA_OK(ctx, cudaMemcpyAsync(out, d_y, (size_t)m * k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (int64_t)m * k * 8;
    return VPCA_OK;
}

// ---- saved model: loadings of a fitted context, scoring of a study context (model.cu) -------------------------------
static int loadings_args(vpca_ctx* ctx, int32_t k, int64_t nv, const double* loadings, const int32_t* carriers) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    if (nv < 0 || (nv > 0 && (loadings == nullptr || carriers == nullptr)))
        return fail(ctx, VPCA_ERR_BAD_ARG, "loadings: nv must be >= 0 and the outputs non-NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->proj_k == 0) return fail(ctx, VPCA_ERR_STATE, "call vpca_compute_pca first");
    if (k < 1 || k > ctx->proj_k)
        return fail(ctx, VPCA_ERR_BAD_ARG, "loadings: k=%d outside [1, %d] (the k of the last vpca_compute_pca)", k, ctx->proj_k);
    return VPCA_OK;
}

static size_t align256(size_t b) { return (b + 255) & ~(size_t)255; }

// Loadings sink of a lane: device output for one chunk in the lane's scratch.
static int lane_loadings_sink(vpca_ctx* ctx, vpca_ctx::Lane& L, int32_t k, double* loadings, int32_t* carriers, ChunkSink& sink) {
    const int64_t cv = ctx->chunk_variants;
    const size_t lb = align256((size_t)cv * k * sizeof(double));
    CUDA_OK(ctx, grow_buffer(&L.d_scratch, &L.cap_scratch, (int64_t)(lb + (size_t)cv * sizeof(int32_t))));
    sink.kind = ChunkSink::LOADINGS;
    sink.k = k;
    sink.d_L = reinterpret_cast<double*>(L.d_scratch);
    sink.d_cnt = reinterpret_cast<int32_t*>(L.d_scratch + lb);
    sink.h_L = loadings;
    sink.h_cnt = carriers;
    return VPCA_OK;
}

int vpca_pca_loadings_calls(vpca_ctx* ctx, int32_t k, const int64_t* offsets, const int32_t* sample_idx, int64_t nv,
                            double* loadings, int32_t* carriers) {
    int rc = loadings_args(ctx, k, nv, loadings, carriers);
    if (rc != VPCA_OK) return rc;
    if (offsets == nullptr || (nv > 0 && sample_idx == nullptr && offsets[nv] > offsets[0]))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_pca_loadings_calls: bad argument");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    LaneGuard lg(ctx);
    if (lg.rc != VPCA_OK) return lg.rc;
    ChunkSink sink;
    rc = lane_loadings_sink(ctx, *lg.lane, k, loadings, carriers, sink);
    if (rc != VPCA_OK) return rc;
    return process_calls(ctx, *lg.lane, offsets, sample_idx, 4, nv, &sink, nullptr, 0);
}

int vpca_pca_loadings_bed(vpca_ctx* ctx, int32_t k, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                          int32_t counted_allele, double* loadings, int32_t* carriers) {
    int rc = loadings_args(ctx, k, nv, loadings, carriers);
    if (rc != VPCA_OK) return rc;
    if (counted_allele != 1 && counted_allele != 2)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_pca_loadings_bed: counted_allele must be 1 (A1) or 2 (A2)");
    rc = packed_args(ctx, rows, nv, stride_bytes, counted_allele);
    if (rc != VPCA_OK) return rc;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    LaneGuard lg(ctx);
    if (lg.rc != VPCA_OK) return lg.rc;
    ChunkSink sink;
    rc = lane_loadings_sink(ctx, *lg.lane, k, loadings, carriers, sink);
    if (rc != VPCA_OK) return rc;
    return packed_chunks(ctx, *lg.lane, rows, nv, stride_bytes, counted_allele, sink);
}

static int panels_args(vpca_ctx* ctx, const void* d_x, int64_t nv, int64_t panel_variants) {
    if (d_x == nullptr || nv < 0 || panel_variants < 128 || (panel_variants % 128) != 0)
        return fail(ctx, VPCA_ERR_BAD_ARG, "panels: panel_variants must be a positive multiple of 128");
    if ((reinterpret_cast<uintptr_t>(d_x) & 31) != 0) return fail(ctx, VPCA_ERR_BAD_ARG, "panels must be 32-byte aligned");
    return VPCA_OK;
}

int vpca_pca_loadings_panels(vpca_ctx* ctx, int32_t k, const void* d_x, int64_t nv, int64_t panel_variants, double* loadings,
                             int32_t* carriers) {
    int rc = loadings_args(ctx, k, nv, loadings, carriers);
    if (rc != VPCA_OK) return rc;
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = panels_args(ctx, d_x, nv, panel_variants);
    if (rc != VPCA_OK) return rc;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    const size_t lb = align256((size_t)nv * k * sizeof(double));
    CUDA_OK(ctx, grow_buffer(&ctx->d_scratch, &ctx->cap_scratch, (int64_t)(lb + (size_t)nv * sizeof(int32_t))));
    ChunkSink sink;
    sink.kind = ChunkSink::LOADINGS;
    sink.k = k;
    sink.d_L = reinterpret_cast<double*>(ctx->d_scratch);
    sink.d_cnt = reinterpret_cast<int32_t*>(ctx->d_scratch + lb);
    sink.h_L = loadings;
    sink.h_cnt = carriers;
    rc = consume_chunk(ctx, ctx->plan, ctx->stream, ctx->ev_t0, ctx->ev_t1, sink, d_x, 0, nv, panel_variants);
    if (rc != VPCA_OK) return rc;
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return VPCA_OK;
}

int vpca_pca_model_terms(vpca_ctx* ctx, int32_t k, double* eigenvalues, double* col_sums, double* rowsum_dots,
                         double* matrix_mean) {
    int rc = loadings_args(ctx, k, 0, nullptr, nullptr);
    if (rc != VPCA_OK) return rc;
    if (eigenvalues == nullptr || col_sums == nullptr || rowsum_dots == nullptr || matrix_mean == nullptr)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_pca_model_terms: NULL argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, grow_buffer(&ctx->d_scratch, &ctx->cap_scratch, (int64_t)(2 * k * sizeof(double))));
    double* d_a = reinterpret_cast<double*>(ctx->d_scratch);
    CUDA_OK(ctx, model_terms(ctx->eig.d_evecs, ctx->eig.d_rowsum, ctx->n, k, d_a, d_a + k, ctx->stream));
    ctx->c_launches += 1;
    CUDA_OK(ctx, cudaMemcpyAsync(col_sums, d_a, k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaMemcpyAsync(rowsum_dots, d_a + k, k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaMemcpyAsync(eigenvalues, ctx->eig.d_evals, k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaMemcpyAsync(matrix_mean, ctx->eig.d_mm, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (3 * k + 1) * 8;
    return VPCA_OK;
}

int vpca_create_scoring(const vpca_config* cfg, const vpca_model* model, vpca_ctx** out) {
    if (out != nullptr) *out = nullptr;
    if (model == nullptr || model->struct_size != sizeof(vpca_model))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "model is NULL or struct_size != sizeof(vpca_model) (%zu)", sizeof(vpca_model));
    if (model->n_fitted < 2 || model->k < 1 || model->n_variants < 0 || model->n_variants > 0x7fffffffll)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "model: need n_fitted >= 2, k >= 1 and 0 <= n_variants < 2^31");
    if ((model->n_variants > 0 && (model->loadings == nullptr || model->carriers == nullptr)) || model->eigenvalues == nullptr ||
        model->col_sums == nullptr || model->rowsum_dots == nullptr)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "model: NULL array");
    if (cfg != nullptr && cfg->struct_size == sizeof(vpca_config) && (cfg->d_gram != nullptr || cfg->gram_band_rows > 0))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "a scoring context has no Gram: d_gram and gram_band_rows must be unset");
    return create_impl(cfg, 0, nullptr, model, out);
}

// Validates the model rows of a scoring call and counts the variants that have one.
static int score_args(vpca_ctx* ctx, int64_t nv, const int32_t* model_rows, int64_t* matched) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    if (!ctx->scoring) return fail(ctx, VPCA_ERR_UNSUPPORTED, "scoring needs a context made by vpca_create_scoring");
    if (nv < 0 || (nv > 0 && model_rows == nullptr)) return fail(ctx, VPCA_ERR_BAD_ARG, "scoring: bad argument");
    int64_t cnt = 0;
    for (int64_t q = 0; q < nv; ++q) {
        const int32_t r = model_rows[q];
        if (r < -1 || r >= ctx->model_nv)
            return fail(ctx, VPCA_ERR_INDEX_OUT_OF_RANGE, "model row %d of variant %lld is outside [-1, %lld)", r, (long long)q,
                        (long long)ctx->model_nv);
        cnt += r >= 0;
    }
    *matched = cnt;
    return VPCA_OK;
}

// Scoring sink: the model rows of the call are copied to the device once, next to the scratch of model_score.
static int score_sink(vpca_ctx* ctx, char** buf, int64_t* cap, cudaStream_t stream, const int32_t* model_rows, int64_t nv,
                      double* acc, ChunkSink& sink) {
    const size_t rb = align256((size_t)nv * sizeof(int32_t));
    CUDA_OK(ctx, grow_buffer(buf, cap, (int64_t)(rb + model_score_scratch(ctx->n, ctx->model_k))));
    CUDA_OK(ctx, cudaMemcpyAsync(*buf, model_rows, (size_t)nv * sizeof(int32_t), cudaMemcpyHostToDevice, stream));
    ctx->c_h2d += nv * 4;
    sink.kind = ChunkSink::SCORE;
    sink.k = ctx->model_k;
    sink.d_mrows = reinterpret_cast<const int32_t*>(*buf);
    sink.d_part = reinterpret_cast<double*>(*buf + rb);
    sink.d_acc = acc;
    return VPCA_OK;
}

// Partition bookkeeping of the host-input scoring routes (commit / abort as for the Gram); `body` runs the chunk loop.
extern "C++" template <typename Body>
int score_on_lane(vpca_ctx* ctx, int64_t partition_id, int64_t nv, int64_t matched, const int32_t* model_rows, Body&& body) {
    std::unique_lock<std::mutex> direct;   // direct input adds into one accumulator, one call at a time, in call order
    if (partition_id < 0) direct = std::unique_lock<std::mutex>(ctx->direct_mu);
    CallScope sc{ctx, partition_id, nv};
    sc.matched = matched;
    int rc = sc.begin();
    if (rc != VPCA_OK) return rc;
    {
        LaneGuard lg(ctx);
        rc = lg.rc;
        if (rc == VPCA_OK) rc = prepare_slot(ctx, *lg.lane, sc);
        ChunkSink sink;
        if (rc == VPCA_OK)
            rc = score_sink(ctx, &lg.lane->d_scratch, &lg.lane->cap_scratch, lg.lane->stream, model_rows, nv,
                            reinterpret_cast<double*>(sc.target), sink);
        if (rc == VPCA_OK) rc = body(*lg.lane, sink);
    }
    return sc.end(rc);
}

int vpca_score_calls(vpca_ctx* ctx, int64_t partition_id, const int64_t* offsets, const int32_t* sample_idx, int64_t nv,
                     const int32_t* model_rows) {
    int64_t matched = 0;
    int rc = score_args(ctx, nv, model_rows, &matched);
    if (rc != VPCA_OK) return rc;
    if (offsets == nullptr || (nv > 0 && sample_idx == nullptr && offsets[nv] > offsets[0]))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_score_calls: bad argument");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    return score_on_lane(ctx, partition_id, nv, matched, model_rows, [&](vpca_ctx::Lane& L, ChunkSink& sink) {
        return process_calls(ctx, L, offsets, sample_idx, 4, nv, &sink, nullptr, 0);
    });
}

int vpca_score_bed(vpca_ctx* ctx, int64_t partition_id, const uint8_t* rows, int64_t nv, int64_t stride_bytes,
                   int32_t counted_allele, const int32_t* model_rows) {
    int64_t matched = 0;
    int rc = score_args(ctx, nv, model_rows, &matched);
    if (rc != VPCA_OK) return rc;
    if (counted_allele != 1 && counted_allele != 2)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_score_bed: counted_allele must be 1 (A1) or 2 (A2)");
    rc = packed_args(ctx, rows, nv, stride_bytes, counted_allele);
    if (rc != VPCA_OK) return rc;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    return score_on_lane(ctx, partition_id, nv, matched, model_rows, [&](vpca_ctx::Lane& L, ChunkSink& sink) {
        return packed_chunks(ctx, L, rows, nv, stride_bytes, counted_allele, sink);
    });
}

int vpca_score_panels(vpca_ctx* ctx, const void* d_x, int64_t nv, int64_t panel_variants, const int32_t* model_rows) {
    int64_t matched = 0;
    int rc = score_args(ctx, nv, model_rows, &matched);
    if (rc != VPCA_OK) return rc;
    std::lock_guard<std::mutex> dl(ctx->direct_mu);
    std::lock_guard<std::mutex> lk(ctx->mu);
    rc = panels_args(ctx, d_x, nv, panel_variants);
    if (rc != VPCA_OK) return rc;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (nv == 0) return VPCA_OK;
    ChunkSink sink;
    rc = score_sink(ctx, &ctx->d_scratch, &ctx->cap_scratch, ctx->stream, model_rows, nv, ctx->d_direct, sink);
    if (rc == VPCA_OK) rc = consume_chunk(ctx, ctx->plan, ctx->stream, ctx->ev_t0, ctx->ev_t1, sink, d_x, 0, nv, panel_variants);
    if (rc != VPCA_OK) return rc;
    ctx->total_variants += nv;
    ctx->st.variants_accumulated += nv;
    ctx->direct_matched += matched;
    return VPCA_OK;
}

int vpca_score_project(vpca_ctx* ctx, int32_t k, double* out, int64_t* matched_variants) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    if (!ctx->scoring) return fail(ctx, VPCA_ERR_UNSUPPORTED, "vpca_score_project needs a context made by vpca_create_scoring");
    std::lock_guard<std::mutex> dl(ctx->direct_mu);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (k < 1 || k > ctx->model_k) return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_score_project: k=%d outside [1, %d]", k, ctx->model_k);
    if (out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "out is NULL");
    for (auto& s : ctx->slots)
        if (s.used) return fail(ctx, VPCA_ERR_STATE, "partition %lld is neither committed nor aborted", (long long)s.pid);
    for (auto& L : ctx->lanes)
        if (L.busy) return fail(ctx, VPCA_ERR_STATE, "vpca_score_project while a scoring call is in flight");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const int m = ctx->n, K = ctx->model_k;
    const size_t ab = align256(ctx->slot_bytes());
    CUDA_OK(ctx, grow_buffer(&ctx->d_scratch, &ctx->cap_scratch, (int64_t)(ab + (size_t)m * k * sizeof(double))));
    double* d_sum = reinterpret_cast<double*>(ctx->d_scratch);
    double* d_y = reinterpret_cast<double*>(ctx->d_scratch + ab);
    // direct input first, then the committed partitions in ascending id
    CUDA_OK(ctx, cudaMemcpyAsync(d_sum, ctx->d_direct, ctx->slot_bytes(), cudaMemcpyDeviceToDevice, ctx->stream));
    int64_t cnt = ctx->direct_matched;
    for (auto& kv : ctx->scored) {
        CUDA_OK(ctx, model_add(d_sum, kv.second.d_acc, m, K, ctx->stream));
        cnt += kv.second.matched;
    }
    CUDA_OK(ctx, model_finish(d_sum, m, K, k, ctx->model_nfit, ctx->d_model_terms, d_y, ctx->stream));
    ctx->c_launches += (int64_t)ctx->scored.size() + 1;
    CUDA_OK(ctx, cudaMemcpyAsync(out, d_y, (size_t)m * k * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (int64_t)m * k * 8;
    if (matched_variants != nullptr) *matched_variants = cnt;
    return VPCA_OK;
}

int vpca_debug_projection_tiles(int32_t n_fit, int32_t n_total, int32_t cta_group, int32_t mxf4, int32_t* out,
                                int32_t max_tiles) {
    if (n_fit < 1 || n_total < n_fit || max_tiles < 0 || (out == nullptr && max_tiles > 0))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_debug_projection_tiles: bad argument");
    return gram_debug_projection_tiles(n_fit, n_total, cta_group, mxf4 != 0, out, max_tiles);
}

int vpca_get_centered(vpca_ctx* ctx, double* out) {
    if (ctx == nullptr || out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "call vpca_finalize_gram first");
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "this context stores a row band of the Gram");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    int rc = run_center(ctx, true);   // the eigensolve overwrites C, so recompute it
    if (rc != VPCA_OK) return rc;
    const size_t bytes = (size_t)ctx->n * ctx->n * sizeof(double);
    CUDA_OK(ctx, cudaMemcpyAsync(out, ctx->eig.d_C, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->c_d2h += (int64_t)bytes;
    ctx->pca_done = false;
    return VPCA_OK;
}

int vpca_get_tridiagonal(vpca_ctx* ctx, double* diag, double* offdiag) {
    if (ctx == nullptr || diag == nullptr || offdiag == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->pca_done) return fail(ctx, VPCA_ERR_STATE, "call vpca_compute_pca first");
    if (ctx->eig.last_method == 2)
        return fail(ctx, VPCA_ERR_STATE, "the last solve used Lanczos and did not tridiagonalise C (set VPCA_EIG=direct)");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaMemcpyAsync(diag, ctx->eig.d_diag, (size_t)ctx->n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaMemcpyAsync(offdiag, ctx->eig.d_off, (size_t)(ctx->n - 1) * 8, cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return VPCA_OK;
}

int vpca_synth_dense_device(vpca_ctx* ctx, uint64_t seed, int64_t v0, int64_t nv, int mode, void* d_x, int64_t ld) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (d_x == nullptr || nv < 0 || ld < nv || v0 < 0 || (mode != 0 && mode != 1))
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_synth_dense_device: bad argument");
    if (mode == 1 && ctx->max_mult < 2)
        return fail(ctx, VPCA_ERR_BAD_ARG, "dosage mode needs max_multiplicity >= 2");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    cudaError_t e = synth_dense(seed, ctx->rows(), v0, nv, mode, ctx->elem_bits, d_x, ld, 0, ctx->stream);
    if (e != cudaSuccess) return fail(ctx, VPCA_ERR_CUDA, "synthetic generator: %s", cudaGetErrorString(e));
    ctx->c_launches += 2 * ((nv + (1 << 22) - 1) >> 22);
    return VPCA_OK;
}

int vpca_get_stats(vpca_ctx* ctx, vpca_stats* out) {
    if (ctx == nullptr || out == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    if (ctx->gram_timed && cudaEventSynchronize(ctx->ev_t1) == cudaSuccess) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev_t0, ctx->ev_t1) == cudaSuccess) ctx->st.last_gram_ms = ms;
    } else if (!ctx->gram_timed) {
        ctx->st.last_gram_ms = ctx->lane_gram_ms.load();
    }
    if (ctx->eig_timed && cudaEventSynchronize(ctx->ev_e1) == cudaSuccess) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, ctx->ev_e0, ctx->ev_e1) == cudaSuccess) ctx->st.last_eig_ms = ms;
    }
    ctx->st.gram_launches = ctx->c_gram.load();
    ctx->st.kernel_launches = ctx->c_launches.load();
    ctx->st.h2d_bytes = ctx->c_h2d.load();
    ctx->st.d2h_bytes = ctx->c_d2h.load();
    *out = ctx->st;
    return VPCA_OK;
}

int vpca_gram_export_ipc(vpca_ctx* ctx, void* handle64) {
    if (ctx == nullptr || handle64 == nullptr) return fail(ctx, VPCA_ERR_BAD_ARG, "NULL argument");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->n_proj > 0) return fail(ctx, VPCA_ERR_UNSUPPORTED, "projecting contexts reduce through vpca_gram_device_ptr");
    if (!ctx->own_S) return fail(ctx, VPCA_ERR_STATE, "the peer-reduce mode needs a library-owned Gram (vpca_config.d_gram == NULL)");
    if (ctx->band_rows != ctx->n) return fail(ctx, VPCA_ERR_STATE, "band-only Grams are shared with vpca_gram_set_peers_local");
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    cudaIpcMemHandle_t h;
    CUDA_OK(ctx, cudaIpcGetMemHandle(&h, ctx->d_S));
    memcpy(handle64, &h, sizeof(h));
    return VPCA_OK;
}

int vpca_gram_set_peers(vpca_ctx* ctx, const void* handles, int32_t world, int32_t rank) {
    if (ctx == nullptr || handles == nullptr || world < 1 || world > 16 || rank < 0 || rank >= world)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_gram_set_peers: bad argument (world <= 16)");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->n_proj > 0) return fail(ctx, VPCA_ERR_UNSUPPORTED, "projecting contexts reduce through vpca_gram_device_ptr");
    if (!ctx->own_S) return fail(ctx, VPCA_ERR_STATE, "the peer-reduce mode needs a library-owned Gram");
    if (ctx->plan.num_peers != 0) return fail(ctx, VPCA_ERR_STATE, "peers already set");
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    const size_t nn = (size_t)ctx->n * ctx->n;
    for (int d = 0; d < world; ++d) {
        int32_t* base = ctx->d_S;
        if (d != rank) {
            cudaIpcMemHandle_t h;
            memcpy(&h, static_cast<const char*>(handles) + (size_t)d * sizeof(h), sizeof(h));
            void* ptr = nullptr;
            cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
            if (e != cudaSuccess) {
                for (int q = 0; q < d; ++q)
                    if (q != rank) cudaIpcCloseMemHandle(ctx->plan.peer_base[q]);
                return fail(ctx, VPCA_ERR_NCCL, "cudaIpcOpenMemHandle(rank %d) failed: %s", d, cudaGetErrorString(e));
            }
            base = static_cast<int32_t*>(ptr);
        }
        ctx->plan.peer_base[d] = base;
        ctx->plan.peer_S[d] = base;
        ctx->plan.peer_flags[d] = base + nn;
    }
    CUDA_OK(ctx, gram_preload_kernels(ctx->stream));   // nothing is loaded lazily behind a spinning barrier
    CUDA_OK(ctx, encode_preload_kernels());
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->plan.peers_ipc = true;
    ctx->plan.peer_rank = rank;
    ctx->plan.num_peers = world;
    sync_peers_to_lanes(ctx);
    return VPCA_OK;
}

// Same-process form of vpca_gram_set_peers: the caller owns all `world` contexts (one JVM driving the GPUs of the box,
// SURVEY 8b "process model"), so the Gram buffers are shared by enabling peer access between the devices instead of
// through IPC handles.  Contexts may also sit on the same device (tests on a 1-GPU box).
int vpca_gram_set_peers_local(vpca_ctx* const* ctxs, int32_t world) {
    if (ctxs == nullptr || world < 1 || world > 16) return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_gram_set_peers_local: world must be in [1, 16]");
    for (int r = 0; r < world; ++r) {
        if (ctxs[r] == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctxs[%d] is NULL", r);
        REFUSE_ON_SCORING(ctxs[r]);
        if (ctxs[r]->n_proj > 0)
            return fail(ctxs[r], VPCA_ERR_UNSUPPORTED, "projecting contexts reduce through vpca_gram_device_ptr");
        if (!ctxs[r]->own_S) return fail(ctxs[r], VPCA_ERR_STATE, "the peer-reduce mode needs a library-owned Gram");
        if (ctxs[r]->n != ctxs[0]->n) return fail(ctxs[r], VPCA_ERR_BAD_ARG, "all contexts must have the same n_samples");
        if (ctxs[r]->plan.num_peers != 0) return fail(ctxs[r], VPCA_ERR_STATE, "peers already set");
        for (int q = 0; q < r; ++q)
            if (ctxs[q] == ctxs[r]) return fail(ctxs[r], VPCA_ERR_BAD_ARG, "ctxs[%d] and ctxs[%d] are the same context", q, r);
    }
    for (int r = 0; r < world; ++r) {
        vpca_ctx* c = ctxs[r];
        CUDA_OK(c, cudaSetDevice(c->cfg.device));
        for (int d = 0; d < world; ++d) {
            const int od = ctxs[d]->cfg.device;
            if (od == c->cfg.device) continue;
            int can = 0;
            CUDA_OK(c, cudaDeviceCanAccessPeer(&can, c->cfg.device, od));
            if (!can) return fail(c, VPCA_ERR_NCCL, "device %d cannot access device %d (no NVLink / PCIe peer path)", c->cfg.device, od);
            cudaError_t e = cudaDeviceEnablePeerAccess(od, 0);
            if (e == cudaErrorPeerAccessAlreadyEnabled) {
                cudaGetLastError();
            } else if (e != cudaSuccess) {
                return fail(c, VPCA_ERR_NCCL, "cudaDeviceEnablePeerAccess(%d -> %d): %s", c->cfg.device, od, cudaGetErrorString(e));
            }
        }
    }
    // one host thread will enqueue barriers for several contexts: no kernel may be loaded lazily behind a spinning one
    for (int r = 0; r < world; ++r) {
        vpca_ctx* c = ctxs[r];
        CUDA_OK(c, cudaSetDevice(c->cfg.device));
        CUDA_OK(c, gram_preload_kernels(c->stream));
        CUDA_OK(c, encode_preload_kernels());
        CUDA_OK(c, cudaStreamSynchronize(c->stream));
    }
    for (int r = 0; r < world; ++r) {
        vpca_ctx* c = ctxs[r];
        std::lock_guard<std::mutex> lk(c->mu);
        for (int d = 0; d < world; ++d) {
            vpca_ctx* o = ctxs[d];
            // a band-only Gram is addressed through the virtual origin of the full matrix: row r of rank d lives at
            // base + (r - band_row0) * n, so (base - band_row0 * n) + r * n is valid for every row the rank owns
            c->plan.peer_base[d] = o->d_S;
            c->plan.peer_S[d] = o->d_S - (ptrdiff_t)o->band_row0 * o->n;
            c->plan.peer_flags[d] = o->d_S + (size_t)o->band_rows * o->n;
            c->plan.band_row0[d] = o->band_row0;
            c->plan.band_rows[d] = o->band_rows;
        }
        c->plan.peers_ipc = false;
        c->plan.peer_rank = r;
        c->plan.num_peers = world;
        sync_peers_to_lanes(c);
    }
    return VPCA_OK;
}

int vpca_gram_set_peer_mode(vpca_ctx* ctx, int32_t mode) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (mode != VPCA_PEER_REPLICATE && mode != VPCA_PEER_OWNER_ROWS)
        return fail(ctx, VPCA_ERR_BAD_ARG, "vpca_gram_set_peer_mode: unknown mode %d", mode);
    if (ctx->plan.num_peers < 1) return fail(ctx, VPCA_ERR_STATE, "call vpca_gram_set_peers first");
    const int world = ctx->plan.num_peers, n = ctx->n;
    if (mode == VPCA_PEER_OWNER_ROWS) {
        if (n < 64 * world)
            return fail(ctx, VPCA_ERR_UNSUPPORTED, "owner-rows mode needs n_samples >= 64 x world (%d < %d)", n, 64 * world);
        int ends[16];
        vpca_owner_row_bands(n, world, ends);
        for (int q = 0; q < 16; ++q) ctx->plan.own_end[q] = q < world ? ends[q] : n;
        // band-only Grams must hold exactly the rows their rank owns
        for (int q = 0; q < world; ++q) {
            const int lo = q == 0 ? 0 : ends[q - 1];
            if (ctx->plan.band_rows[q] != 0 && ctx->plan.band_rows[q] != n &&
                (ctx->plan.band_row0[q] != lo || ctx->plan.band_rows[q] != ends[q] - lo))
                return fail(ctx, VPCA_ERR_BAD_ARG, "rank %d stores rows [%d, %d) but owns [%d, %d) (see vpca_owner_row_bands)", q,
                            ctx->plan.band_row0[q], ctx->plan.band_row0[q] + ctx->plan.band_rows[q], lo, ends[q]);
        }
    } else if (ctx->band_rows != n) {
        return fail(ctx, VPCA_ERR_BAD_ARG, "a band-only Gram supports VPCA_PEER_OWNER_ROWS only");
    }
    ctx->plan.peer_mode = mode;
    sync_peers_to_lanes(ctx);
    return VPCA_OK;
}

int vpca_owner_row_bands(int32_t n_samples, int32_t world, int32_t* row_end) {
    if (row_end == nullptr || world < 1 || world > 16 || n_samples < 64 * world)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_owner_row_bands: need 1 <= world <= 16 and n_samples >= 64 x world");
    // equal shares of the lower triangle: rows [0, R) hold R^2 / 2 cells -> R_q = n sqrt(q / world), on multiples of 32
    const int n = n_samples;
    int prev = 0;
    for (int q = 0; q < world; ++q) {
        int end = (q + 1 == world) ? n : (int)(std::sqrt((double)(q + 1) / world) * n / 32.0 + 0.5) * 32;
        end = std::max(end, prev + 32);
        if (q + 1 < world) end = std::min(end, n - 32 * (world - 1 - q));
        row_end[q] = end;
        prev = end;
    }
    return VPCA_OK;
}

int vpca_gram_gather(vpca_ctx* ctx) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->finalized) return fail(ctx, VPCA_ERR_STATE, "Gram already finalized");
    if (ctx->plan.num_peers < 2) return VPCA_OK;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, gram_peer_barrier(ctx->plan, ctx->stream));          // every rank's contributions have landed
    ctx->c_launches += 1;
    if (ctx->plan.peer_mode == 1 && ctx->band_rows == ctx->n) {
        CUDA_OK(ctx, gram_gather_rows(ctx->plan, ctx->d_S, ctx->n, ctx->stream));
        CUDA_OK(ctx, gram_peer_barrier(ctx->plan, ctx->stream));      // nobody resets a Gram a peer is still reading
        ctx->c_launches += 2;
    }
    return VPCA_OK;
}

int vpca_peer_barrier(vpca_ctx* ctx) {
    if (ctx == nullptr) return fail(nullptr, VPCA_ERR_BAD_ARG, "ctx is NULL");
    REFUSE_ON_SCORING(ctx);
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (ctx->plan.num_peers < 2) return VPCA_OK;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, gram_peer_barrier(ctx->plan, ctx->stream));
    ctx->c_launches += 1;
    return VPCA_OK;
}

int vpca_debug_gram_profile(vpca_ctx* ctx, int64_t* out, int32_t max_ctas) {
    if (ctx == nullptr || out == nullptr || max_ctas <= 0) return fail(ctx, VPCA_ERR_BAD_ARG, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    return gram_read_profile(ctx->plan, reinterpret_cast<long long*>(out), max_ctas);
}

int vpca_debug_lanczos_profile(vpca_ctx* ctx, int64_t* out, int32_t max_steps) {
    if (ctx == nullptr || out == nullptr || max_steps <= 0) return fail(ctx, VPCA_ERR_BAD_ARG, "bad argument");
    std::lock_guard<std::mutex> lk(ctx->mu);
    if (!ctx->eig_ready || ctx->eig.d_lzprof == nullptr) return 0;
    CUDA_OK(ctx, cudaSetDevice(ctx->cfg.device));
    CUDA_OK(ctx, cudaStreamSynchronize(ctx->stream));
    const int steps = std::min(max_steps, 32);
    CUDA_OK(ctx, cudaMemcpy(out, ctx->eig.d_lzprof, (size_t)steps * 8 * sizeof(long long), cudaMemcpyDeviceToHost));
    return steps;
}

int vpca_debug_band_tiles(int32_t n_samples, int32_t cta_group, int32_t row0, int32_t rows, int32_t* out, int32_t max_tiles) {
    if (n_samples < 2 || max_tiles < 0 || row0 < 0 || rows < 1 || row0 + rows > n_samples)
        return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_debug_band_tiles: bad argument");
    return gram_debug_band_tiles(n_samples, cta_group, row0, row0 + rows, out, max_tiles);
}

int vpca_debug_max_clusters(int32_t device, int32_t cluster_size) {
    if (cluster_size < 1 || cluster_size > 16) return fail(nullptr, VPCA_ERR_BAD_ARG, "cluster_size must be in [1, 16]");
    if (cudaSetDevice(device) != cudaSuccess) return fail(nullptr, VPCA_ERR_CUDA, "cudaSetDevice(%d) failed", device);
    const int c = gram_debug_max_clusters(cluster_size);
    if (c < 0) return fail(nullptr, VPCA_ERR_CUDA, "cudaOccupancyMaxActiveClusters failed for cluster size %d", cluster_size);
    return c;
}

int vpca_debug_tiles(int32_t n_samples, int32_t cta_group, int32_t exact, int32_t* out, int32_t max_tiles) {
    if (n_samples < 2 || max_tiles < 0) return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_debug_tiles: bad argument");
    return gram_debug_tiles(n_samples, cta_group, exact, out, max_tiles);
}

int vpca_debug_plan(const int32_t* tiles, int32_t num_tiles, int32_t workers, int32_t kb_window, int32_t* out, int32_t max_pieces) {
    if (tiles == nullptr || num_tiles < 1 || workers < 1 || kb_window < 1 || (out == nullptr && max_pieces > 0))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_debug_plan: bad argument");
    const int rc = gram_debug_plan(tiles, num_tiles, workers, kb_window, out, max_pieces);
    if (rc < 0) return fail(nullptr, VPCA_ERR_STATE, "vpca_debug_plan: the accumulators of a worker do not fit TMEM (large-N schedule)");
    return rc;
}

int vpca_debug_rebalance(const int32_t* tiles, int32_t num_tiles, int32_t workers, int32_t kb_window, int32_t col_limit,
                         double* cum, int32_t* out, int32_t max_pieces) {
    if (tiles == nullptr || num_tiles < 1 || workers < 1 || kb_window < 1 || cum == nullptr || col_limit < 32 ||
        (out == nullptr && max_pieces > 0))
        return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_debug_rebalance: bad argument");
    const int rc = gram_debug_repair(tiles, num_tiles, workers, kb_window, col_limit, cum, out, max_pieces);
    if (rc < 0) return fail(nullptr, VPCA_ERR_STATE, "vpca_debug_rebalance: no feasible repair of this split");
    return rc;
}

/* Pinned host memory for callers that stage rows themselves (JNI direct ByteBuffers): the H2D copies of accumulate_*
 * then run at full PCIe rate and truly asynchronously.  Portable across devices. */
int vpca_host_alloc(size_t bytes, void** out) {
    if (out == nullptr || bytes == 0) return fail(nullptr, VPCA_ERR_BAD_ARG, "vpca_host_alloc: bad argument");
    cudaError_t e = cudaHostAlloc(out, bytes, cudaHostAllocPortable);
    if (e != cudaSuccess) {
        *out = nullptr;
        return fail(nullptr, VPCA_ERR_NOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
    }
    return VPCA_OK;
}

int vpca_host_free(void* p) {
    if (p == nullptr) return VPCA_OK;
    cudaError_t e = cudaFreeHost(p);
    if (e != cudaSuccess) return fail(nullptr, VPCA_ERR_CUDA, "cudaFreeHost: %s", cudaGetErrorString(e));
    return VPCA_OK;
}

}  // extern "C"
