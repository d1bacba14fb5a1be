// csrc/api.cu -- libobboot C ABI (include/obboot.h): context, packed design, bootstrap driver.
//
// Takes over OaxacaBuilder::run() from the group split to the assembled results
// (builder.rs:808-950).  Host code only orchestrates: every number is produced by the CUDA kernels
// in this directory; there is no CPU compute path.
#include "internal.h"

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstring>
#include <exception>
#include <memory>
#include <atomic>
#include <mutex>
#include <optional>
#include <set>
#include <type_traits>

using namespace ob;

// K + T <= 280: two 32-row stages of a design row block (plus the count and A tiles) must fit the Gram CTA's 227 KB
static constexpr int MAX_DESIGN_COLS = 280;

struct ob_ctx {
    int device = 0;
    int num_sms = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream_side = nullptr;  // point-estimate residuals + their D2H, overlapped with the gather / reduction
    cudaStream_t stream_copy = nullptr;  // ob_design_pack_async: chunked column uploads + pack, under the bootstrap's first kernels
    // page-locked landing slots for the deferred flags of asynchronous packs, allocated once per context: pinning and
    // unpinning host memory per call (cudaHostAlloc / cudaFreeHost) costs milliseconds to hundreds of milliseconds
    static constexpr int PACK_SLOTS = 8;
    int* h_pack_flags = nullptr;         // [PACK_SLOTS][4]
    ob_design* pack_slot_owner[PACK_SLOTS] = {};
    unsigned pack_seq = 0;
    cudaMemPool_t pool = nullptr;   // stream-ordered workspace pool: freed blocks stay cached between calls
    cudaMemPool_t pool_pack = nullptr;   // separate pool for the pack's column staging, so its many small blocks do
                                         // not fragment the bootstrap workspace (20 GB count buffer at n = 1e7)
    cudaMemPool_t pool_design = nullptr; // packed designs (outlive a call): their own pool, so re-packing reuses the blocks
    std::unique_ptr<Comm> comm;          // row-sharding collectives (mode N); null = single GPU
    std::string err;
    // designs created on this context and still alive.  ob_ctx_destroy releases their device memory (it dies with the
    // context's pools anyway) and orphans them, so that an ob_design_destroy arriving late -- a garbage collector
    // finalising objects in arbitrary order, possibly on another thread -- only frees the host struct.
    std::mutex designs_mu;
    std::set<ob_design*> designs;
    std::set<ob_gram_cache*> caches;     // Gram caches of this context, orphaned the same way (under designs_mu)
};

struct ob_local_group { LocalGroup* g = nullptr; int world = 0; };

struct PendingPack;   // an upload + pack still in flight on the copy stream (ob_design_pack_async)

struct ob_design {
    PendingPack* pending = nullptr;
    ob_status failed = OB_OK;        // a deferred pack error (negative weight, bad code): the design is unusable
    std::string fail_msg;
    ob_ctx* owner = nullptr;         // context that created the design; null once that context has been destroyed
    cudaStream_t stream = nullptr;   // owning context's stream: buffers come from its pack pool and are freed on it
    int device = 0;
    int K = 0, n_cont = 0, V = 0, ldx = 0;
    int T = 1;                       // outcome columns K .. K+T-1 of a design row (ob_design_apply_rif_multi: one per quantile)
    int K1 = 0;                      // selection-equation columns incl. the intercept (ob_design_attach_selection), 0 = none
    std::vector<int> cat_levels;     // level counts of the categorical predictors (empty: unknown, ob_design_from_dense): the
                                     // products of two dummies of one predictor are structural zeros of X'WX (gram_columns)
    bool weighted = false;
    int64_t n_frame = 0;             // rows of the frame the design was packed from (ob_design_update_outcome)
    int world = 1, rank = 0;         // row sharding (mode N): this design holds rank's rows of a world-way split
    double ms_h2d = 0.0, ms_pack = 0.0;   // device time of the column upload and of the pack kernels (ob_design_pack)
    GroupData g[2];
    // clusters (ob_design_attach_clusters): ob_cluster_strata and the resampling units of each stratum (JOINT: both = M);
    // the unit of every packed row is GroupData::uid
    int cl_strata = OB_CLUSTER_NONE;
    int64_t cl_units[2] = {0, 0};
    // identity for ob_gram_cache keys: a process-wide unique id (addresses are reused after destroy), the generation of
    // the design columns / weights / rows / row-shard marking, and the generation of the outcome columns
    uint64_t id = 0, x_gen = 0, y_gen = 0;
};

// ob_bootstrap_run_cached: the reduced Gram cells of every slot of a run, kept in HBM for the next run on the same
// resamples (layouts: gram_cache_map in gram.cu)
struct ob_gram_cache {
    ob_ctx* owner = nullptr;         // context that created the cache; null once that context has been destroyed
    int device = 0;
    int last_use = OB_CACHE_NONE;
    double* xx = nullptr; size_t xx_bytes = 0;   // [2][slots][K(K+1)/2]
    double* yy = nullptr; size_t yy_bytes = 0;   // [2][slots][K T + 1]
    long long* rows = nullptr; size_t rows_bytes = 0;   // clustered designs: [2][slots] group row counts (a SOLVE_ONLY run draws none)
    double* esum = nullptr; size_t esum_bytes = 0;      // Bayesian bootstrap: [2][slots] sums of the raw weights per slot
    // key of xx (valid while xx_ok): what decides the resamples and the design's X'WX
    bool xx_ok = false;
    uint64_t design_id = 0, x_gen = 0, seed = 0;
    int64_t reps = 0, rep_begin = 0, rep_end = 0, slots = 0;
    int shard_reps = 0, rep_world = 1, rep_rank = 0, row_world = 1, row_rank = 0, K = 0;
    int count_bytes = 1;             // multiplicity width the fill ended with (a saturation already known)
    bool bayes = false;              // resampling scheme of the fill: Bayesian (Dirichlet) weights or multinomial counts
    // key of yy (valid while y_ok): the design's outcome generation and outcome count
    bool y_ok = false;
    uint64_t y_gen = 0; int T = 0;
};

namespace {

// RAII workspace allocation from the context's stream-ordered pool (cudaMallocFromPoolAsync): the
// multi-GB multiplicity / partial buffers are reused across calls instead of paying cudaMalloc/cudaFree
// (hundreds of ms at n = 1e7) every bootstrap.
thread_local ob_ctx* g_alloc_ctx = nullptr;
thread_local bool g_alloc_pack = false;

struct DevBuf {
    void* p = nullptr; size_t bytes = 0;
    ob_ctx* ctx = nullptr;
    bool pack = false;
    DevBuf() : ctx(g_alloc_ctx), pack(g_alloc_pack) {}
    explicit DevBuf(size_t b) : ctx(g_alloc_ctx), pack(g_alloc_pack) { alloc(b); }
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    DevBuf(DevBuf&& o) noexcept : p(o.p), bytes(o.bytes), ctx(o.ctx), pack(o.pack) { o.p = nullptr; o.bytes = 0; }
    ~DevBuf() { release(); }
    void release() {
        if (p) { cudaFreeAsync(p, ctx->stream); p = nullptr; }
        bytes = 0;
    }
    void alloc(size_t b) {
        release();
        bytes = b;
        if (b) OB_CUDA(cudaMallocFromPoolAsync(&p, b, pack ? ctx->pool_pack : ctx->pool, ctx->stream));
    }
    template <typename T> T* as() const { return static_cast<T*>(p); }
};

// the cleaned, coded frame staged in HBM (input of the pack kernels)
struct StagedFrame {
    int64_t n = 0; int n_cont = 0, n_cat = 0;
    std::vector<DevBuf> cols, cats;     // [n] f64 / int32 level codes
    DevBuf y, w, grp;                   // outcome, weights (optional), group byte
    bool weighted = false;
    double ms_h2d = 0.0;
};

}  // namespace

// ob_design_pack_async: the frame is uploaded and packed in row chunks on the context's copy stream while the caller
// goes on (typically straight into ob_bootstrap_run, whose replicate generation needs no design rows at all and whose
// Gram contraction starts on the leaves that have arrived).  Everything the in-flight work touches lives here.
struct PendingPack {
    StagedFrame sf;
    DevBuf d_bc, d_tot, d_flags, d_cont_ptrs, d_cat_ptrs, d_levels, d_dstart;
    std::vector<cudaEvent_t> chunk_done;     // recorded on the copy stream after chunk c's rows are packed
    int64_t ready_lo[2] = {0, 0};            // design rows [ready_lo[g], rows_ready[g][c]) of group g are final once chunk c is done
    std::vector<int64_t> rows_ready[2];
    // row-shard packs (ob_design_pack_row_shard_async): the slice's rows that belong to other ranks wait in export buffers
    // for ONE exchange over the communicator (after the last chunk, on the context's stream, a collective)
    bool exchange_pending = false;
    DevBuf EX[2], Ew[2], Esrc[2];
    std::vector<size_t> ex_rows[2], ex_send_row[2], ex_recv_row[2];   // rows[src * world + dst]; offsets in rows
    std::vector<long long> ex_frame_off;
    cudaEvent_t ev_begin = nullptr, ev_h2d_end = nullptr;   // timing: first upload .. last pack kernel
    int* h_flags = nullptr;                  // pinned [4] (a slot of the context's): pack flags, valid after the last chunk
    int slot = -1;
    ~PendingPack() {
        for (cudaEvent_t e : chunk_done) cudaEventDestroy(e);
        if (ev_begin) cudaEventDestroy(ev_begin);
        if (ev_h2d_end) cudaEventDestroy(ev_h2d_end);
    }
};

namespace {

// bytes the pool holds but is not using: available to the next call in addition to cudaMemGetInfo's free
size_t pool_idle_bytes(ob_ctx* ctx) {
    unsigned long long reserved = 0, used = 0;
    cudaMemPoolGetAttribute(ctx->pool, cudaMemPoolAttrReservedMemCurrent, &reserved);
    cudaMemPoolGetAttribute(ctx->pool, cudaMemPoolAttrUsedMemCurrent, &used);
    return reserved > used ? (size_t)(reserved - used) : 0;
}

struct Timer {
    cudaEvent_t a, b; cudaStream_t st; double* acc;
    Timer(cudaStream_t s, double* accum) : st(s), acc(accum) {
        cudaEventCreate(&a); cudaEventCreate(&b); cudaEventRecord(a, st);
    }
    void stop() { cudaEventRecord(b, st); }
    void collect() { float ms = 0; cudaEventSynchronize(b); cudaEventElapsedTime(&ms, a, b); *acc += ms; }
    ~Timer() { cudaEventDestroy(a); cudaEventDestroy(b); }
};

// OBBOOT_TRACE=1: host wall-clock marks of ob_bootstrap_run's phases on stderr (diagnosing per-call fixed costs)
struct Trace {
    bool on; std::chrono::steady_clock::time_point t0, last;
    Trace() : on(getenv("OBBOOT_TRACE") != nullptr), t0(std::chrono::steady_clock::now()), last(t0) {}
    void mark(const char* what, cudaStream_t st = nullptr, bool sync = false) {
        if (!on) return;
        if (sync) cudaStreamSynchronize(st);
        const auto now = std::chrono::steady_clock::now();
        fprintf(stderr, "[obboot] %-28s +%8.3f ms  (t = %9.3f ms)\n", what,
                std::chrono::duration<double, std::milli>(now - last).count(),
                std::chrono::duration<double, std::milli>(now - t0).count());
        last = now;
    }
};

template <typename F>
ob_status guarded(ob_ctx* ctx, F&& f) {
    try {
        if (ctx) OB_CUDA(cudaSetDevice(ctx->device));
        g_alloc_ctx = ctx;
        g_alloc_pack = false;
        f();
        return OB_OK;
    } catch (const CudaError& e) {
        if (ctx) {
            char buf[512];
            snprintf(buf, sizeof buf, "CUDA error: %s (%s) at %s:%d", cudaGetErrorString(e.code), e.what, e.file, e.line);
            ctx->err = buf;
        }
        cudaGetLastError();
        return (e.code == cudaErrorNoDevice || e.code == cudaErrorInsufficientDriver) ? OB_ERR_NO_DEVICE : OB_ERR_CUDA;
    } catch (const StatusError& e) {
        if (ctx) ctx->err = e.msg;
        return e.code;
    } catch (const std::bad_alloc&) {
        if (ctx) ctx->err = "host allocation failed";
        return OB_ERR_INVALID_ARG;
    }
}

[[noreturn]] void fail(ob_status c, const std::string& m) { throw StatusError{c, m}; }

// zero-fill on the context's (non-blocking) stream: a legacy-default-stream cudaMemset would not be ordered
// before the copies / pack kernels that follow on that stream
// Design buffers come from the context's pack pool (stream-ordered): re-packing the same shapes reuses the
// blocks instead of paying multi-GB cudaMalloc/cudaFree (random 100s-of-ms stalls) on every call.
// zero_all = false: the caller's pack kernel writes every column of every valid row (pad columns included), so only
// the pad rows [n, n_pad) are cleared -- no multi-GB memset in front of the pack
void alloc_group(ob_ctx* ctx, GroupData& g, int64_t n, int ldx, bool weighted, bool zero_all = true) {
    cudaStream_t st = ctx->stream;
    g.n = n; g.n_pad = pad_rows(n);
    g.shard = row_shard(n, 0, 1);
    const size_t xbytes = sizeof(double) * (size_t)g.n_pad * ldx;
    const size_t tail_off = zero_all ? 0 : sizeof(double) * (size_t)n * ldx;
    OB_CUDA(cudaMallocFromPoolAsync((void**)&g.X, xbytes, ctx->pool_design, st));
    OB_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(g.X) + tail_off, 0, xbytes - tail_off, st));
    if (weighted) {
        OB_CUDA(cudaMallocFromPoolAsync((void**)&g.w, sizeof(double) * (size_t)g.n_pad, ctx->pool_design, st));
        OB_CUDA(cudaMemsetAsync(g.w, 0, sizeof(double) * (size_t)g.n_pad, st));
        OB_CUDA(cudaMallocFromPoolAsync((void**)&g.Xs, xbytes, ctx->pool_design, st));
        OB_CUDA(cudaMemsetAsync(reinterpret_cast<char*>(g.Xs) + tail_off, 0, xbytes - tail_off, st));   // pad rows stay zero
    }
    OB_CUDA(cudaMallocFromPoolAsync((void**)&g.src, sizeof(uint32_t) * (size_t)g.n_pad, ctx->pool_design, st));
}

void design_register(ob_ctx* ctx, ob_design* d) {
    static std::atomic<uint64_t> next_id{0};
    d->id = ++next_id;
    d->owner = ctx;
    std::lock_guard<std::mutex> lk(ctx->designs_mu);
    ctx->designs.insert(d);
}

void design_release_device(ob_design* d) {
    cudaStream_t st = d->stream;
    for (auto& g : d->g) {
        if (g.X) cudaFreeAsync(g.X, st);
        if (g.w) cudaFreeAsync(g.w, st);
        if (g.Xs) cudaFreeAsync(g.Xs, st);
        if (g.src) cudaFreeAsync(g.src, st);
        if (g.y_raw) cudaFreeAsync(g.y_raw, st);
        if (g.hk_Z) cudaFreeAsync(g.hk_Z, st);
        if (g.hk_sel) cudaFreeAsync(g.hk_sel, st);
        if (g.hk_Xm) cudaFreeAsync(g.hk_Xm, st);
        if (g.uid) cudaFreeAsync(g.uid, st);
        g.X = g.w = g.Xs = g.y_raw = g.hk_Z = g.hk_Xm = nullptr; g.src = g.uid = nullptr; g.hk_sel = nullptr;
    }
}

// empties a Gram cache (its device memory goes back to the owner's design pool)
void cache_release_device(ob_gram_cache* c) {
    if (c->owner) {
        cudaStream_t st = c->owner->stream;
        if (c->xx) cudaFreeAsync(c->xx, st);
        if (c->yy) cudaFreeAsync(c->yy, st);
        if (c->rows) cudaFreeAsync(c->rows, st);
        if (c->esum) cudaFreeAsync(c->esum, st);
    }
    c->xx = c->yy = nullptr; c->rows = nullptr; c->esum = nullptr; c->xx_bytes = c->yy_bytes = c->rows_bytes = c->esum_bytes = 0;
    c->xx_ok = c->y_ok = false;
}

// The one exchange of an asynchronous row-shard pack: every rank sends the rows of its slice that other ranks own (they
// sit in its export buffers) and receives its own from the slices of others, straight into place; then scales what it
// imported.  Enqueued on the context's stream after the last chunk; a collective (all ranks, same order).
void pending_exchange(ob_design* d) {
    PendingPack* P = d->pending;
    if (!P || !P->exchange_pending) return;
    ob_ctx* ctx = d->owner;
    Comm* comm = ctx->comm.get();
    if (!comm) fail(OB_ERR_NCCL, "the communicator of an asynchronous row-shard pack was destroyed before its exchange");
    cudaStream_t st = ctx->stream;
    const int world = comm->world, me = comm->rank;
    OB_CUDA(cudaStreamWaitEvent(st, P->chunk_done.back(), 0));
    for (int g = 0; g < 2; ++g) {
        GroupData& G = d->g[g];
        auto exchange = [&](const void* sendbuf, void* recvbuf, size_t row_bytes) {
            std::vector<size_t> b(P->ex_rows[g].size()), so((size_t)world), ro((size_t)world);
            for (size_t i = 0; i < b.size(); ++i) b[i] = P->ex_rows[g][i] * row_bytes;
            for (int r = 0; r < world; ++r) { so[r] = P->ex_send_row[g][r] * row_bytes; ro[r] = P->ex_recv_row[g][r] * row_bytes; }
            comm->alltoallv(sendbuf, so.data(), recvbuf, ro.data(), b.data(), st);
        };
        exchange(P->EX[g].p, G.X, sizeof(double) * (size_t)d->ldx);
        if (d->weighted) exchange(P->Ew[g].p, G.w, sizeof(double));
        exchange(P->Esrc[g].p, G.src, sizeof(uint32_t));
        for (int r = 0; r < world; ++r) {
            const int64_t rows = (int64_t)P->ex_rows[g][(size_t)r * world + me];
            if (!rows) continue;
            scale_rows_range_launch(G, d->ldx, (int64_t)P->ex_recv_row[g][r], rows, st);
        }
    }
    OB_CUDA(cudaStreamSynchronize(st));      // the byte tables of the exchange live on this stack frame
    P->exchange_pending = false;
}

// Completes an asynchronous pack: waits for the copy stream, releases the staging buffers (on the context's stream,
// ordered after the last pack kernel), collects timings and the deferred error flags.  quiet: never throws (destroy).
void pending_finish(ob_design* d, bool quiet = false) {
    PendingPack* P = d->pending;
    if (!P) return;
    ob_ctx* ctx = d->owner;
    if (P->exchange_pending && ctx && !quiet) pending_exchange(d);   // (a design destroyed unused skips the collective)
    d->pending = nullptr;
    cudaEvent_t last = P->chunk_done.back();
    if (ctx) cudaStreamWaitEvent(ctx->stream, last, 0);      // the DevBufs of P are freed on ctx->stream
    const cudaError_t e = cudaEventSynchronize(last);
    float ms_all = 0, ms_h2d = 0;
    cudaEventElapsedTime(&ms_all, P->ev_begin, last);
    cudaEventElapsedTime(&ms_h2d, P->ev_begin, P->ev_h2d_end);
    d->ms_h2d = ms_h2d; d->ms_pack = ms_all - ms_h2d;        // what follows the last upload: the exposed part of the pack
    const int f0 = P->h_flags[0], f1 = P->h_flags[1];
    if (ctx && P->slot >= 0 && ctx->pack_slot_owner[P->slot] == d) ctx->pack_slot_owner[P->slot] = nullptr;
    g_alloc_ctx = ctx;
    const auto t_del = std::chrono::steady_clock::now();
    delete P;
    if (getenv("OBBOOT_TRACE"))
        fprintf(stderr, "[obboot] async pack: staging released in %.3f ms (host)\n",
                std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t_del).count());
    if (e != cudaSuccess) { d->failed = OB_ERR_CUDA; d->fail_msg = std::string("asynchronous pack failed: ") + cudaGetErrorString(e); }
    else if (f0) { d->failed = OB_ERR_INVALID_GROUP; d->fail_msg = "Invalid group variable: Weights cannot be negative"; }   // ols.rs:60-66
    else if (f1) { d->failed = OB_ERR_INVALID_ARG; d->fail_msg = "categorical code outside [0, levels)"; }
    if (d->failed != OB_OK && !quiet) fail(d->failed, d->fail_msg);
}

void design_alive(const ob_design* d) {
    if (!d->owner) fail(OB_ERR_INVALID_ARG, "this design's context has been destroyed (designs die with their context)");
    if (d->failed != OB_OK) fail(d->failed, d->fail_msg);
}

// entry points that need every row: complete an asynchronous pack first
void design_ready(const ob_design* d) {
    design_alive(d);
    pending_finish(const_cast<ob_design*>(d));
}

const char* status_text(int s) {
    switch (s) {
    case OB_ERR_INVALID_GROUP: return "Invalid group variable: No data in groups for weighted coefficients.";
    case OB_ERR_NALGEBRA: return "Nalgebra error: Failed to perform Cholesky decomposition. Matrix may be singular or not positive definite due to multicollinearity.";
    case OB_ERR_INSUFFICIENT_DATA: return "Insufficient data: Insufficient data for OLS calculation: n_obs must be strictly greater than k";
    default: return "error";
    }
}

// ---- the replicate-batch skeleton shared by the bootstrap drivers (bootstrap_body, heckman_run, mm_run) ----

// The replicate range of a call, from the fields ob_boot_opts and ob_mm_opts share: global replicate ids [rb, re), whether
// the library shards the work over the context's communicator (mode R), and the multiplicity width to start with.
// OLS and Heckman then narrow [rb, re) to the rank's share; Machado-Mata shards its regressions instead.
struct RepRange {
    bool shard_reps; int64_t rb, re, nrep;
    bool index_mode; int count_bytes;
};

// On a clustered design an explicit index stream draws units: BY_GROUP idx_a [reps x M_A] and idx_b [reps x M_B], JOINT
// idx_a [reps x M] alone.
template <typename Opts>
RepRange replicate_range(const ob_ctx* ctx, const ob_design* d, const Opts* o) {
    if (o->reps < 0) fail(OB_ERR_INVALID_ARG, "negative reps");
    RepRange r;
    r.shard_reps = o->shard_replicates != 0 && ctx->comm && ctx->comm->world > 1;
    if (r.shard_reps && (o->rep_begin != 0 || o->rep_end != 0 || o->skip_reduce))
        fail(OB_ERR_INVALID_ARG, "shard_replicates computes the shard itself: rep_begin / rep_end / skip_reduce must be 0");
    r.rb = o->rep_begin; r.re = o->rep_end > 0 ? o->rep_end : o->reps;
    if (r.rb < 0 || r.re < r.rb || r.re > o->reps) fail(OB_ERR_INVALID_ARG, "bad replicate shard");
    r.nrep = r.re - r.rb;
    r.index_mode = o->idx_a != nullptr || o->idx_b != nullptr;
    if (d->cl_strata == OB_CLUSTER_JOINT) {
        if (o->idx_b) fail(OB_ERR_INVALID_ARG, "a JOINT cluster design takes one unit stream: idx_a [reps x M] and idx_b = NULL");
    } else if (r.index_mode && r.nrep > 0 && (!o->idx_a || !o->idx_b)) fail(OB_ERR_INVALID_ARG, "index stream needs both idx_a and idx_b");
    if (o->count_bits != 0 && o->count_bits != 8 && o->count_bits != 16) fail(OB_ERR_INVALID_ARG, "count_bits must be 0, 8 or 16");
    if (o->count_bits == 16 && !gram_fits(d->ldx, 2)) fail(OB_ERR_UNSUPPORTED, "16-bit multiplicities need K + outcomes <= 268");
    r.count_bytes = o->count_bits == 16 ? 2 : 1;
    return r;
}

// One batch of the panel loop: panels [p0, p0 + pn) of the multiplicity matrix hold slots [slot_lo, slot_hi) of the call's
// 1 + nrep (slot 0 of the first batch is the point estimate)
struct Batch {
    int64_t pn, slot_lo, slot_hi, bslots;
    int first_slot;
    int64_t brep;                 // replicates in this batch
    int64_t rep0;                 // global replicate id of the batch's slot 0
    Batch(int64_t p0, int64_t ppb, int64_t panels_total, int64_t slots, int64_t rb)
        : pn(std::min(ppb, panels_total - p0)), slot_lo(p0 * BM), slot_hi(std::min(slots, (p0 + pn) * BM)),
          bslots(slot_hi - slot_lo), first_slot(p0 == 0 ? 1 : 0), brep(bslots - first_slot), rep0(rb + slot_lo - 1) {}
    // GramArgs::tail_mi: valid slots of the batch's last panel -> 8-slot groups, rounded up to a multiple of 4
    int tail_mi() const {
        const int64_t last = bslots - (pn - 1) * BM;
        return (int)std::min<int64_t>(16, ((last + 7) / 8 + 3) / 4 * 4);
    }
};

// The batch's multiplicity columns of both groups (resample.cu), from the caller's index stream or the native Philox
// stream.  The native fix-up tops every replicate up to exactly n_global draws, so it needs the column sums over all row
// shards: row_comm is the mode-N communicator (null otherwise; ms_comm then goes unused).  On a design that is not row
// sharded, shard.n_global == n and shard.row_begin == 0: alloc_group sets row_shard(n, 0, 1), and ob_design_set_row_shard
// with world 1 accepts only n_global == n.  colsum holds 2 x ppb * BM sums.  Returns the number of kernels launched.
// A clustered design (cw non-null) draws the same streams over its units into cw->U (unit_mats matrices: one per group, or
// one for both under JOINT, keyed with stream tag 2), then expands them to the row matrices C and sums the per-slot row
// counts into cw->rows [2][b.pn * BM].
struct ClusterWork {
    DevBuf U[2];                  // [ppb][pad_rows(M)][BM]
    long long* rows = nullptr;    // [2][ppb * BM]
};
int unit_mats(const ob_design* d) { return d->cl_strata == OB_CLUSTER_JOINT ? 1 : 2; }

template <typename Opts>
int generate_counts(const ob_design* d, const Opts* o, const Batch& b, int count_bytes, int64_t ppb, DevBuf (&C)[2],
                    DevBuf (&idx)[2], DevBuf& colsum, DevBuf& lut, int* flags, Comm* row_comm, double* ms_comm, cudaStream_t st,
                    ClusterWork* cw = nullptr) {
    CountsArgs ca[2];
    const int mats = cw ? unit_mats(d) : 2;
    for (int g = 0; g < mats; ++g) {
        const GroupData& G = d->g[g];
        ca[g].C = C[g].p; ca[g].count_bytes = count_bytes; ca[g].n = G.n; ca[g].n_pad = G.n_pad;
        ca[g].n_global = G.shard.n_global; ca[g].row_begin = G.shard.row_begin;
        ca[g].panels = (int)b.pn; ca[g].slots = b.bslots; ca[g].first_slot = b.first_slot; ca[g].rep0 = b.rep0;
        ca[g].group = g; ca[g].seed = o->seed;
        if (cw) {                 // units take the place of rows: M of them, in ascending cluster code
            const int64_t M = d->cl_units[g];
            ca[g].C = cw->U[g].p; ca[g].n = ca[g].n_global = M; ca[g].n_pad = pad_rows(M); ca[g].row_begin = 0;
            ca[g].group = mats == 1 ? 2 : g;
        }
    }
    int launches = 0;
    auto expand = [&] {
        if (!cw) return;
        OB_CUDA(cudaMemsetAsync(cw->rows, 0, sizeof(long long) * 2 * (size_t)b.pn * BM, st));
        for (int g = 0; g < 2; ++g) {
            const int m = mats == 1 ? 0 : g;
            ExpandArgs ea{C[g].p, cw->U[m].p, d->g[g].uid, count_bytes, d->g[g].n, d->g[g].n_pad, pad_rows(d->cl_units[m]),
                          (int)b.pn, b.bslots, cw->rows + (size_t)g * b.pn * BM};
            counts_expand_launch(ea, st);
            launches += 1;
        }
    };
    if (o->idx_a || o->idx_b) {
        for (int g = 0; g < mats; ++g) {
            const uint32_t* h = g == 0 ? o->idx_a : o->idx_b;
            const int64_t n_glob = ca[g].n_global;
            const size_t nb = sizeof(uint32_t) * (size_t)std::max<int64_t>(b.brep, 1) * n_glob;
            if (idx[g].bytes < nb) idx[g].alloc(nb);
            if (b.brep > 0)
                OB_CUDA(cudaMemcpyAsync(idx[g].p, h + (size_t)(b.rep0 + b.first_slot) * n_glob,
                                        sizeof(uint32_t) * (size_t)b.brep * n_glob, cudaMemcpyHostToDevice, st));
            counts_from_indices(ca[g], idx[g].as<uint32_t>(), flags, st);
            launches += 1 + (b.brep > 0 ? (int)((b.brep + 32767) / 32768) : 0);
        }
        expand();
        return launches;
    }
    long long* sums[2] = {colsum.as<long long>(), colsum.as<long long>() + (size_t)ppb * BM};
    OB_CUDA(cudaMemsetAsync(colsum.p, 0, colsum.bytes, st));
    for (int g = 0; g < mats; ++g) {
        counts_philox_body_launch(ca[g], sums[g], lut.as<unsigned char>() + (size_t)g * counts_lut_bytes(), st);
        launches += 2;
    }
    if (row_comm) {
        Timer t_c(st, ms_comm);
        row_comm->allreduce(colsum.p, 2 * (size_t)ppb * BM, CommDType::I64, CommOp::SUM, st);
        t_c.stop(); OB_CUDA(cudaStreamSynchronize(st)); t_c.collect();
    }
    for (int g = 0; g < mats; ++g) {
        counts_philox_fixup_launch(ca[g], sums[g], flags, st);
        launches += b.brep > 0 ? 1 : 0;
    }
    expand();
    return launches;
}

// The batch's Bayesian-bootstrap weights of both groups (resample.cu: native stream, or the caller's explicit fp32 stream
// uploaded per batch into wt) and their per-slot sums esum [2][b.pn * BM]: leaf partials into part, summed by the Gram's
// aligned leaf tree.  Mode N: each rank sums its aligned subtree into esum_local, the per-rank sums are gathered and the top
// of the tree evaluated on every rank (gram_combine_launch), so esum is bit-identical to the single-GPU sums.
struct BayesWork {
    DevBuf wt[2], part, esum, esum_local, gathered;
    int ranks_with_rows[2];
};
int generate_weights(const ob_design* d, const ob_boot_opts* o, const ob_bayes_opts* bo, const Batch& b, DevBuf (&C)[2],
                     BayesWork& w, int* flags, Comm* row_comm, double* ms_comm, cudaStream_t st) {
    const int64_t spad = b.pn * BM;
    int segs[2];
    int64_t leaf0 = 0;
    for (int g = 0; g < 2; ++g) {
        const GroupData& G = d->g[g];
        BayesArgs a;
        a.C = C[g].as<float>(); a.n = G.n; a.n_pad = G.n_pad; a.panels = (int)b.pn;
        a.n_global = G.shard.n_global; a.row_begin = G.shard.row_begin;
        a.slots = b.bslots; a.first_slot = b.first_slot; a.rep0 = b.rep0; a.group = g; a.seed = o->seed;
        a.segs = segs[g] = G.shard.leaf_hi - G.shard.leaf_lo; a.seg_rows = G.shard.seg_rows;
        a.wt = nullptr; a.flags = flags;
        a.part = w.part.as<double>() + (size_t)leaf0 * spad;
        leaf0 += a.segs;
        const float* h = bo ? (g == 0 ? bo->wt_a : bo->wt_b) : nullptr;
        if (h) {
            const size_t nb = sizeof(float) * (size_t)std::max<int64_t>(b.brep, 1) * a.n_global;
            if (w.wt[g].bytes < nb) w.wt[g].alloc(nb);
            if (b.brep > 0)
                OB_CUDA(cudaMemcpyAsync(w.wt[g].p, h + (size_t)(b.rep0 + b.first_slot) * a.n_global,
                                        sizeof(float) * (size_t)b.brep * a.n_global, cudaMemcpyHostToDevice, st));
            a.wt = w.wt[g].as<float>();
        }
        bayes_weights_launch(a, st);
    }
    const int span = d->g[0].shard.leaf_span;
    leaf_sum_launch(w.part.as<double>(), segs, spad, span, row_comm ? w.esum_local.as<double>() : w.esum.as<double>(), st);
    int launches = 3;
    if (row_comm) {
        Timer t_c(st, ms_comm);
        row_comm->allgather(w.esum_local.p, w.gathered.p, sizeof(double) * 2 * (size_t)spad, st);
        gram_combine_launch(w.gathered.as<double>(), row_comm->world, w.ranks_with_rows, spad, w.esum.as<double>(), st);
        t_c.stop(); OB_CUDA(cudaStreamSynchronize(st)); t_c.collect();
        launches += 1;
    }
    return launches;
}

// A batch's deferred error flags (multiplicity kernels): a bad index or a Poisson overshoot fails the call.  A saturated
// count returns true when the run may widen to 16-bit counts and redo, and fails when it may not: already 16-bit, 8 bits
// asked for, or a design (row stride ldx) too wide for the Gram kernel at 16 bits.
bool check_batch_flags(const int flags[4], int count_bytes, int count_bits, int ldx) {
    if (flags[2]) fail(OB_ERR_INVALID_ARG, "resample index out of range");
    if (flags[3]) fail(OB_ERR_INVALID_ARG, "explicit Bayesian weight that is not a positive normal float");
    if (flags[0]) fail(OB_ERR_CUDA, "Poisson body overshot n (probability < 1e-15 per replicate); rerun with another seed");
    if (flags[1] && (count_bytes == 2 || count_bits == 8 || !gram_fits(ldx, 2)))
        fail(OB_ERR_UNSUPPORTED, "row multiplicity overflows the count width");
    return flags[1] != 0;
}

// A host value through an all-reduce over comm (int: I32, long long: I64); every rank returns the same result.
template <typename T>
T allreduce_scalar(Comm* comm, T v, CommOp op, cudaStream_t st) {
    static_assert(std::is_same<T, int>::value || std::is_same<T, long long>::value, "I32 or I64");
    DevBuf d(sizeof v);
    OB_CUDA(cudaMemcpyAsync(d.p, &v, sizeof v, cudaMemcpyHostToDevice, st));
    comm->allreduce(d.p, 1, std::is_same<T, int>::value ? CommDType::I32 : CommDType::I64, op, st);
    OB_CUDA(cudaMemcpyAsync(&v, d.p, sizeof v, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaStreamSynchronize(st));
    return v;
}

// Runs body.  With a communicator all ranks leave together: a rank that failed (a bad index in its share, device memory it
// could not get) must not leave its peers waiting in their next collective.  The ranks agree on the highest status; a
// rank that failed raises its own error, the others peer_msg with the agreed status.
template <typename F>
void agree_on_status(Comm* comm, cudaStream_t st, F&& body, const char* peer_msg) {
    if (!comm) { body(); return; }
    int rc = OB_OK;
    std::exception_ptr own;
    try { body(); }
    catch (const StatusError& e) { rc = e.code; own = std::current_exception(); }
    catch (const CudaError& e) {
        cudaGetLastError();
        if (e.code != cudaErrorMemoryAllocation) throw;
        rc = OB_ERR_CUDA; own = std::current_exception();
    }
    const int agreed = allreduce_scalar(comm, rc, CommOp::MAX, st);
    if (own) std::rethrow_exception(own);
    if (agreed != OB_OK) fail((ob_status)agreed, std::string(peer_msg) + ": " + status_text(agreed));
}

// All-gather of per-rank rows in shard order: rank r contributes rows [b, e) of ob_replicate_shard(total, world, r) from
// `mine`, `unit` elements each; every rank receives all `total` rows in `all` (grown as needed), which is returned.
template <typename T>
T* allgather_shards(Comm* comm, int64_t total, size_t unit, const T* mine, DevBuf& all, cudaStream_t st) {
    const size_t row = sizeof(T) * unit, need = row * (size_t)std::max<int64_t>(total, 1);
    if (all.bytes < need) all.alloc(need);
    std::vector<size_t> off(comm->world), sz(comm->world);
    for (int r = 0; r < comm->world; ++r) {
        int64_t b = 0, e = 0;
        ob_replicate_shard(total, comm->world, r, &b, &e);
        off[r] = (size_t)b * row; sz[r] = (size_t)(e - b) * row;
    }
    comm->allgatherv(mine, all.p, off.data(), sz.data(), st);
    return all.as<T>();
}

// (5) The replicate rows reduced to standard errors, p-values, percentile CIs and t statistics (reduce_stats.cu), each
// [S] result downloaded to dst[k] unless that is null.  ms (may be null) accumulates the reduction's device time.
void reduce_to_host(cudaStream_t st, const double* stats_rows, const int* status_rows, int64_t reps, int S,
                    const double* point, double* const dst[5], int64_t* n_ok, double* ms) {
    DevBuf d_out(sizeof(double) * 5 * (size_t)S), d_nok(sizeof(long long)), d_rs(reduce_stats_scratch_bytes(reps, S));
    std::optional<Timer> t_red;
    if (ms) t_red.emplace(st, ms);
    reduce_stats_launch(stats_rows, status_rows, reps, S, point, d_out.as<double>(), d_nok.as<long long>(), st, d_rs.as<double>());
    if (t_red) t_red->stop();
    std::vector<double> out5(5 * (size_t)S);
    long long nok = 0;
    OB_CUDA(cudaMemcpyAsync(out5.data(), d_out.p, d_out.bytes, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaMemcpyAsync(&nok, d_nok.p, sizeof nok, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaStreamSynchronize(st));
    if (t_red) t_red->collect();
    if (n_ok) *n_ok = nok;
    for (int k = 0; k < 5; ++k)
        if (dst[k]) memcpy(dst[k], out5.data() + (size_t)k * S, sizeof(double) * S);
}

}  // namespace

extern "C" {

uint32_t ob_abi_version(void) { return OBBOOT_ABI_VERSION; }

ob_status ob_device_count(int32_t* n_out) {
    if (!n_out) return OB_ERR_INVALID_ARG;
    int n = 0;
    const cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) { cudaGetLastError(); *n_out = 0; return OB_ERR_NO_DEVICE; }
    *n_out = n;
    return OB_OK;
}

ob_status ob_ctx_create(int32_t device, ob_ctx** out) {
    if (!out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess || n == 0) { cudaGetLastError(); return OB_ERR_NO_DEVICE; }
    if (device < 0 || device >= n) return OB_ERR_INVALID_ARG;
    auto ctx = std::make_unique<ob_ctx>();
    ctx->device = device;
    const ob_status st = guarded(ctx.get(), [&] {
        cudaDeviceProp prop;
        OB_CUDA(cudaGetDeviceProperties(&prop, device));
        if (prop.major != 10) fail(OB_ERR_NO_DEVICE, "libobboot is built for sm_100a (B200) only");
        ctx->num_sms = prop.multiProcessorCount;
        OB_CUDA(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        OB_CUDA(cudaStreamCreateWithFlags(&ctx->stream_side, cudaStreamNonBlocking));
        OB_CUDA(cudaStreamCreateWithFlags(&ctx->stream_copy, cudaStreamNonBlocking));
        OB_CUDA(cudaHostAlloc((void**)&ctx->h_pack_flags, sizeof(int) * 4 * ob_ctx::PACK_SLOTS, cudaHostAllocDefault));
        cudaMemPoolProps props{};
        props.allocType = cudaMemAllocationTypePinned;
        props.handleTypes = cudaMemHandleTypeNone;
        props.location.type = cudaMemLocationTypeDevice;
        props.location.id = device;
        OB_CUDA(cudaMemPoolCreate(&ctx->pool, &props));
        OB_CUDA(cudaMemPoolCreate(&ctx->pool_pack, &props));
        OB_CUDA(cudaMemPoolCreate(&ctx->pool_design, &props));
        unsigned long long keep = ~0ull;   // never trim on synchronisation: the workspace is reused by the next call
        OB_CUDA(cudaMemPoolSetAttribute(ctx->pool, cudaMemPoolAttrReleaseThreshold, &keep));
        OB_CUDA(cudaMemPoolSetAttribute(ctx->pool_pack, cudaMemPoolAttrReleaseThreshold, &keep));
        OB_CUDA(cudaMemPoolSetAttribute(ctx->pool_design, cudaMemPoolAttrReleaseThreshold, &keep));
    });
    if (st != OB_OK) return st;
    *out = ctx.release();
    return OB_OK;
}

void ob_ctx_destroy(ob_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream_copy) cudaStreamSynchronize(ctx->stream_copy);
    {   // designs that outlive their context: free their device memory now, leave the host structs to their owners
        std::lock_guard<std::mutex> lk(ctx->designs_mu);
        for (ob_design* d : ctx->designs) { pending_finish(d, true); design_release_device(d); d->owner = nullptr; d->stream = nullptr; }
        ctx->designs.clear();
        for (ob_gram_cache* c : ctx->caches) { cache_release_device(c); c->owner = nullptr; }
        ctx->caches.clear();
    }
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    if (ctx->stream_side) { cudaStreamSynchronize(ctx->stream_side); cudaStreamDestroy(ctx->stream_side); }
    if (ctx->stream_copy) cudaStreamDestroy(ctx->stream_copy);
    if (ctx->h_pack_flags) cudaFreeHost(ctx->h_pack_flags);
    ctx->comm.reset();
    if (ctx->pool) cudaMemPoolDestroy(ctx->pool);
    if (ctx->pool_pack) cudaMemPoolDestroy(ctx->pool_pack);
    if (ctx->pool_design) cudaMemPoolDestroy(ctx->pool_design);
    if (ctx->stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
}

ob_status ob_host_alloc(size_t bytes, void** out) {
    if (!out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    const cudaError_t e = cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return e == cudaErrorNoDevice ? OB_ERR_NO_DEVICE : OB_ERR_CUDA; }
    return OB_OK;
}

void ob_host_free(void* p) { if (p) cudaFreeHost(p); }

ob_status ob_host_register(void* p, size_t bytes) {
    if (!p || !bytes) return OB_ERR_INVALID_ARG;
    const cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { cudaGetLastError(); return OB_ERR_CUDA; }
    return OB_OK;
}

ob_status ob_host_unregister(void* p) {
    if (!p) return OB_ERR_INVALID_ARG;
    const cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) { cudaGetLastError(); return OB_ERR_CUDA; }
    return OB_OK;
}

ob_status ob_replicate_shard(int64_t reps, int32_t world, int32_t rank, int64_t* rep_begin, int64_t* rep_end) {
    if (reps < 0 || world < 1 || rank < 0 || rank >= world) return OB_ERR_INVALID_ARG;
    const int64_t base = reps / world, extra = reps % world;
    const int64_t b = rank * base + std::min<int64_t>(rank, extra);
    if (rep_begin) *rep_begin = b;
    if (rep_end) *rep_end = b + base + (rank < extra ? 1 : 0);
    return OB_OK;
}

const char* ob_last_error(const ob_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int32_t ob_num_stats(int32_t K, int32_t n_norm, const int32_t* norm_has_base) {
    int nb = 0;
    for (int v = 0; v < n_norm; ++v) nb += (norm_has_base && norm_has_base[v]) ? 1 : 0;
    return 5 + 2 * (K + nb);
}

// ---- multi-GPU: communicators and row sharding (SURVEY.md 8e, mode N) ----
ob_status ob_comm_unique_id(uint8_t* id128) {
    if (!id128) return OB_ERR_INVALID_ARG;
    try { nccl_unique_id(id128); } catch (const StatusError&) { return OB_ERR_NCCL; } catch (const CudaError&) { return OB_ERR_CUDA; }
    return OB_OK;
}

ob_status ob_comm_init_nccl(ob_ctx* ctx, const uint8_t* id128, int32_t rank, int32_t world) {
    if (!ctx || !id128) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        // any world size shards replicates (mode R); row shards (mode N) additionally need a power of two,
        // checked by ob_design_set_row_shard
        if (world < 1 || world > MAX_WORLD || rank < 0 || rank >= world)
            fail(OB_ERR_INVALID_ARG, "1 <= world <= 64 and 0 <= rank < world");
        ctx->comm.reset(comm_create_nccl(id128, rank, world));
    });
}

ob_status ob_local_group_create(int32_t world, ob_local_group** out) {
    if (!out || world < 1 || world > MAX_WORLD) return OB_ERR_INVALID_ARG;
    auto* g = new ob_local_group;
    g->g = local_group_create(world); g->world = world;
    *out = g;
    return OB_OK;
}

void ob_local_group_destroy(ob_local_group* g) {
    if (!g) return;
    local_group_destroy(g->g);
    delete g;
}

ob_status ob_comm_init_local(ob_ctx* ctx, ob_local_group* group, int32_t rank) {
    if (!ctx || !group) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        if (rank < 0 || rank >= group->world) fail(OB_ERR_INVALID_ARG, "rank outside the group");
        ctx->comm.reset(comm_create_local(group->g, rank, ctx->device));
    });
}

void ob_comm_destroy(ob_ctx* ctx) {
    if (!ctx) return;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    ctx->comm.reset();
}

ob_status ob_row_shard_plan(int64_t n_group, int32_t world, int32_t rank, int64_t* row_begin, int64_t* row_end) {
    if (n_group < 0 || world < 1 || world > MAX_WORLD || (world & (world - 1)) || rank < 0 || rank >= world) return OB_ERR_INVALID_ARG;
    const RowShard r = row_shard(n_group, rank, world);
    if (row_begin) *row_begin = r.row_begin;
    if (row_end) *row_end = r.row_begin + r.n_local;
    return OB_OK;
}

ob_status ob_design_set_row_shard(ob_design* d, int64_t n_a_global, int64_t n_b_global, int32_t world, int32_t rank) {
    if (!d || world < 1 || world > MAX_WORLD || (world & (world - 1)) || rank < 0 || rank >= world) return OB_ERR_INVALID_ARG;
    // (a design whose asynchronous pack is still in flight can be marked: only the metadata changes, and the upload's
    //  progress is tracked in local rows either way)
    if (d->failed != OB_OK) return d->failed;
    if (d->pending && d->pending->exchange_pending) return OB_ERR_INVALID_ARG;    // already a row shard
    const RowShard ra = row_shard(n_a_global, rank, world), rb = row_shard(n_b_global, rank, world);
    if (ra.n_local != d->g[0].n || rb.n_local != d->g[1].n) return OB_ERR_INVALID_ARG;   // rows must follow ob_row_shard_plan
    d->g[0].shard = ra; d->g[1].shard = rb;
    d->world = world; d->rank = rank;
    ++d->x_gen;
    return OB_OK;
}

// Mode R with a distributed upload: every rank packed a contiguous slice of the frame (slices in rank order); the
// full per-group designs are assembled on every rank by one variable-size all-gather over NVLink, so a rank moves
// only 1/world of the frame across PCIe.
ob_status ob_design_allgather_rows(ob_ctx* ctx, const ob_design* local, ob_design** out) {
    if (!ctx || !local || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        design_ready(local);
        Comm* comm = ctx->comm.get();
        if (!comm) fail(OB_ERR_NCCL, "ob_design_allgather_rows needs ob_comm_init_* on this context");
        if (local->world != 1) fail(OB_ERR_INVALID_ARG, "the local design is a row shard (mode N); gather applies to frame slices");
        cudaStream_t st = ctx->stream;
        const int world = comm->world;
        // row counts of every rank's slice, per group (+ a consistency word: K, n_cont, weighted)
        // word 2: shape; bit 0 of word 3: the slice carries a frame-row map; rest of word 3: rows of the slice's frame
        std::vector<long long> mine = {(long long)local->g[0].n, (long long)local->g[1].n,
                                       ((long long)local->K << 32) | ((long long)local->n_cont << 1) | (local->weighted ? 1 : 0),
                                       ((long long)local->n_frame << 1) | ((local->g[0].src && local->g[1].src) ? 1 : 0)};
        DevBuf d_mine(sizeof(long long) * 4), d_all(sizeof(long long) * 4 * world);
        OB_CUDA(cudaMemcpyAsync(d_mine.p, mine.data(), sizeof(long long) * 4, cudaMemcpyHostToDevice, st));
        comm->allgather(d_mine.p, d_all.p, sizeof(long long) * 4, st);
        std::vector<long long> all4(4 * (size_t)world), all(3 * (size_t)world);
        OB_CUDA(cudaMemcpyAsync(all4.data(), d_all.p, sizeof(long long) * 4 * world, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        bool have_src = true;
        std::vector<long long> frame_off((size_t)world + 1, 0);
        for (int r = 0; r < world; ++r) {
            for (int k = 0; k < 3; ++k) all[3 * r + k] = all4[4 * r + k];
            if (all[3 * r + 2] != mine[2]) fail(OB_ERR_INVALID_ARG, "ranks disagree on the design shape (K, n_cont, weights)");
            have_src = have_src && (all4[4 * r + 3] & 1);
            frame_off[r + 1] = frame_off[r] + (all4[4 * r + 3] >> 1);
        }
        if (frame_off[world] > 0xFFFFFFFFll) have_src = false;

        std::unique_ptr<ob_design, void (*)(ob_design*)> d(new ob_design, ob_design_destroy);
        design_register(ctx, d.get()); d->stream = ctx->stream; d->device = ctx->device; d->K = local->K; d->n_cont = local->n_cont; d->V = local->V;
        d->ldx = local->ldx; d->weighted = local->weighted; d->cat_levels = local->cat_levels;
        for (int g = 0; g < 2; ++g) {
            std::vector<size_t> off_x(world), sz_x(world), off_w(world), sz_w(world);
            long long total = 0;
            for (int r = 0; r < world; ++r) {
                const long long nr = all[3 * r + g];
                off_x[r] = (size_t)total * d->ldx * sizeof(double); sz_x[r] = (size_t)nr * d->ldx * sizeof(double);
                off_w[r] = (size_t)total * sizeof(double);          sz_w[r] = (size_t)nr * sizeof(double);
                total += nr;
            }
            alloc_group(ctx, d->g[g], total, d->ldx, d->weighted);
            comm->allgatherv(local->g[g].X, d->g[g].X, off_x.data(), sz_x.data(), st);
            if (d->weighted) comm->allgatherv(local->g[g].w, d->g[g].w, off_w.data(), sz_w.data(), st);
            if (have_src) {
                // the frame-row map travels too (ob_design_update_outcome on the gathered design): a slice's rows point into
                // its own frame slice, so rank r's block is shifted by the rows of the slices before it
                std::vector<size_t> off_s(world), sz_s(world);
                for (int r = 0; r < world; ++r) { off_s[r] = off_w[r] / 2; sz_s[r] = sz_w[r] / 2; }
                comm->allgatherv(local->g[g].src, d->g[g].src, off_s.data(), sz_s.data(), st);
                for (int r = 0; r < world; ++r)
                    add_u32_launch(d->g[g].src + off_s[r] / sizeof(uint32_t), (int64_t)(sz_s[r] / sizeof(uint32_t)), (uint32_t)frame_off[r], st);
            } else {
                cudaFreeAsync(d->g[g].src, st); d->g[g].src = nullptr;
            }
            scale_rows_launch(d->g[g], d->ldx, st);
        }
        d->n_frame = frame_off[world];
        OB_CUDA(cudaStreamSynchronize(st));
        *out = d.release();
    });
}

// Frame slices -> row shards (mode N) without a host round trip: every rank packed a contiguous slice of the frame
// (slices in rank order); the rows of each group are re-cut along ob_row_shard_plan and exchanged over the communicator
// (NVLink).  When the groups are spread evenly over the frame almost nothing moves -- a slice already holds about the
// rows its rank will own -- and a frame sorted by group still moves every row at most once.
ob_status ob_design_redistribute_rows(ob_ctx* ctx, const ob_design* local, ob_design** out) {
    if (!ctx || !local || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        design_ready(local);
        Comm* comm = ctx->comm.get();
        if (!comm) fail(OB_ERR_NCCL, "ob_design_redistribute_rows needs ob_comm_init_* on this context");
        if (local->world != 1) fail(OB_ERR_INVALID_ARG, "the local design is already a row shard");
        const int world = comm->world, me = comm->rank;
        if (world & (world - 1)) fail(OB_ERR_INVALID_ARG, "row shards need a power-of-two world");
        cudaStream_t st = ctx->stream;
        std::vector<long long> mine = {(long long)local->g[0].n, (long long)local->g[1].n,
                                       ((long long)local->K << 32) | ((long long)local->n_cont << 1) | (local->weighted ? 1 : 0),
                                       ((long long)local->n_frame << 1) | ((local->g[0].src && local->g[1].src) ? 1 : 0)};
        DevBuf d_mine(sizeof(long long) * 4), d_all(sizeof(long long) * 4 * world);
        OB_CUDA(cudaMemcpyAsync(d_mine.p, mine.data(), sizeof(long long) * 4, cudaMemcpyHostToDevice, st));
        comm->allgather(d_mine.p, d_all.p, sizeof(long long) * 4, st);
        std::vector<long long> all(4 * (size_t)world);
        OB_CUDA(cudaMemcpyAsync(all.data(), d_all.p, sizeof(long long) * 4 * world, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        bool have_src = true;
        std::vector<long long> frame_off((size_t)world + 1, 0);
        for (int r = 0; r < world; ++r) {
            if (all[4 * r + 2] != mine[2]) fail(OB_ERR_INVALID_ARG, "ranks disagree on the design shape (K, n_cont, weights)");
            have_src = have_src && (all[4 * r + 3] & 1);
            frame_off[r + 1] = frame_off[r] + (all[4 * r + 3] >> 1);
        }
        if (frame_off[world] > 0xFFFFFFFFll) have_src = false;

        std::unique_ptr<ob_design, void (*)(ob_design*)> d(new ob_design, ob_design_destroy);
        design_register(ctx, d.get()); d->stream = ctx->stream; d->device = ctx->device; d->K = local->K; d->n_cont = local->n_cont; d->V = local->V;
        d->ldx = local->ldx; d->weighted = local->weighted; d->cat_levels = local->cat_levels;
        d->world = world; d->rank = me;
        d->n_frame = frame_off[world];
        for (int g = 0; g < 2; ++g) {
            std::vector<long long> off((size_t)world + 1, 0);          // group rows held by the slices before rank r
            for (int r = 0; r < world; ++r) off[r + 1] = off[r] + all[4 * r + g];
            const long long n_glob = off[world];
            std::vector<RowShard> plan((size_t)world);
            for (int t = 0; t < world; ++t) plan[t] = row_shard(n_glob, t, world);
            alloc_group(ctx, d->g[g], plan[me].n_local, d->ldx, d->weighted);
            d->g[g].shard = plan[me];
            std::vector<size_t> rows((size_t)world * world, 0), send_row((size_t)world, 0), recv_row((size_t)world, 0);
            for (int sidx = 0; sidx < world; ++sidx)
                for (int t = 0; t < world; ++t) {
                    const long long lo = std::max<long long>(off[sidx], plan[t].row_begin);
                    const long long hi = std::min<long long>(off[sidx + 1], plan[t].row_begin + plan[t].n_local);
                    rows[(size_t)sidx * world + t] = hi > lo ? (size_t)(hi - lo) : 0;
                }
            for (int r = 0; r < world; ++r) {
                send_row[r] = (size_t)(std::max<long long>(off[me], plan[r].row_begin) - off[me]);              // in my slice
                recv_row[r] = (size_t)(std::max<long long>(off[r], plan[me].row_begin) - plan[me].row_begin);   // in my shard
            }
            auto exchange = [&](const void* sendbuf, void* recvbuf, size_t row_bytes) {
                std::vector<size_t> b(rows.size()), so((size_t)world), ro((size_t)world);
                for (size_t i = 0; i < rows.size(); ++i) b[i] = rows[i] * row_bytes;
                for (int r = 0; r < world; ++r) { so[r] = send_row[r] * row_bytes; ro[r] = recv_row[r] * row_bytes; }
                comm->alltoallv(sendbuf, so.data(), recvbuf, ro.data(), b.data(), st);
                OB_CUDA(cudaStreamSynchronize(st));      // the offset tables live on this stack frame
            };
            exchange(local->g[g].X, d->g[g].X, sizeof(double) * (size_t)d->ldx);
            if (d->weighted) exchange(local->g[g].w, d->g[g].w, sizeof(double));
            if (have_src) {       // frame-row map (ob_design_update_outcome on the shard): blocks from rank r shift by its frame offset
                exchange(local->g[g].src, d->g[g].src, sizeof(uint32_t));
                for (int r = 0; r < world; ++r)
                    add_u32_launch(d->g[g].src + recv_row[r], (int64_t)rows[(size_t)r * world + me], (uint32_t)frame_off[r], st);
            } else {
                cudaFreeAsync(d->g[g].src, st); d->g[g].src = nullptr;
            }
            scale_rows_launch(d->g[g], d->ldx, st);
        }
        OB_CUDA(cudaStreamSynchronize(st));
        *out = d.release();
    });
}

void ob_design_destroy(ob_design* d) {
    if (!d) return;
    if (ob_ctx* ctx = d->owner) {      // orphaned designs (context already destroyed) hold no device memory any more
        int prev = -1;
        cudaGetDevice(&prev);          // may run on a foreign thread (finalisers): leave its current device as it was
        cudaSetDevice(d->device);
        pending_finish(d, true);
        {
            std::lock_guard<std::mutex> lk(ctx->designs_mu);
            ctx->designs.erase(d);
        }
        design_release_device(d);
        if (prev >= 0 && prev != d->device) cudaSetDevice(prev);
    }
    delete d;
}

ob_status ob_design_shape(const ob_design* d, int64_t* na, int64_t* nb, int32_t* K, int32_t* n_cont) {
    if (!d) return OB_ERR_INVALID_ARG;
    if (na) *na = d->g[0].n;
    if (nb) *nb = d->g[1].n;
    if (K) *K = d->K;
    if (n_cont) *n_cont = d->n_cont;
    return OB_OK;
}

ob_status ob_design_row_shard(const ob_design* d, int64_t* n_a_global, int64_t* n_b_global, int32_t* world, int32_t* rank) {
    if (!d) return OB_ERR_INVALID_ARG;
    if (n_a_global) *n_a_global = d->g[0].shard.n_global;
    if (n_b_global) *n_b_global = d->g[1].shard.n_global;
    if (world) *world = d->world;
    if (rank) *rank = d->rank;
    return OB_OK;
}

ob_status ob_design_pack_timings(const ob_design* d, double* ms_h2d, double* ms_pack_kernels) {
    if (!d) return OB_ERR_INVALID_ARG;
    if (d->pending) { cudaSetDevice(d->device); pending_finish(const_cast<ob_design*>(d), true); }
    if (ms_h2d) *ms_h2d = d->ms_h2d;
    if (ms_pack_kernels) *ms_pack_kernels = d->ms_pack;
    return OB_OK;
}

ob_status ob_design_from_dense(ob_ctx* ctx, int32_t K, int32_t n_cont,
                               const double* Xa, const double* ya, const double* wa, int64_t na,
                               const double* Xb, const double* yb, const double* wb, int64_t nb,
                               ob_design** out) {
    if (!ctx || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        if (K < 1 || n_cont < 0 || n_cont > K - 1 || na < 0 || nb < 0) fail(OB_ERR_INVALID_ARG, "bad design shape");
        if ((na && (!Xa || !ya)) || (nb && (!Xb || !yb))) fail(OB_ERR_INVALID_ARG, "null design pointer");
        if ((wa == nullptr) != (wb == nullptr) && na && nb) fail(OB_ERR_INVALID_ARG, "weights must be given for both groups or neither");
        if (K + 1 > MAX_DESIGN_COLS) fail(OB_ERR_UNSUPPORTED, "design wider than 280 columns (the Gram kernel stages whole rows in shared memory)");
        const double* ws[2] = {wa, wb};
        const int64_t ns[2] = {na, nb};
        for (int g = 0; g < 2; ++g)
            if (ws[g])
                for (int64_t i = 0; i < ns[g]; ++i)
                    if (ws[g][i] < 0.0) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: Weights cannot be negative");  // ols.rs:60-66
        std::unique_ptr<ob_design, void (*)(ob_design*)> d(new ob_design, ob_design_destroy);
        design_register(ctx, d.get()); d->stream = ctx->stream; d->device = ctx->device; d->K = K; d->n_cont = n_cont; d->V = K + 1; d->ldx = design_ldx(K + 1);
        d->weighted = (wa != nullptr) || (wb != nullptr);
        const double* Xs[2] = {Xa, Xb};
        const double* ys[2] = {ya, yb};
        for (int g = 0; g < 2; ++g) {
            alloc_group(ctx, d->g[g], ns[g], d->ldx, d->weighted);
            if (ns[g] == 0) continue;
            OB_CUDA(cudaMemcpy2DAsync(d->g[g].X, sizeof(double) * d->ldx, Xs[g], sizeof(double) * K, sizeof(double) * K,
                                      (size_t)ns[g], cudaMemcpyHostToDevice, ctx->stream));
            OB_CUDA(cudaMemcpy2DAsync(d->g[g].X + K, sizeof(double) * d->ldx, ys[g], sizeof(double), sizeof(double),
                                      (size_t)ns[g], cudaMemcpyHostToDevice, ctx->stream));
            if (d->weighted && ws[g])
                OB_CUDA(cudaMemcpyAsync(d->g[g].w, ws[g], sizeof(double) * (size_t)ns[g], cudaMemcpyHostToDevice, ctx->stream));
            iota_launch(d->g[g].src, ns[g], (uint32_t)(g == 0 ? 0 : na), ctx->stream);
        }
        d->n_frame = na + nb;
        for (int g = 0; g < 2; ++g) scale_rows_launch(d->g[g], d->ldx, ctx->stream);
        OB_CUDA(cudaStreamSynchronize(ctx->stream));
        *out = d.release();
    });
}

}  // extern "C"

namespace {

// pack kernels over a staged frame -> resident design (prepare_data + split_groups, once)
std::unique_ptr<ob_design, void (*)(ob_design*)> pack_staged(ob_ctx* ctx, StagedFrame& sf, const int32_t* cat_levels) {
    cudaStream_t st = ctx->stream;
    const int64_t n = sf.n;
    int K = 1 + sf.n_cont;
    std::vector<int32_t> dummy_start(std::max(sf.n_cat, 1), 0);
    for (int q = 0; q < sf.n_cat; ++q) {
        if (cat_levels[q] < 1) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: Could not get reference category");  // builder.rs:392-399
        dummy_start[q] = K;
        K += cat_levels[q] - 1;
    }
    if (K + 1 > MAX_DESIGN_COLS) fail(OB_ERR_UNSUPPORTED, "design wider than 280 columns (the Gram kernel stages whole rows in shared memory)");
    if (n > 0xFFFFFFFFll) fail(OB_ERR_UNSUPPORTED, "frames beyond 2^32 rows (IdxSize is u32 in the reference too)");
    g_alloc_pack = true;
    std::vector<const double*> h_cont(std::max(sf.n_cont, 1), nullptr);
    std::vector<const int32_t*> h_cat(std::max(sf.n_cat, 1), nullptr);
    for (int c = 0; c < sf.n_cont; ++c) h_cont[c] = sf.cols[c].as<double>();
    for (int q = 0; q < sf.n_cat; ++q) h_cat[q] = sf.cats[q].as<int32_t>();
    DevBuf d_cont_ptrs(sizeof(void*) * h_cont.size()), d_cat_ptrs(sizeof(void*) * h_cat.size());
    DevBuf d_levels(sizeof(int32_t) * std::max(sf.n_cat, 1)), d_dstart(sizeof(int32_t) * dummy_start.size());
    OB_CUDA(cudaMemcpyAsync(d_cont_ptrs.p, h_cont.data(), sizeof(void*) * h_cont.size(), cudaMemcpyHostToDevice, st));
    OB_CUDA(cudaMemcpyAsync(d_cat_ptrs.p, h_cat.data(), sizeof(void*) * h_cat.size(), cudaMemcpyHostToDevice, st));
    if (sf.n_cat) OB_CUDA(cudaMemcpyAsync(d_levels.p, cat_levels, sizeof(int32_t) * sf.n_cat, cudaMemcpyHostToDevice, st));
    OB_CUDA(cudaMemcpyAsync(d_dstart.p, dummy_start.data(), sizeof(int32_t) * dummy_start.size(), cudaMemcpyHostToDevice, st));

    PackArgs pa;
    pa.n = n; pa.n_cont = sf.n_cont; pa.n_cat = sf.n_cat;
    pa.d_cont = d_cont_ptrs.as<const double*>(); pa.d_cat = d_cat_ptrs.as<const int32_t*>();
    pa.d_cat_levels = d_levels.as<int32_t>(); pa.d_dummy_start = d_dstart.as<int32_t>();
    pa.d_y = sf.y.as<double>(); pa.d_w = sf.weighted ? sf.w.as<double>() : nullptr; pa.d_group = sf.grp.as<uint8_t>();
    pa.K = K; pa.ldx = design_ldx(K + 1);

    const int nblk = pack_num_blocks(n);
    DevBuf d_bc(sizeof(long long) * 2 * (size_t)std::max(nblk, 1)), d_tot(sizeof(long long) * 2), d_flags(sizeof(int) * 4);
    OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
    double ms_pack = 0.0;
    Timer t_pack(st, &ms_pack);
    pack_count_scan(pa, d_bc.as<long long>(), d_tot.as<long long>(), d_flags.as<int>(), st);
    long long tot[2]; int flags[4];
    OB_CUDA(cudaMemcpyAsync(tot, d_tot.p, sizeof tot, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaStreamSynchronize(st));
    if (flags[0]) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: Weights cannot be negative");

    std::unique_ptr<ob_design, void (*)(ob_design*)> d(new ob_design, ob_design_destroy);
    design_register(ctx, d.get()); d->stream = ctx->stream; d->device = ctx->device; d->K = K; d->n_cont = sf.n_cont; d->V = K + 1; d->ldx = pa.ldx;
    d->weighted = sf.weighted;
    d->cat_levels.assign(cat_levels, cat_levels + sf.n_cat);
    d->n_frame = n;
    alloc_group(ctx, d->g[0], tot[0], d->ldx, d->weighted, false);
    alloc_group(ctx, d->g[1], tot[1], d->ldx, d->weighted, false);
    pack_scatter(pa, d_bc.as<long long>(), d->g[0], d->g[1], d_flags.as<int>(), st);   // writes X, w, src and the scaled copy
    t_pack.stop();
    OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaStreamSynchronize(st));
    t_pack.collect();
    d->ms_h2d = sf.ms_h2d; d->ms_pack = ms_pack;
    if (flags[1]) fail(OB_ERR_INVALID_ARG, "categorical code outside [0, levels)");
    return d;
}

template <typename T>
void stage_column(DevBuf& buf, const T* host, int64_t n, cudaStream_t st) {
    buf.alloc(sizeof(T) * (size_t)std::max<int64_t>(n, 1));
    if (n) OB_CUDA(cudaMemcpyAsync(buf.p, host, sizeof(T) * (size_t)n, cudaMemcpyHostToDevice, st));
}

}  // namespace

// raw frame staged on the device between ob_ingest_begin and ob_ingest_finish
struct ob_ingest {
    ob_ctx* ctx = nullptr;
    StagedFrame sf;
    std::vector<DevBuf> valid;            // validity bytes of numeric columns that carry nulls
    DevBuf group_codes, row_valid;
    std::vector<DevBuf> present;          // per dictionary column (categoricals.., group)
    std::vector<int32_t> dict_size;
    std::vector<std::vector<uint8_t>> h_present;
    int64_t kept = 0;
};

extern "C" {

ob_status ob_design_pack(ob_ctx* ctx, const ob_frame_view* f, ob_design** out) {
    if (!ctx || !f || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        if (f->n < 0 || f->n_cont < 0 || f->n_cat < 0) fail(OB_ERR_INVALID_ARG, "bad frame shape");
        if (f->n && (!f->outcome || !f->group)) fail(OB_ERR_INVALID_ARG, "null frame column");
        cudaStream_t st = ctx->stream;
        g_alloc_pack = true;
        StagedFrame sf;
        sf.n = f->n; sf.n_cont = f->n_cont; sf.n_cat = f->n_cat; sf.weighted = f->weights != nullptr;
        sf.cols.resize(f->n_cont); sf.cats.resize(f->n_cat);
        Timer t_h2d(st, &sf.ms_h2d);
        for (int c = 0; c < f->n_cont; ++c) {
            if (!f->cont[c]) fail(OB_ERR_INVALID_ARG, "null predictor column");
            stage_column(sf.cols[c], f->cont[c], f->n, st);
        }
        for (int q = 0; q < f->n_cat; ++q) {
            if (!f->cat_codes[q]) fail(OB_ERR_INVALID_ARG, "null categorical column");
            stage_column(sf.cats[q], f->cat_codes[q], f->n, st);
        }
        stage_column(sf.y, f->outcome, f->n, st);
        stage_column(sf.grp, f->group, f->n, st);
        if (f->weights) stage_column(sf.w, f->weights, f->n, st);
        t_h2d.stop();
        OB_CUDA(cudaStreamSynchronize(st));
        t_h2d.collect();
        *out = pack_staged(ctx, sf, f->cat_levels).release();
    });
}

// Asynchronous pack.  Host part (about a millisecond): upload the group column, count and scan it, size and allocate
// the design.  Everything else is queued on the copy stream in row chunks -- the column slices of a chunk, then the
// pack kernel over its blocks -- with one event per chunk that ob_bootstrap_run waits on.
static ob_status pack_async_impl(ob_ctx* ctx, const ob_frame_view* f, bool shard, ob_design** out) {
    if (!ctx || !f || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        Comm* comm = shard ? ctx->comm.get() : nullptr;
        if (shard && !comm) fail(OB_ERR_NCCL, "ob_design_pack_row_shard_async needs ob_comm_init_* on this context");
        if (shard && (comm->world & (comm->world - 1))) fail(OB_ERR_INVALID_ARG, "row shards need a power-of-two world");
        if (f->n < 0 || f->n_cont < 0 || f->n_cat < 0) fail(OB_ERR_INVALID_ARG, "bad frame shape");
        if (f->n && (!f->outcome || !f->group)) fail(OB_ERR_INVALID_ARG, "null frame column");
        for (int c = 0; c < f->n_cont; ++c) if (!f->cont[c]) fail(OB_ERR_INVALID_ARG, "null predictor column");
        for (int q = 0; q < f->n_cat; ++q) if (!f->cat_codes[q]) fail(OB_ERR_INVALID_ARG, "null categorical column");
        const int64_t n = f->n;
        int K = 1 + f->n_cont;
        std::vector<int32_t> dummy_start(std::max(f->n_cat, 1), 0);
        for (int q = 0; q < f->n_cat; ++q) {
            if (f->cat_levels[q] < 1) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: Could not get reference category");
            dummy_start[q] = K;
            K += f->cat_levels[q] - 1;
        }
        if (K + 1 > MAX_DESIGN_COLS) fail(OB_ERR_UNSUPPORTED, "design wider than 280 columns (the Gram kernel stages whole rows in shared memory)");
        if (n > 0xFFFFFFFFll) fail(OB_ERR_UNSUPPORTED, "frames beyond 2^32 rows (IdxSize is u32 in the reference too)");
        cudaStream_t st = ctx->stream, sc = ctx->stream_copy;
        g_alloc_pack = true;
        std::unique_ptr<PendingPack> P(new PendingPack);
        P->slot = (int)(ctx->pack_seq++ % ob_ctx::PACK_SLOTS);
        if (ob_design* prev = ctx->pack_slot_owner[P->slot]) pending_finish(prev, true);   // 8 packs in flight: complete the oldest
        P->h_flags = ctx->h_pack_flags + 4 * P->slot;
        P->h_flags[0] = P->h_flags[1] = P->h_flags[2] = P->h_flags[3] = 0;
        OB_CUDA(cudaEventCreate(&P->ev_begin)); OB_CUDA(cudaEventCreate(&P->ev_h2d_end));
        StagedFrame& sf = P->sf;
        sf.n = n; sf.n_cont = f->n_cont; sf.n_cat = f->n_cat; sf.weighted = f->weights != nullptr;
        sf.cols.resize(f->n_cont); sf.cats.resize(f->n_cat);
        const size_t nn = (size_t)std::max<int64_t>(n, 1);
        for (int c = 0; c < f->n_cont; ++c) sf.cols[c].alloc(sizeof(double) * nn);
        for (int q = 0; q < f->n_cat; ++q) sf.cats[q].alloc(sizeof(int32_t) * nn);
        sf.y.alloc(sizeof(double) * nn); sf.grp.alloc(nn);
        if (sf.weighted) sf.w.alloc(sizeof(double) * nn);
        std::vector<const double*> h_cont(std::max(sf.n_cont, 1), nullptr);
        std::vector<const int32_t*> h_cat(std::max(sf.n_cat, 1), nullptr);
        for (int c = 0; c < sf.n_cont; ++c) h_cont[c] = sf.cols[c].as<double>();
        for (int q = 0; q < sf.n_cat; ++q) h_cat[q] = sf.cats[q].as<int32_t>();
        P->d_cont_ptrs.alloc(sizeof(void*) * h_cont.size()); P->d_cat_ptrs.alloc(sizeof(void*) * h_cat.size());
        P->d_levels.alloc(sizeof(int32_t) * std::max(sf.n_cat, 1)); P->d_dstart.alloc(sizeof(int32_t) * dummy_start.size());
        OB_CUDA(cudaMemcpyAsync(P->d_cont_ptrs.p, h_cont.data(), sizeof(void*) * h_cont.size(), cudaMemcpyHostToDevice, st));
        OB_CUDA(cudaMemcpyAsync(P->d_cat_ptrs.p, h_cat.data(), sizeof(void*) * h_cat.size(), cudaMemcpyHostToDevice, st));
        if (sf.n_cat) OB_CUDA(cudaMemcpyAsync(P->d_levels.p, f->cat_levels, sizeof(int32_t) * sf.n_cat, cudaMemcpyHostToDevice, st));
        OB_CUDA(cudaMemcpyAsync(P->d_dstart.p, dummy_start.data(), sizeof(int32_t) * dummy_start.size(), cudaMemcpyHostToDevice, st));

        PackArgs pa;
        pa.n = n; pa.n_cont = sf.n_cont; pa.n_cat = sf.n_cat;
        pa.d_cont = P->d_cont_ptrs.as<const double*>(); pa.d_cat = P->d_cat_ptrs.as<const int32_t*>();
        pa.d_cat_levels = P->d_levels.as<int32_t>(); pa.d_dummy_start = P->d_dstart.as<int32_t>();
        pa.d_y = sf.y.as<double>(); pa.d_w = nullptr; pa.d_group = sf.grp.as<uint8_t>();   // weights are checked by the pack kernel
        pa.K = K; pa.ldx = design_ldx(K + 1);

        // group column first: it alone fixes the group sizes and where every row goes
        const int nblk = pack_num_blocks(n);
        P->d_bc.alloc(sizeof(long long) * 2 * (size_t)std::max(nblk, 1)); P->d_tot.alloc(sizeof(long long) * 2); P->d_flags.alloc(sizeof(int) * 4);
        OB_CUDA(cudaMemsetAsync(P->d_flags.p, 0, sizeof(int) * 4, st));
        OB_CUDA(cudaEventRecord(P->ev_begin, st));
        if (n) OB_CUDA(cudaMemcpyAsync(sf.grp.p, f->group, (size_t)n, cudaMemcpyHostToDevice, st));
        pack_count_scan(pa, P->d_bc.as<long long>(), P->d_tot.as<long long>(), P->d_flags.as<int>(), st);
        // row chunks (multiples of the pack kernel's 128-row blocks): a first quarter the Gram contraction can start on,
        // then the rest; small frames go in one piece
        std::vector<int> cut = {0};
        if (n >= (1 << 18)) cut.push_back(nblk / 4);
        cut.push_back(nblk);
        const int nchunks = (int)cut.size() - 1;
        long long tot[2];
        std::vector<long long> base(2 * (size_t)nchunks, 0);
        OB_CUDA(cudaMemcpyAsync(tot, P->d_tot.p, sizeof tot, cudaMemcpyDeviceToHost, st));
        for (int c = 1; c < nchunks; ++c)     // rows of each group before the chunk boundary = exclusive scan at that block
            OB_CUDA(cudaMemcpyAsync(&base[2 * (size_t)c], P->d_bc.as<long long>() + 2 * (size_t)cut[c], 2 * sizeof(long long), cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));

        std::unique_ptr<ob_design, void (*)(ob_design*)> d(new ob_design, ob_design_destroy);
        design_register(ctx, d.get()); d->stream = ctx->stream; d->device = ctx->device; d->K = K; d->n_cont = sf.n_cont; d->V = K + 1; d->ldx = pa.ldx;
        d->weighted = sf.weighted;
        d->cat_levels.assign(f->cat_levels, f->cat_levels + sf.n_cat);
        d->n_frame = n;
        PackWindow win{};
        const PackWindow* winp = nullptr;
        if (!shard) {
            alloc_group(ctx, d->g[0], tot[0], d->ldx, d->weighted, false);
            alloc_group(ctx, d->g[1], tot[1], d->ldx, d->weighted, false);
        } else {
            // where this slice's rows sit inside the whole groups: every rank's group sizes, shape word and frame rows
            const int world = comm->world, me = comm->rank;
            std::vector<long long> mine = {tot[0], tot[1], ((long long)K << 32) | ((long long)sf.n_cont << 1) | (sf.weighted ? 1 : 0), (long long)n};
            DevBuf d_mine(sizeof(long long) * 4), d_all(sizeof(long long) * 4 * world);
            OB_CUDA(cudaMemcpyAsync(d_mine.p, mine.data(), sizeof(long long) * 4, cudaMemcpyHostToDevice, st));
            comm->allgather(d_mine.p, d_all.p, sizeof(long long) * 4, st);
            std::vector<long long> all(4 * (size_t)world);
            OB_CUDA(cudaMemcpyAsync(all.data(), d_all.p, sizeof(long long) * 4 * world, cudaMemcpyDeviceToHost, st));
            OB_CUDA(cudaStreamSynchronize(st));
            P->ex_frame_off.assign((size_t)world + 1, 0);
            for (int r = 0; r < world; ++r) {
                if (all[4 * r + 2] != mine[2]) fail(OB_ERR_INVALID_ARG, "ranks disagree on the design shape (K, n_cont, weights)");
                P->ex_frame_off[r + 1] = P->ex_frame_off[r] + all[4 * r + 3];
            }
            if (P->ex_frame_off[world] > 0xFFFFFFFFll) fail(OB_ERR_UNSUPPORTED, "frames beyond 2^32 rows");
            d->n_frame = P->ex_frame_off[world];
            d->world = world; d->rank = me;
            win.src_add = (uint32_t)P->ex_frame_off[me];
            for (int g = 0; g < 2; ++g) {
                std::vector<long long> off((size_t)world + 1, 0);
                for (int r = 0; r < world; ++r) off[r + 1] = off[r] + all[4 * r + g];
                std::vector<RowShard> plan((size_t)world);
                for (int t = 0; t < world; ++t) plan[t] = row_shard(off[world], t, world);
                alloc_group(ctx, d->g[g], plan[me].n_local, d->ldx, d->weighted, false);
                d->g[g].shard = plan[me];
                const long long rb = plan[me].row_begin, re = rb + plan[me].n_local;
                const long long lo_cnt = std::max<long long>(0, std::min<long long>(rb, off[me + 1]) - off[me]);   // my rows below my shard
                const long long hi_cnt = std::max<long long>(0, off[me + 1] - std::max<long long>(re, off[me]));   // my rows above it
                win.shift[g] = off[me] - rb; win.n_local[g] = plan[me].n_local;
                win.lo_add[g] = rb - off[me];                                             // low-side rows keep their slice order from 0
                win.hi_base[g] = lo_cnt - std::max<long long>(0, off[me] - re);             // high-side rows follow the low-side ones
                const size_t erows = (size_t)std::max<long long>(lo_cnt + hi_cnt, 1);
                P->EX[g].alloc(sizeof(double) * erows * d->ldx); P->Ew[g].alloc(sizeof(double) * erows); P->Esrc[g].alloc(sizeof(uint32_t) * erows);
                win.EX[g] = P->EX[g].as<double>(); win.Ew[g] = P->Ew[g].as<double>(); win.Esrc[g] = P->Esrc[g].as<uint32_t>();
                // exchange tables: rows[src * world + dst]; what a rank keeps (src == dst) was written in place by the pack
                P->ex_rows[g].assign((size_t)world * world, 0); P->ex_send_row[g].assign((size_t)world, 0); P->ex_recv_row[g].assign((size_t)world, 0);
                for (int sidx = 0; sidx < world; ++sidx)
                    for (int t = 0; t < world; ++t) {
                        if (sidx == t) continue;
                        const long long lo = std::max<long long>(off[sidx], plan[t].row_begin);
                        const long long hi = std::min<long long>(off[sidx + 1], plan[t].row_begin + plan[t].n_local);
                        P->ex_rows[g][(size_t)sidx * world + t] = hi > lo ? (size_t)(hi - lo) : 0;
                    }
                for (int r = 0; r < world; ++r) {
                    // position inside MY export buffer of the first row I hold for rank r: low-side rows keep their slice
                    // order from 0, high-side rows follow at lo_cnt
                    const long long first = std::max<long long>(off[me], plan[r].row_begin);      // global position
                    P->ex_send_row[g][r] = (size_t)std::max<long long>(0, first < rb ? first - off[me] : lo_cnt + (first - std::max<long long>(re, off[me])));
                    P->ex_recv_row[g][r] = (size_t)std::max<long long>(0, std::max<long long>(off[r], rb) - rb);                  // inside my shard
                }
                // rows the pack writes in place: [ready_lo, ..) in shard-local coordinates
                P->ready_lo[g] = std::min<long long>(std::max<long long>(win.shift[g], 0), plan[me].n_local);
            }
            P->exchange_pending = true;
            winp = &win;
        }
        pa.d_w = sf.weighted ? sf.w.as<double>() : nullptr;
        // an error from here on must not release buffers the copy stream is still writing
        struct CopyJoin { cudaStream_t s; bool armed = true; ~CopyJoin() { if (armed) cudaStreamSynchronize(s); } } copy_join{sc};
        // the copy stream starts once the allocations and the pad-row memsets are ordered before it
        cudaEvent_t ev_alloc = nullptr;
        OB_CUDA(cudaEventCreateWithFlags(&ev_alloc, cudaEventDisableTiming));
        OB_CUDA(cudaEventRecord(ev_alloc, st));
        OB_CUDA(cudaStreamWaitEvent(sc, ev_alloc, 0));
        cudaEventDestroy(ev_alloc);
        P->chunk_done.resize((size_t)nchunks, nullptr);
        for (int c = 0; c < nchunks; ++c) {
            const int64_t r0 = (int64_t)cut[c] * PACK_BLOCK_ROWS, r1 = std::min<int64_t>(n, (int64_t)cut[c + 1] * PACK_BLOCK_ROWS);
            const size_t rows = (size_t)std::max<int64_t>(r1 - r0, 0);
            if (rows) {
                for (int k = 0; k < f->n_cont; ++k)
                    OB_CUDA(cudaMemcpyAsync(sf.cols[k].as<double>() + r0, f->cont[k] + r0, sizeof(double) * rows, cudaMemcpyHostToDevice, sc));
                for (int q = 0; q < f->n_cat; ++q)
                    OB_CUDA(cudaMemcpyAsync(sf.cats[q].as<int32_t>() + r0, f->cat_codes[q] + r0, sizeof(int32_t) * rows, cudaMemcpyHostToDevice, sc));
                OB_CUDA(cudaMemcpyAsync(sf.y.as<double>() + r0, f->outcome + r0, sizeof(double) * rows, cudaMemcpyHostToDevice, sc));
                if (sf.weighted) OB_CUDA(cudaMemcpyAsync(sf.w.as<double>() + r0, f->weights + r0, sizeof(double) * rows, cudaMemcpyHostToDevice, sc));
            }
            if (c == nchunks - 1) OB_CUDA(cudaEventRecord(P->ev_h2d_end, sc));
            pack_scatter(pa, P->d_bc.as<long long>(), d->g[0], d->g[1], P->d_flags.as<int>(), sc, cut[c], cut[c + 1], winp);
            if (c == nchunks - 1) OB_CUDA(cudaMemcpyAsync(P->h_flags, P->d_flags.p, sizeof(int) * 4, cudaMemcpyDeviceToHost, sc));
            OB_CUDA(cudaEventCreate(&P->chunk_done[(size_t)c]));
            OB_CUDA(cudaEventRecord(P->chunk_done[(size_t)c], sc));
            for (int g = 0; g < 2; ++g) {
                const long long q = c == nchunks - 1 ? tot[g] : base[2 * (size_t)(c + 1) + g];     // slice rows of the group packed so far
                // in place up to shard row q + shift (clamped); the last chunk of a shard still lacks the imported rows
                P->rows_ready[g].push_back(shard ? std::min<long long>(std::max<long long>(q + win.shift[g], P->ready_lo[g]), win.n_local[g]) : q);
            }
        }
        ctx->pack_slot_owner[P->slot] = d.get();
        d->pending = P.release();
        copy_join.armed = false;
        *out = d.release();
    });
}

ob_status ob_design_pack_async(ob_ctx* ctx, const ob_frame_view* f, ob_design** out) { return pack_async_impl(ctx, f, false, out); }

ob_status ob_design_pack_row_shard_async(ob_ctx* ctx, const ob_frame_view* slice, ob_design** out) { return pack_async_impl(ctx, slice, true, out); }

ob_status ob_design_wait(ob_ctx* ctx, ob_design* d) {
    if (!ctx || !d) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] { design_ready(d); });
}

// ---- ingest: null filter + dictionary coding on the device (SURVEY.md 8f-1) ----
ob_status ob_ingest_begin(ob_ctx* ctx, const ob_raw_frame* f, ob_ingest** out) {
    if (!ctx || !f || !out) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        if (f->n < 0 || f->n_cont < 0 || f->n_cat < 0) fail(OB_ERR_INVALID_ARG, "bad frame shape");
        if (f->n_cont + 2 > INGEST_MAX_COLS || f->n_cat + 1 > INGEST_MAX_COLS) fail(OB_ERR_UNSUPPORTED, "too many columns");
        if (f->n && (!f->outcome.data || !f->group.codes)) fail(OB_ERR_INVALID_ARG, "null frame column");
        if (f->n > 0xFFFFFFFFll) fail(OB_ERR_UNSUPPORTED, "frames beyond 2^32 rows");
        cudaStream_t st = ctx->stream;
        g_alloc_pack = true;
        std::unique_ptr<ob_ingest> ing(new ob_ingest);
        ing->ctx = ctx;
        StagedFrame& sf = ing->sf;
        const int64_t n = f->n;
        sf.n = n; sf.n_cont = f->n_cont; sf.n_cat = f->n_cat; sf.weighted = f->weights.data != nullptr;
        sf.cols.resize(f->n_cont); sf.cats.resize(f->n_cat);
        Timer t_h2d(st, &sf.ms_h2d);
        IngestScanArgs a{};
        a.n = n;
        auto add_f64 = [&](const ob_raw_f64& c, DevBuf& dst) {
            if (n && !c.data) fail(OB_ERR_INVALID_ARG, "null numeric column");
            stage_column(dst, c.data, n, st);
            if (f->nan_is_null) a.nan_cols[a.n_nan++] = dst.as<double>();
            if (c.valid) {
                ing->valid.emplace_back();
                stage_column(ing->valid.back(), c.valid, n, st);
                a.valid[a.n_valid++] = ing->valid.back().as<uint8_t>();
            }
        };
        ing->valid.reserve((size_t)f->n_cont + 2);
        for (int c = 0; c < f->n_cont; ++c) add_f64(f->cont[c], sf.cols[c]);
        add_f64(f->outcome, sf.y);
        if (sf.weighted) add_f64(f->weights, sf.w);
        ing->present.resize((size_t)f->n_cat + 1);
        auto add_dict = [&](const ob_raw_dict& c, DevBuf& dst) {
            if (n && !c.codes) fail(OB_ERR_INVALID_ARG, "null dictionary column");
            if (c.dict_size < 0) fail(OB_ERR_INVALID_ARG, "negative dictionary size");
            stage_column(dst, c.codes, n, st);
            DevBuf& pr = ing->present[(size_t)a.n_dict];
            pr.alloc((size_t)std::max(c.dict_size, 1));
            OB_CUDA(cudaMemsetAsync(pr.p, 0, pr.bytes, st));
            a.codes[a.n_dict] = dst.as<int32_t>(); a.dict_size[a.n_dict] = c.dict_size; a.present[a.n_dict] = pr.as<uint8_t>();
            ing->dict_size.push_back(c.dict_size);
            ++a.n_dict;
        };
        for (int q = 0; q < f->n_cat; ++q) add_dict(f->cat[q], sf.cats[q]);
        add_dict(f->group, ing->group_codes);
        t_h2d.stop();
        ing->row_valid.alloc((size_t)std::max<int64_t>(n, 1));
        sf.grp.alloc((size_t)std::max<int64_t>(n, 1));
        DevBuf d_kept(sizeof(long long)), d_flags(sizeof(int) * 4);
        OB_CUDA(cudaMemsetAsync(d_kept.p, 0, sizeof(long long), st));
        OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
        a.row_valid = ing->row_valid.as<uint8_t>(); a.kept = d_kept.as<long long>(); a.flags = d_flags.as<int>();
        ingest_scan_launch(a, st);
        long long kept = 0; int flags[4];
        OB_CUDA(cudaMemcpyAsync(&kept, d_kept.p, sizeof kept, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
        ing->h_present.resize(ing->present.size());
        for (size_t c = 0; c < ing->present.size(); ++c) {
            ing->h_present[c].assign((size_t)std::max(ing->dict_size[c], 1), 0);
            OB_CUDA(cudaMemcpyAsync(ing->h_present[c].data(), ing->present[c].p, ing->h_present[c].size(), cudaMemcpyDeviceToHost, st));
        }
        OB_CUDA(cudaStreamSynchronize(st));
        t_h2d.collect();
        if (flags[0] & 1) fail(OB_ERR_POLARS, "Polars error: dictionary code outside the dictionary");
        ing->kept = kept;
        *out = ing.release();
    });
}

ob_status ob_ingest_rows_kept(const ob_ingest* ing, int64_t* rows_kept) {
    if (!ing || !rows_kept) return OB_ERR_INVALID_ARG;
    *rows_kept = ing->kept;
    return OB_OK;
}

ob_status ob_ingest_presence(const ob_ingest* ing, int32_t column, uint8_t* present_out) {
    if (!ing || !present_out) return OB_ERR_INVALID_ARG;
    const int n_cat = ing->sf.n_cat;
    const int c = column < 0 ? n_cat : column;            // -1 = the group column
    if (c < 0 || c > n_cat) return OB_ERR_INVALID_ARG;
    memcpy(present_out, ing->h_present[(size_t)c].data(), (size_t)ing->dict_size[(size_t)c]);
    return OB_OK;
}

ob_status ob_ingest_finish(ob_ctx* ctx, ob_ingest* ing, const int32_t* group_map, const int32_t* const* cat_remap,
                           const int32_t* cat_levels, ob_design** out) {
    if (!ctx || !ing || !group_map || !out || ing->ctx != ctx) return OB_ERR_INVALID_ARG;
    *out = nullptr;
    return guarded(ctx, [&] {
        cudaStream_t st = ctx->stream;
        g_alloc_pack = true;
        StagedFrame& sf = ing->sf;
        if (sf.n_cat && (!cat_remap || !cat_levels)) fail(OB_ERR_INVALID_ARG, "categorical remap tables missing");
        IngestApplyArgs a{};
        a.n = sf.n; a.n_cat = sf.n_cat;
        std::vector<int32_t> remap;
        for (int q = 0; q < sf.n_cat; ++q) {
            a.remap_off[q] = (int)remap.size();
            remap.insert(remap.end(), cat_remap[q], cat_remap[q] + ing->dict_size[(size_t)q]);
            a.cat_codes[q] = sf.cats[q].as<int32_t>();
        }
        const int gsize = ing->dict_size[(size_t)sf.n_cat];
        DevBuf d_remap(sizeof(int32_t) * std::max<size_t>(remap.size(), 1)), d_gmap(sizeof(int32_t) * std::max(gsize, 1)), d_flags(sizeof(int) * 4);
        if (!remap.empty()) OB_CUDA(cudaMemcpyAsync(d_remap.p, remap.data(), sizeof(int32_t) * remap.size(), cudaMemcpyHostToDevice, st));
        if (gsize) OB_CUDA(cudaMemcpyAsync(d_gmap.p, group_map, sizeof(int32_t) * gsize, cudaMemcpyHostToDevice, st));
        OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
        a.row_valid = ing->row_valid.as<uint8_t>(); a.group_codes = ing->group_codes.as<int32_t>();
        a.group_map = d_gmap.as<int32_t>(); a.remap = d_remap.as<int32_t>(); a.group_out = sf.grp.as<uint8_t>();
        a.flags = d_flags.as<int>();
        ingest_apply_launch(a, st);
        int flags[4];
        OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        if (flags[0] & 2) fail(OB_ERR_INVALID_ARG, "a categorical value present in the cleaned frame has no level code");
        *out = pack_staged(ctx, sf, cat_levels).release();
    });
}

void ob_ingest_destroy(ob_ingest* ing) {
    if (!ing) return;
    cudaSetDevice(ing->ctx->device);
    g_alloc_ctx = ing->ctx;            // DevBuf destructors free on the owning context's stream
    delete ing;
}

ob_status ob_design_download(ob_ctx* ctx, const ob_design* d, double* Xa, double* ya, double* wa,
                             double* Xb, double* yb, double* wb) {
    if (!ctx || !d) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        double* Xs[2] = {Xa, Xb}; double* ys[2] = {ya, yb}; double* ws[2] = {wa, wb};
        for (int g = 0; g < 2; ++g) {
            const GroupData& G = d->g[g];
            if (G.n == 0) continue;
            if (Xs[g]) OB_CUDA(cudaMemcpy2DAsync(Xs[g], sizeof(double) * d->K, G.X, sizeof(double) * d->ldx,
                                                 sizeof(double) * d->K, (size_t)G.n, cudaMemcpyDeviceToHost, ctx->stream));
            if (ys[g]) OB_CUDA(cudaMemcpy2DAsync(ys[g], sizeof(double), G.X + d->K, sizeof(double) * d->ldx, sizeof(double),
                                                 (size_t)G.n, cudaMemcpyDeviceToHost, ctx->stream));
            if (ws[g] && G.w) OB_CUDA(cudaMemcpyAsync(ws[g], G.w, sizeof(double) * (size_t)G.n, cudaMemcpyDeviceToHost, ctx->stream));
        }
        OB_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

ob_status ob_design_update_outcome(ob_ctx* ctx, ob_design* d, const double* y_frame, int64_t n_frame) {
    if (!ctx || !d || !y_frame) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        if (n_frame != d->n_frame) fail(OB_ERR_INVALID_ARG, "outcome length differs from the frame the design was packed from");
        if (!d->g[0].src || !d->g[1].src) fail(OB_ERR_UNSUPPORTED, "this design carries no frame-row map (gathered design)");
        g_alloc_pack = true;
        ++d->y_gen;
        DevBuf d_y(sizeof(double) * (size_t)std::max<int64_t>(n_frame, 1));
        OB_CUDA(cudaMemcpyAsync(d_y.p, y_frame, sizeof(double) * (size_t)n_frame, cudaMemcpyHostToDevice, ctx->stream));
        for (int g = 0; g < 2; ++g) {
            update_outcome_launch(d->g[g], d->K, d->ldx, d_y.as<double>(), ctx->stream);
            if (d->g[g].y_raw) { cudaFreeAsync(d->g[g].y_raw, ctx->stream); d->g[g].y_raw = nullptr; }   // new raw outcome
            d->T = 1; d->V = d->K + 1;      // back to a single outcome column
            if (d->g[g].hk_Xm) hk_mask_launch(d->g[g].X, d->g[g].hk_sel, d->g[g].hk_Xm, d->g[g].n_pad, d->ldx, ctx->stream);
        }
        OB_CUDA(cudaStreamSynchronize(ctx->stream));
    });
}

// One RIF outcome per quantile, side by side in the design rows (columns K .. K+T-1): a quantile sweep then costs ONE
// pass of the Gram contraction -- X'WX is shared, only K more columns of X'Wy per extra quantile -- instead of T.
ob_status ob_design_apply_rif_multi(ob_ctx* ctx, ob_design* d, const double* taus, int32_t n_tau) {
    if (!ctx || !d || !taus) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        if (n_tau < 1 || n_tau > 8) fail(OB_ERR_INVALID_ARG, "1 to 8 quantiles per pass");
        // a row shard: the order statistics, the bandwidth and the density need all rows of a group -- the library's
        // communicator all-reduces the radix histograms and the leaf partial sums (a collective: every rank calls)
        Comm* comm = d->world > 1 ? ctx->comm.get() : nullptr;
        if (d->world > 1 && (!comm || comm->world != d->world || comm->rank != d->rank))
            fail(OB_ERR_NCCL, "row-sharded design needs ob_comm_init_* on this context with the same world/rank");
        if (d->K + n_tau > MAX_DESIGN_COLS) fail(OB_ERR_UNSUPPORTED, "design plus outcome columns wider than 280");
        cudaStream_t st = ctx->stream;
        const int K = d->K;
        ++d->y_gen;
        const int ldx_new = std::max(d->ldx, design_ldx(K + n_tau));
        for (int g = 0; g < 2; ++g) {
            GroupData& G = d->g[g];
            if (!G.y_raw && G.n > 0) {   // first transform: keep the raw outcome, later quantiles start from it again
                OB_CUDA(cudaMallocFromPoolAsync((void**)&G.y_raw, sizeof(double) * (size_t)G.n, ctx->pool_design, st));
                OB_CUDA(cudaMemcpy2DAsync(G.y_raw, sizeof(double), G.X + K, sizeof(double) * d->ldx, sizeof(double), (size_t)G.n,
                                          cudaMemcpyDeviceToDevice, st));
            }
            if (ldx_new != d->ldx) {     // make room for the outcome columns: rows move to a wider stride, once
                const size_t xbytes = sizeof(double) * (size_t)G.n_pad * ldx_new;
                double* X2 = nullptr;
                OB_CUDA(cudaMallocFromPoolAsync((void**)&X2, xbytes, ctx->pool_design, st));
                relayout_launch(G.X, d->ldx, X2, ldx_new, G.n_pad, K, st);
                cudaFreeAsync(G.X, st); G.X = X2;
                if (G.Xs) {
                    cudaFreeAsync(G.Xs, st); G.Xs = nullptr;
                    OB_CUDA(cudaMallocFromPoolAsync((void**)&G.Xs, xbytes, ctx->pool_design, st));
                }
            }
        }
        d->ldx = ldx_new; d->T = n_tau; d->V = K + n_tau;
        for (int g = 0; g < 2; ++g) {
            const size_t sb = rif_scratch_bytes(d->g[g].n);
            DevBuf scratch(sb);
            for (int t = 0; t < n_tau; ++t) rif_transform(d->g[g], K + t, d->ldx, taus[t], scratch.p, sb, st, comm);
            scale_rows_launch(d->g[g], d->ldx, st);   // the RIF outcomes are weighted like any outcome
            if (d->g[g].hk_Xm) hk_mask_launch(d->g[g].X, d->g[g].hk_sel, d->g[g].hk_Xm, d->g[g].n_pad, d->ldx, st);
            OB_CUDA(cudaStreamSynchronize(st));
        }
    });
}

ob_status ob_design_apply_rif(ob_ctx* ctx, ob_design* d, double tau) { return ob_design_apply_rif_multi(ctx, d, &tau, 1); }

ob_status ob_design_num_outcomes(const ob_design* d, int32_t* n_out) {
    if (!d || !n_out) return OB_ERR_INVALID_ARG;
    *n_out = d->T;
    return OB_OK;
}

int32_t ob_num_stats_heckman(int32_t K, int32_t K1) { return 5 + 2 * (K + 1) + K1; }

ob_status ob_design_selection_cols(const ob_design* d, int32_t* k1_out) {
    if (!d || !k1_out) return OB_ERR_INVALID_ARG;
    *k1_out = d->K1;
    return OB_OK;
}

ob_status ob_design_attach_selection(ob_ctx* ctx, ob_design* d, const ob_selection_view* sv, int64_t n_frame) {
    if (!ctx || !d || !sv) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        if (sv->n_pred < 0 || sv->n_pred + 1 > HK_MAX_SEL) fail(OB_ERR_UNSUPPORTED, "at most 7 selection predictors");
        if (!sv->outcome || (sv->n_pred && !sv->pred)) fail(OB_ERR_INVALID_ARG, "null selection column");
        if (n_frame != d->n_frame) fail(OB_ERR_INVALID_ARG, "selection columns differ in length from the frame the design was packed from");
        if (d->world > 1) fail(OB_ERR_UNSUPPORTED, "Heckman selection on a row-sharded design");
        if (d->cl_strata != OB_CLUSTER_NONE)
            fail(OB_ERR_UNSUPPORTED, "Heckman selection on a clustered design: its estimator assumes constant group sizes (detach the clusters)");
        if (d->weighted) fail(OB_ERR_UNSUPPORTED, "Heckman selection with sample weights (the reference's estimator ignores them, estimation.rs:132-133)");
        if (!d->g[0].src || !d->g[1].src) fail(OB_ERR_UNSUPPORTED, "this design carries no frame-row map");
        cudaStream_t st = ctx->stream;
        g_alloc_pack = true;
        const int K1 = 1 + sv->n_pred;
        const size_t nn = (size_t)std::max<int64_t>(n_frame, 1);
        std::vector<DevBuf> cols((size_t)sv->n_pred);
        std::vector<const double*> h_ptrs((size_t)std::max(sv->n_pred, 1), nullptr);
        for (int j = 0; j < sv->n_pred; ++j) {
            if (!sv->pred[j]) fail(OB_ERR_INVALID_ARG, "null selection predictor column");
            cols[(size_t)j].alloc(sizeof(double) * nn);
            OB_CUDA(cudaMemcpyAsync(cols[(size_t)j].p, sv->pred[j], sizeof(double) * (size_t)n_frame, cudaMemcpyHostToDevice, st));
            h_ptrs[(size_t)j] = cols[(size_t)j].as<double>();
        }
        DevBuf d_out(sizeof(double) * nn), d_ptrs(sizeof(void*) * h_ptrs.size()), d_flags(sizeof(int) * 4);
        OB_CUDA(cudaMemcpyAsync(d_out.p, sv->outcome, sizeof(double) * (size_t)n_frame, cudaMemcpyHostToDevice, st));
        OB_CUDA(cudaMemcpyAsync(d_ptrs.p, h_ptrs.data(), sizeof(void*) * h_ptrs.size(), cudaMemcpyHostToDevice, st));
        OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
        for (int g = 0; g < 2; ++g) {
            GroupData& G = d->g[g];
            if (G.hk_Z) { cudaFreeAsync(G.hk_Z, st); G.hk_Z = nullptr; }
            if (G.hk_sel) { cudaFreeAsync(G.hk_sel, st); G.hk_sel = nullptr; }
            if (G.hk_Xm) { cudaFreeAsync(G.hk_Xm, st); G.hk_Xm = nullptr; }
            OB_CUDA(cudaMallocFromPoolAsync((void**)&G.hk_Z, sizeof(double) * (size_t)std::max<int64_t>(G.n, 1) * K1, ctx->pool_design, st));
            OB_CUDA(cudaMallocFromPoolAsync((void**)&G.hk_sel, (size_t)G.n_pad, ctx->pool_design, st));
            OB_CUDA(cudaMallocFromPoolAsync((void**)&G.hk_Xm, sizeof(double) * (size_t)G.n_pad * d->ldx, ctx->pool_design, st));
            OB_CUDA(cudaMemsetAsync(G.hk_sel, 0, (size_t)G.n_pad, st));
            hk_gather_launch(G.src, G.n, K1, d_ptrs.as<const double*>(), d_out.as<double>(), G.hk_Z, G.hk_sel, d_flags.as<int>(), st);
            hk_mask_launch(G.X, G.hk_sel, G.hk_Xm, G.n_pad, d->ldx, st);
        }
        int flags[4];
        OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        d->K1 = K1;
        if (flags[0]) { d->K1 = 0; fail(OB_ERR_INVALID_GROUP, "Invalid group variable: Selection outcome contains nulls"); }   // estimation.rs:179-185
    });
}

// Cluster labels (cluster.cu): the codes of the kept rows are gathered through each group's frame-row map, checked on the
// device, and the codes present in a stratum numbered in ascending order (the units).  The design is changed only once
// everything has succeeded.
ob_status ob_design_attach_clusters(ob_ctx* ctx, ob_design* d, const int32_t* codes_frame, int64_t n_frame, int32_t n_codes,
                                    int32_t strata) {
    if (!ctx || !d) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        cudaStream_t st = ctx->stream;
        if (strata != OB_CLUSTER_NONE && strata != OB_CLUSTER_BY_GROUP && strata != OB_CLUSTER_JOINT)
            fail(OB_ERR_INVALID_ARG, "strata must be OB_CLUSTER_NONE, OB_CLUSTER_BY_GROUP or OB_CLUSTER_JOINT");
        auto install = [&](uint32_t* const uid[2], int st_new, const int64_t units[2]) {
            for (int g = 0; g < 2; ++g) {
                if (d->g[g].uid) cudaFreeAsync(d->g[g].uid, st);
                d->g[g].uid = uid[g];
                d->cl_units[g] = units[g];
            }
            d->cl_strata = st_new;
            ++d->x_gen;              // the resamples change: a Gram cache refills
        };
        if (strata == OB_CLUSTER_NONE) {
            uint32_t* none[2] = {nullptr, nullptr};
            const int64_t zero[2] = {0, 0};
            install(none, OB_CLUSTER_NONE, zero);
            return;
        }
        if (n_frame != d->n_frame) fail(OB_ERR_INVALID_ARG, "cluster codes differ in length from the frame the design was packed from");
        if (!codes_frame && n_frame > 0) fail(OB_ERR_INVALID_ARG, "null cluster codes");
        if (n_codes < 1) fail(OB_ERR_INVALID_ARG, "n_codes must be at least 1");
        if (d->world > 1) fail(OB_ERR_UNSUPPORTED, "clusters on a row-sharded design (mode N): a unit's rows may sit on several ranks");
        if (d->K1 > 0)
            fail(OB_ERR_UNSUPPORTED, "clusters on a design with a selection equation: the Heckman estimator assumes constant group sizes");
        if (!d->g[0].src || !d->g[1].src) fail(OB_ERR_UNSUPPORTED, "this design carries no frame-row map");
        g_alloc_pack = true;
        struct Uids {               // the new maps, released unless installed
            uint32_t* p[2] = {nullptr, nullptr}; cudaStream_t st;
            ~Uids() { for (auto q : p) if (q) cudaFreeAsync(q, st); }
        } nu{{nullptr, nullptr}, st};
        for (int g = 0; g < 2; ++g)
            OB_CUDA(cudaMallocFromPoolAsync((void**)&nu.p[g], sizeof(uint32_t) * (size_t)std::max<int64_t>(d->g[g].n, 1), ctx->pool_design, st));
        const int nstrata = strata == OB_CLUSTER_JOINT ? 1 : 2;
        DevBuf d_codes(sizeof(int32_t) * (size_t)std::max<int64_t>(n_frame, 1)), d_flags(sizeof(int) * 4);
        DevBuf d_present((size_t)nstrata * n_codes), d_unit(sizeof(uint32_t) * (size_t)nstrata * n_codes), d_units(sizeof(long long) * 2);
        if (n_frame) OB_CUDA(cudaMemcpyAsync(d_codes.p, codes_frame, sizeof(int32_t) * (size_t)n_frame, cudaMemcpyHostToDevice, st));
        OB_CUDA(cudaMemsetAsync(d_flags.p, 0, d_flags.bytes, st));
        OB_CUDA(cudaMemsetAsync(d_present.p, 0, d_present.bytes, st));
        OB_CUDA(cudaMemsetAsync(d_units.p, 0, d_units.bytes, st));
        for (int g = 0; g < 2; ++g) {
            const int m = nstrata == 1 ? 0 : g;
            cluster_gather_launch(d_codes.as<int32_t>(), d->g[g].src, d->g[g].n, n_codes, nu.p[g],
                                  d_present.as<uint8_t>() + (size_t)m * n_codes, d_flags.as<int>(), st);
        }
        for (int m = 0; m < nstrata; ++m)
            cluster_scan_launch(d_present.as<uint8_t>() + (size_t)m * n_codes, n_codes, d_unit.as<uint32_t>() + (size_t)m * n_codes,
                                d_units.as<long long>() + m, st);
        for (int g = 0; g < 2; ++g)
            cluster_remap_launch(nu.p[g], d->g[g].n, d_unit.as<uint32_t>() + (size_t)(nstrata == 1 ? 0 : g) * n_codes, st);
        int flags[4];
        long long units[2];
        OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaMemcpyAsync(units, d_units.p, sizeof units, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        if (flags[0]) fail(OB_ERR_INVALID_ARG, "cluster code outside [0, n_codes) on a row the design holds");
        if (nstrata == 1) units[1] = units[0];
        const int64_t u[2] = {units[0], units[1]};
        install(nu.p, strata, u);
        nu.p[0] = nu.p[1] = nullptr;
    });
}

ob_status ob_design_clusters(const ob_design* d, int32_t* strata, int64_t* units_a, int64_t* units_b) {
    if (!d) return OB_ERR_INVALID_ARG;
    if (strata) *strata = d->cl_strata;
    if (units_a) *units_a = d->cl_units[0];
    if (units_b) *units_b = d->cl_units[1];
    return OB_OK;
}

}  // extern "C"

namespace {

// ob_bootstrap_run on a design with a selection equation: the Heckman two-step estimator per replicate (heckman.cu).
void heckman_run(ob_ctx* ctx, const ob_design* d, const ob_boot_opts* o, ob_result* res) {
    cudaStream_t st = ctx->stream;
    const int K = d->K, Ka = K + 1, K1 = d->K1;
    if (o->ref_kind < 0 || o->ref_kind > 3) fail(OB_ERR_INVALID_ARG, "ref_kind out of range");
    if (o->ref_kind == OB_REF_POOLED)
        fail(OB_ERR_UNSUPPORTED, "Pooled / Neumark reference coefficients with Heckman selection: the reference's pooled regression has K "
                                 "coefficients, the Heckman fits K + 1 (builder.rs:548-589 vs estimation.rs:139-141)");
    if (d->T != 1) fail(OB_ERR_UNSUPPORTED, "Heckman selection on a multi-outcome design");
    if (d->world > 1) fail(OB_ERR_UNSUPPORTED, "Heckman selection on a row-sharded design");
    RepRange rr = replicate_range(ctx, d, o);
    // mode R inside the library, as for the OLS path: this rank's contiguous share of the global replicate ids
    if (rr.shard_reps) { ob_replicate_shard(o->reps, ctx->comm->world, ctx->comm->rank, &rr.rb, &rr.re); rr.nrep = rr.re - rr.rb; }
    if (d->g[0].n == 0 || d->g[1].n == 0) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: One group has no data");
    int count_bytes = rr.count_bytes;
    const int S = ob_num_stats_heckman(K, K1);

    res->ms_counts = res->ms_gram = res->ms_solve = res->ms_reduce = res->ms_total = res->ms_gram_kernel = res->ms_comm = 0.0;
    res->gpu_launches = 0; res->n_ok = 0;
    Timer t_total(st, &res->ms_total);
    const int64_t slots = 1 + rr.nrep, panels_total = (slots + BM - 1) / BM;
    const bool want_beta = res->rep_beta_a || res->rep_beta_b || res->beta_a || res->beta_b;
    DevBuf d_stats(sizeof(double) * (size_t)slots * S), d_status(sizeof(int) * (size_t)slots);
    DevBuf d_ba(want_beta ? sizeof(double) * (size_t)slots * Ka : 0), d_bb(want_beta ? sizeof(double) * (size_t)slots * Ka : 0);
    const size_t PE = 3 * (size_t)Ka + 2 * (size_t)K1 + 1;
    DevBuf d_point(sizeof(double) * PE), d_flags(sizeof(int) * 4), d_lut(2 * counts_lut_bytes()), d_nact(sizeof(int));
    const int ntiles = gram_ntiles(K, 1), Pld = gram_pld(K, 1);
    const int64_t n_pad[2] = {d->g[0].n_pad, d->g[1].n_pad}, n_g[2] = {d->g[0].n, d->g[1].n};
    const int nch[2] = {hk_num_chunks(n_g[0]), hk_num_chunks(n_g[1])};
    const int nacc_p = K1 + K1 * (K1 + 1) / 2, nacc_t = K1 + 5;
    const int64_t leaves = (int64_t)d->g[0].shard.segs + d->g[1].shard.segs;

    std::vector<double> point(PE);
    auto run_batches = [&] {
    for (int attempt = 0; attempt < 2; ++attempt) {
        size_t free_b = 0, total_b = 0;
        OB_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const double budget = o->max_workspace_bytes > 0 ? (double)o->max_workspace_bytes : 0.6 * ((double)free_b + (double)pool_idle_bytes(ctx));
        const double per_panel = (double)(n_pad[0] + n_pad[1]) * BM * (count_bytes + 8.0) +        // counts + L = c * IMR
                                 (rr.index_mode ? (double)(n_g[0] + n_g[1]) * BM * 4.0 : 0.0) + 2.0 * BM * Pld * 8.0 +
                                 (double)leaves * ntiles * (BM * BN * 8.0) +
                                 (double)(nch[0] + nch[1]) * BM * 8.0 * std::max(std::max(nacc_p, nacc_t), K);
        int64_t ppb = std::max<int64_t>(1, std::min<int64_t>((int64_t)std::floor(budget / per_panel), panels_total));
        DevBuf d_C[2], d_L[2], d_idx[2], d_colsum(sizeof(long long) * 2 * (size_t)ppb * BM);
        DevBuf d_gamma[2], d_active[2], d_pst[2], d_terms[2], d_xterm[2];
        for (int g = 0; g < 2; ++g) {
            d_C[g].alloc((size_t)ppb * n_pad[g] * BM * count_bytes);
            d_L[g].alloc(sizeof(double) * (size_t)ppb * n_pad[g] * BM);
            d_gamma[g].alloc(sizeof(double) * (size_t)ppb * BM * HK_MAX_SEL);
            d_active[g].alloc(sizeof(int) * (size_t)ppb * BM); d_pst[g].alloc(sizeof(int) * (size_t)ppb * BM);
            d_terms[g].alloc(sizeof(double) * (size_t)nacc_t * ppb * BM); d_xterm[g].alloc(sizeof(double) * (size_t)K * ppb * BM);
        }
        DevBuf d_part(sizeof(double) * (size_t)std::max(nch[0], nch[1]) * ppb * BM * std::max(std::max(nacc_p, nacc_t), K));
        DevBuf d_gram(sizeof(double) * 2 * (size_t)ppb * BM * Pld), d_partials, d_pairs, d_colmap;
        const GramColumns gcols = gram_columns(K, 1, d->n_cont, d->cat_levels);
        {
            d_pairs.alloc(sizeof(uint16_t) * gcols.pairs.size());
            d_colmap.alloc(sizeof(int32_t) * gcols.colmap.size());
            OB_CUDA(cudaMemcpyAsync(d_pairs.p, gcols.pairs.data(), sizeof(uint16_t) * gcols.pairs.size(), cudaMemcpyHostToDevice, st));
            OB_CUDA(cudaMemcpyAsync(d_colmap.p, gcols.colmap.data(), sizeof(int32_t) * gcols.colmap.size(), cudaMemcpyHostToDevice, st));
            OB_CUDA(cudaStreamSynchronize(st));
        }
        GramPlan plan; int64_t plan_panels = -1;
        bool saturated = false;
        for (int64_t p0 = 0; p0 < panels_total && !saturated; p0 += ppb) {
            const Batch b(p0, ppb, panels_total, slots, rr.rb);
            const int64_t pn = b.pn, bslots = b.bslots, slots_pad = pn * BM;
            OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
            // (2) replicate generation: the same multiplicity matrix as the OLS path
            Timer t_counts(st, &res->ms_counts);
            res->gpu_launches += generate_counts(d, o, b, count_bytes, ppb, d_C, d_idx, d_colsum, d_lut, d_flags.as<int>(), nullptr, nullptr, st);
            t_counts.stop();

            // (3a) probit of every slot, both groups: Fisher scoring until every slot has converged (<= 100 steps)
            Timer t_solve(st, &res->ms_solve);
            for (int g = 0; g < 2; ++g) {
                const HkGroup hg{d->g[g].hk_Z, d->g[g].hk_sel, n_g[g], n_pad[g]};
                std::vector<int> act((size_t)slots_pad, 0);
                for (int64_t s_ = 0; s_ < bslots; ++s_) act[(size_t)s_] = 1;
                OB_CUDA(cudaMemcpyAsync(d_active[g].p, act.data(), sizeof(int) * (size_t)slots_pad, cudaMemcpyHostToDevice, st));
                OB_CUDA(cudaMemsetAsync(d_gamma[g].p, 0, sizeof(double) * (size_t)slots_pad * HK_MAX_SEL, st));     // probit.rs:41: start at 0
                OB_CUDA(cudaMemsetAsync(d_pst[g].p, 0, sizeof(int) * (size_t)slots_pad, st));
                for (int it = 0; it < 100; ++it) {                                                                  // heckman.rs:46: probit(.., 100, 1e-6)
                    OB_CUDA(cudaMemsetAsync(d_nact.p, 0, sizeof(int), st));
                    hk_probit_accum_launch(hg, K1, d_C[g].p, count_bytes, (int)pn, d_gamma[g].as<double>(), d_active[g].as<int>(), slots_pad, d_part.as<double>(), st);
                    hk_probit_update_launch(d_part.as<double>(), nch[g], (int)pn, K1, bslots, 1e-6, it == 99, d_gamma[g].as<double>(), d_active[g].as<int>(),
                                            d_pst[g].as<int>(), d_nact.as<int>(), st);
                    res->gpu_launches += 2;
                    int nact = 0;
                    OB_CUDA(cudaMemcpyAsync(&nact, d_nact.p, sizeof(int), cudaMemcpyDeviceToHost, st));
                    OB_CUDA(cudaStreamSynchronize(st));
                    if (nact == 0) break;
                }
                // (3b) inverse Mills ratio sums and the cross term X'(c IMR)
                hk_terms_launch(hg, d->g[g].X, d->ldx, K, K1, d_C[g].p, count_bytes, (int)pn, d_gamma[g].as<double>(), d_L[g].as<double>(), d_part.as<double>(), st);
                hk_reduce_launch(d_part.as<double>(), nch[g], (int)pn, nacc_t, d_terms[g].as<double>(), slots_pad, st);
                hk_xterm_launch(hg, d->g[g].X, d->ldx, K, (int)pn, d_L[g].as<double>(), d_part.as<double>(), st);
                hk_reduce_launch(d_part.as<double>(), nch[g], (int)pn, K, d_xterm[g].as<double>(), slots_pad, st);
                res->gpu_launches += 4;
            }
            t_solve.stop();

            // (3c) X'CX, X'Cy and column sums over the selected rows: the DMMA contraction on the masked design
            if (plan_panels != pn) {
                plan = gram_make_plan(K, 1, d->ldx, (int)pn, d->g, count_bytes, ctx->num_sms, gcols);
                plan_panels = pn;
                d_partials.alloc(sizeof(double) * (size_t)std::max<int64_t>(plan.num_partials, 1) * BM * BN);
            }
            Timer t_gram(st, &res->ms_gram);
            GramArgs ga;
            for (int g = 0; g < 2; ++g) { ga.X[g] = d->g[g].hk_Xm; ga.C[g] = d_C[g].p; }
            ga.count_bytes = count_bytes; ga.partials = d_partials.as<double>(); ga.d_pairs = d_pairs.as<uint16_t>(); ga.d_colmap = d_colmap.as<int32_t>(); ga.gram = d_gram.as<double>();
            ga.tail_mi = b.tail_mi();
            gram_launch(plan, ga, st);
            res->gpu_launches += 2;
            t_gram.stop();

            // (4) augmented solves + decomposition
            Timer t_solve2(st, &res->ms_solve);
            HkSolveArgs sa;
            sa.gram = d_gram.as<double>(); sa.slots_pad = slots_pad; sa.Pld = Pld; sa.slots = bslots; sa.K = K; sa.K1 = K1; sa.ref_kind = o->ref_kind;
            for (int g = 0; g < 2; ++g) { sa.terms[g] = d_terms[g].as<double>(); sa.xterm[g] = d_xterm[g].as<double>(); sa.gamma[g] = d_gamma[g].as<double>(); sa.pstatus[g] = d_pst[g].as<int>(); }
            sa.na = (double)n_g[0]; sa.nb = (double)n_g[1]; sa.S = S;
            sa.stats = d_stats.as<double>() + (size_t)b.slot_lo * S; sa.status = d_status.as<int>() + b.slot_lo;
            sa.beta_a = want_beta ? d_ba.as<double>() + (size_t)b.slot_lo * Ka : nullptr;
            sa.beta_b = want_beta ? d_bb.as<double>() + (size_t)b.slot_lo * Ka : nullptr;
            sa.point_extra = p0 == 0 ? d_point.as<double>() : nullptr;
            hk_solve_launch(sa, st);
            res->gpu_launches += 1;
            t_solve2.stop();
            int flags[4];
            OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
            OB_CUDA(cudaStreamSynchronize(st));
            t_counts.collect(); t_solve.collect(); t_gram.collect(); t_solve2.collect();
            saturated = check_batch_flags(flags, count_bytes, o->count_bits, d->ldx);
        }
        if (!saturated) break;
        count_bytes = 2;
        res->ms_counts = res->ms_gram = res->ms_solve = 0.0;
    }
    int point_status = 0;
    OB_CUDA(cudaMemcpyAsync(&point_status, d_status.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaMemcpyAsync(point.data(), d_point.p, sizeof(double) * PE, cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaStreamSynchronize(st));
    if (point_status != OB_OK)
        fail((ob_status)point_status, point_status == OB_ERR_INVALID_GROUP ? "Invalid group variable: No observed outcomes in group" : status_text(point_status));
    };   // run_batches
    agree_on_status(rr.shard_reps ? ctx->comm.get() : nullptr, st, run_batches, "another rank of the replicate-sharded run failed");
    res->total_gap = point[3 * Ka + 2 * K1];
    if (res->xa_mean) memcpy(res->xa_mean, point.data(), sizeof(double) * Ka);
    if (res->xb_mean) memcpy(res->xb_mean, point.data() + Ka, sizeof(double) * Ka);
    if (res->beta_star) memcpy(res->beta_star, point.data() + 2 * Ka, sizeof(double) * Ka);
    if (res->sel_gamma_a) memcpy(res->sel_gamma_a, point.data() + 3 * Ka, sizeof(double) * K1);
    if (res->sel_gamma_b) memcpy(res->sel_gamma_b, point.data() + 3 * Ka + K1, sizeof(double) * K1);
    if (res->total_gap_multi) res->total_gap_multi[0] = res->total_gap;
    if (res->residuals_b) memset(res->residuals_b, 0, sizeof(double) * (size_t)d->g[1].n);      // estimation.rs:156-157: zeros
    if (res->point_stats) OB_CUDA(cudaMemcpyAsync(res->point_stats, d_stats.p, sizeof(double) * S, cudaMemcpyDeviceToHost, st));
    if (res->beta_a) OB_CUDA(cudaMemcpyAsync(res->beta_a, d_ba.p, sizeof(double) * Ka, cudaMemcpyDeviceToHost, st));
    if (res->beta_b) OB_CUDA(cudaMemcpyAsync(res->beta_b, d_bb.p, sizeof(double) * Ka, cudaMemcpyDeviceToHost, st));
    const int64_t reps_all = rr.shard_reps ? o->reps : rr.nrep;
    DevBuf d_gstats, d_gstatus, d_gba, d_gbb;
    const double* stats_rows = d_stats.as<double>() + S;
    const int* status_rows = d_status.as<int>() + 1;
    const double* ba_rows = want_beta ? d_ba.as<double>() + Ka : nullptr;
    const double* bb_rows = want_beta ? d_bb.as<double>() + Ka : nullptr;
    if (rr.shard_reps) {      // replicate rows of all ranks, device to device, into global replicate order
        Timer t_c(st, &res->ms_comm);
        Comm* cm = ctx->comm.get();
        stats_rows = allgather_shards(cm, o->reps, S, stats_rows, d_gstats, st);
        status_rows = allgather_shards(cm, o->reps, 1, status_rows, d_gstatus, st);
        if (res->rep_beta_a) ba_rows = allgather_shards(cm, o->reps, Ka, ba_rows, d_gba, st);
        if (res->rep_beta_b) bb_rows = allgather_shards(cm, o->reps, Ka, bb_rows, d_gbb, st);
        t_c.stop(); OB_CUDA(cudaStreamSynchronize(st)); t_c.collect();
    }
    if (!o->skip_reduce) {
        double* dst[5] = {res->std_err, res->p_value, res->ci_lower, res->ci_upper, res->t_stat};
        reduce_to_host(st, stats_rows, status_rows, reps_all, S, d_stats.as<double>(), dst, &res->n_ok, &res->ms_reduce);
        res->gpu_launches += 1;
    }
    if (reps_all > 0) {
        if (res->rep_stats) OB_CUDA(cudaMemcpyAsync(res->rep_stats, stats_rows, sizeof(double) * (size_t)reps_all * S, cudaMemcpyDeviceToHost, st));
        if (res->rep_status) OB_CUDA(cudaMemcpyAsync(res->rep_status, status_rows, sizeof(int) * (size_t)reps_all, cudaMemcpyDeviceToHost, st));
        if (res->rep_beta_a) OB_CUDA(cudaMemcpyAsync(res->rep_beta_a, ba_rows, sizeof(double) * (size_t)reps_all * Ka, cudaMemcpyDeviceToHost, st));
        if (res->rep_beta_b) OB_CUDA(cudaMemcpyAsync(res->rep_beta_b, bb_rows, sizeof(double) * (size_t)reps_all * Ka, cudaMemcpyDeviceToHost, st));
    }
    t_total.stop();
    OB_CUDA(cudaStreamSynchronize(st));
    t_total.collect();
}


// ob_mm_run: the Machado-Mata passes (mm.cu) over columns of the same multiplicity matrix as the OLS bootstrap.
void mm_run(ob_ctx* ctx, const ob_design* d, const ob_mm_opts* o, ob_mm_result* res) {
    cudaStream_t st = ctx->stream;
    const int K = d->K, sims = o->simulations, nq = o->n_quantiles, S = 3 * nq;
    if (sims < 1 || sims > MM_MAX_SIMS) fail(OB_ERR_INVALID_ARG, "simulations must be in [1, 4096]");
    if (nq < 1 || nq > 1024 || !o->quantiles) fail(OB_ERR_INVALID_ARG, "n_quantiles must be in [1, 1024]");
    if (K > MM_MAX_COLS) fail(OB_ERR_UNSUPPORTED, "Machado-Mata: more than 47 design columns");
    if (d->weighted) fail(OB_ERR_UNSUPPORTED, "Machado-Mata on a weighted design (QuantileDecompositionBuilder has no weights)");
    if (d->T != 1 || d->g[0].y_raw || d->g[1].y_raw) fail(OB_ERR_UNSUPPORTED, "Machado-Mata needs the raw outcome (the design carries RIF outcomes)");
    if (d->world > 1) fail(OB_ERR_UNSUPPORTED, "Machado-Mata on a row-sharded design");
    if (d->g[0].n < 2 || d->g[1].n < 2) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: One group has insufficient data");   // :210-214
    // Mode R inside the library shards the REGRESSIONS, not the passes: every rank builds the multiplicity columns and the
    // streams of all passes (cheap), solves a contiguous balanced share of each batch's (pass, simulation, group) problems,
    // the coefficients are all-gathered device to device, and effects + reduction run on every rank.  With the builder's
    // default of 20 passes a pass-level split over 8 GPUs would leave ranks with 4 or 3 passes (the point pass included)
    // against 2.6 on average; the problem-level split is even to one regression.
    const RepRange rr = replicate_range(ctx, d, o);
    const bool draws_given = o->draw_a != nullptr || o->draw_b != nullptr;
    if (draws_given && (!o->draw_a || !o->draw_b)) fail(OB_ERR_INVALID_ARG, "simulated-row stream needs both draw_a and draw_b");
    if (draws_given && rr.nrep > 0 && !rr.index_mode)
        fail(OB_ERR_INVALID_ARG, "draw_a / draw_b are positions in the resampled frames: they need the explicit resample stream idx_a / idx_b");
    // Without draw_a / draw_b the simulated rows of an explicit resample are drawn natively (mm_streams_kernel), by
    // rejection with acceptance min(c_i, 64) / 64: that is row i with probability c_i / n only while every multiplicity is
    // <= 64.  Native multiplicities never get there; an explicit stream that does is refused.
    if (rr.index_mode && !draws_given) {
        for (int g = 0; g < 2; ++g) {
            const uint32_t* ix = g == 0 ? o->idx_a : o->idx_b;
            const int64_t n = d->g[g].n;
            std::vector<uint32_t> cnt((size_t)n);
            for (int64_t r = rr.rb; r < rr.re; ++r) {
                std::fill(cnt.begin(), cnt.end(), 0u);
                for (int64_t i = 0; i < n; ++i) {
                    const uint32_t row = ix[(size_t)r * n + i];
                    if (row < n && ++cnt[row] > 64)
                        fail(OB_ERR_UNSUPPORTED, "an explicit resample draws a row more than 64 times: the native simulated-row "
                                                 "draw is exact only up to 64; pass draw_a / draw_b explicitly");
                }
            }
        }
    }
    for (int q = 0; q < nq; ++q)
        if (!(o->quantiles[q] >= 0.0 && o->quantiles[q] <= 1.0)) fail(OB_ERR_INVALID_ARG, "target quantiles must lie in [0, 1]");
    int count_bytes = rr.count_bytes;

    res->ms_counts = res->ms_qr = res->ms_effects = res->ms_reduce = res->ms_total = 0.0;
    res->gpu_launches = 0; res->n_ok = 0;
    res->qr_total = res->qr_vertex = res->qr_approx = res->qr_failed = res->qr_iterations = 0;
    Timer t_total(st, &res->ms_total);
    const int64_t slots = 1 + rr.nrep, panels_total = (slots + BM - 1) / BM;
    const int64_t n_pad[2] = {d->g[0].n_pad, d->g[1].n_pad}, n_g[2] = {d->g[0].n, d->g[1].n};
    DevBuf d_stats(sizeof(double) * (size_t)slots * S), d_status(sizeof(int) * (size_t)slots);
    DevBuf d_q(sizeof(double) * (size_t)nq), d_flags(sizeof(int) * 4), d_lut(2 * counts_lut_bytes()), d_counter(sizeof(int));
    OB_CUDA(cudaMemcpyAsync(d_q.p, o->quantiles, sizeof(double) * (size_t)nq, cudaMemcpyHostToDevice, st));
    const int64_t stride = (std::max(n_g[0], n_g[1]) + 31) / 32 * 32;
    std::vector<int> h_info;
    std::vector<double> h_taus, h_pbetas;
    std::vector<uint32_t> h_rows[2];

    auto run_batches = [&] {
    for (int attempt = 0; attempt < 2; ++attempt) {
        size_t free_b = 0, total_b = 0;
        OB_CUDA(cudaMemGetInfo(&free_b, &total_b));
        const double budget = o->max_workspace_bytes > 0 ? (double)o->max_workspace_bytes : 0.6 * ((double)free_b + (double)pool_idle_bytes(ctx));
        // blocks in flight: two per SM unless their iterate slabs (6 vectors of the larger group) would take more than
        // half of the budget
        const double slab = 8.0 * mm_state_vectors() * (double)stride;
        int grid = ctx->num_sms * mm_blocks_per_sm(K, std::max(n_g[0], n_g[1]));
        grid = (int)std::max<int64_t>(1, std::min<int64_t>(grid, (int64_t)std::floor(0.5 * budget / slab)));
        const double per_panel = (double)(n_pad[0] + n_pad[1]) * BM * count_bytes + (rr.index_mode ? (double)(n_g[0] + n_g[1]) * BM * 4.0 : 0.0) +
                                 (double)BM * sims * (2.0 * K * 8.0 + 2.0 * 4.0 + 8.0 + 8.0);
        int64_t ppb = std::max<int64_t>(1, std::min<int64_t>((int64_t)std::floor((budget - grid * slab) / per_panel), panels_total));
        DevBuf d_C[2], d_idx[2], d_colsum(sizeof(long long) * 2 * (size_t)ppb * BM);
        for (int g = 0; g < 2; ++g) d_C[g].alloc((size_t)ppb * n_pad[g] * BM * count_bytes);
        const size_t bs_max = (size_t)std::min<int64_t>(ppb * BM, slots);
        DevBuf d_state(sizeof(double) * (size_t)mm_state_vectors() * (size_t)stride * (size_t)grid);
        DevBuf d_betas(sizeof(double) * 2 * bs_max * sims * K), d_info(sizeof(int) * 2 * bs_max * sims);
        DevBuf d_betas_all, d_info_all;      // mode R: every rank's share of them (allgather_shards)
        DevBuf d_taus(sizeof(double) * bs_max * sims), d_rows_a(sizeof(uint32_t) * bs_max * sims), d_rows_b(sizeof(uint32_t) * bs_max * sims);
        bool saturated = false;
        for (int64_t p0 = 0; p0 < panels_total && !saturated; p0 += ppb) {
            const Batch b(p0, ppb, panels_total, slots, rr.rb);
            const int64_t bslots = b.bslots;
            OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
            // (1) the passes' multiplicity columns: the same replicate generation as ob_bootstrap_run
            Timer t_counts(st, &res->ms_counts);
            res->gpu_launches += generate_counts(d, o, b, count_bytes, ppb, d_C, d_idx, d_colsum, d_lut, d_flags.as<int>(), nullptr, nullptr, st);
            t_counts.stop();
            // (2) random quantiles and simulated rows of the batch's passes
            MmArgs ma;
            for (int g = 0; g < 2; ++g) { ma.X[g] = d->g[g].X; ma.C[g] = d_C[g].p; ma.n[g] = n_g[g]; ma.n_pad[g] = n_pad[g]; }
            ma.ldx = d->ldx; ma.K = K; ma.count_bytes = count_bytes; ma.sims = sims; ma.slots = bslots;
            ma.taus = d_taus.as<double>(); ma.state = d_state.as<double>(); ma.state_stride = stride;
            ma.betas = d_betas.as<double>(); ma.info = d_info.as<int>(); ma.counter = d_counter.as<int>();
            // global pass ids: 0 = point estimates (slot 0 of the first batch), r + 1 = replicate r.  With a replicate shard
            // the batch's slots 1.. are replicates rb.., so consecutive only from slot 1 on: the point slot is special-cased
            const int64_t gpass0 = b.rep0 + 1;        // pass id slot 0 of this batch WOULD have as a replicate slot
            if (!o->taus || !draws_given) {
                mm_streams_launch(ma, gpass0, b.first_slot, o->seed, d_taus.as<double>(), d_rows_a.as<uint32_t>(), d_rows_b.as<uint32_t>(), st);
                res->gpu_launches += 1;
            }
            if (o->taus) {      // explicit quantiles: rows of the [(reps + 1) x sims] table, row 0 = point pass, row r + 1 = replicate r
                h_taus.resize((size_t)bslots * sims);
                for (int64_t s_ = 0; s_ < bslots; ++s_) {
                    const int64_t pass = (p0 == 0 && s_ == 0) ? 0 : b.rep0 + s_ + 1;
                    memcpy(h_taus.data() + (size_t)s_ * sims, o->taus + (size_t)pass * sims, sizeof(double) * (size_t)sims);
                }
                OB_CUDA(cudaMemcpyAsync(d_taus.p, h_taus.data(), sizeof(double) * h_taus.size(), cudaMemcpyHostToDevice, st));
            }
            if (draws_given) {  // positions in the resampled frame -> original rows through the resample stream
                for (int g = 0; g < 2; ++g) {
                    const uint32_t* dr = g == 0 ? o->draw_a : o->draw_b;
                    const uint32_t* ix = g == 0 ? o->idx_a : o->idx_b;
                    h_rows[g].resize((size_t)bslots * sims);
                    for (int64_t s_ = 0; s_ < bslots; ++s_) {
                        const int64_t pass = (p0 == 0 && s_ == 0) ? 0 : b.rep0 + s_ + 1;
                        for (int i = 0; i < sims; ++i) {
                            const uint32_t pos = dr[(size_t)pass * sims + i];
                            if ((int64_t)pos >= n_g[g]) fail(OB_ERR_INVALID_ARG, "simulated-row position out of range");
                            h_rows[g][(size_t)s_ * sims + i] = pass == 0 ? pos : ix[(size_t)(pass - 1) * n_g[g] + pos];
                            if ((int64_t)h_rows[g][(size_t)s_ * sims + i] >= n_g[g]) fail(OB_ERR_INVALID_ARG, "resample index out of range");
                        }
                    }
                    OB_CUDA(cudaMemcpyAsync((g == 0 ? d_rows_a : d_rows_b).p, h_rows[g].data(), sizeof(uint32_t) * h_rows[g].size(), cudaMemcpyHostToDevice, st));
                }
            }
            // (3) the quantile regressions: one block per (group, pass, simulation)
            Timer t_qr(st, &res->ms_qr);
            OB_CUDA(cudaMemsetAsync(d_counter.p, 0, sizeof(int), st));
            const int64_t nprob = 2 * bslots * sims;
            ma.p_begin = 0; ma.p_end = nprob;
            if (rr.shard_reps) ob_replicate_shard(nprob, ctx->comm->world, ctx->comm->rank, &ma.p_begin, &ma.p_end);
            if (ma.p_end > ma.p_begin) {
                mm_qr_launch(ma, (int)std::min<int64_t>(grid, ma.p_end - ma.p_begin), st);
                res->gpu_launches += 1;
            }
            t_qr.stop();
            if (rr.shard_reps) {      // every rank's coefficients and status words, device to device, in problem order
                Comm* cm = ctx->comm.get();
                ma.betas = allgather_shards(cm, nprob, (size_t)K, d_betas.as<double>() + (size_t)ma.p_begin * K, d_betas_all, st);
                ma.info = allgather_shards(cm, nprob, 1, d_info.as<int>() + ma.p_begin, d_info_all, st);
            }
            // (4) simulation, empirical quantiles, effects
            Timer t_eff(st, &res->ms_effects);
            mm_effects_launch(ma, d_rows_a.as<uint32_t>(), d_rows_b.as<uint32_t>(), nq, d_q.as<double>(), d_stats.as<double>() + (size_t)b.slot_lo * S,
                              d_status.as<int>() + b.slot_lo, nullptr, st);
            res->gpu_launches += 1;
            t_eff.stop();
            int flags[4];
            h_info.resize((size_t)2 * bslots * sims);
            OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
            OB_CUDA(cudaMemcpyAsync(h_info.data(), ma.info, sizeof(int) * h_info.size(), cudaMemcpyDeviceToHost, st));
            if (p0 == 0 && (res->point_betas_a || res->point_betas_b)) {      // slot 0: [sims][2][K], groups interleaved
                h_pbetas.resize((size_t)2 * sims * K);
                OB_CUDA(cudaMemcpyAsync(h_pbetas.data(), ma.betas, sizeof(double) * h_pbetas.size(), cudaMemcpyDeviceToHost, st));
            }
            OB_CUDA(cudaStreamSynchronize(st));
            t_counts.collect(); t_qr.collect(); t_eff.collect();
            saturated = check_batch_flags(flags, count_bytes, o->count_bits, d->ldx);
            if (saturated) break;
            if (p0 == 0 && (res->point_betas_a || res->point_betas_b))
                for (int s_ = 0; s_ < sims; ++s_) {
                    if (res->point_betas_a) memcpy(res->point_betas_a + (size_t)s_ * K, h_pbetas.data() + ((size_t)2 * s_ + 0) * K, sizeof(double) * (size_t)K);
                    if (res->point_betas_b) memcpy(res->point_betas_b + (size_t)s_ * K, h_pbetas.data() + ((size_t)2 * s_ + 1) * K, sizeof(double) * (size_t)K);
                }
            for (size_t i = 0; i < h_info.size(); ++i) {
                const int st_ = h_info[i] & 0xff;
                ++res->qr_total;
                if (st_ == 0) ++res->qr_vertex; else if (st_ == 1) ++res->qr_approx; else ++res->qr_failed;
                res->qr_iterations += (h_info[i] >> 8) & 0xff;
            }
            if (p0 == 0)
                for (int s_ = 0; s_ < sims; ++s_) {
                    if (res->point_qr_info_a) res->point_qr_info_a[s_] = h_info[(size_t)2 * s_];
                    if (res->point_qr_info_b) res->point_qr_info_b[s_] = h_info[(size_t)2 * s_ + 1];
                }
        }
        if (!saturated) break;
        count_bytes = 2;
        res->ms_counts = res->ms_qr = res->ms_effects = 0.0;
        res->qr_total = res->qr_vertex = res->qr_approx = res->qr_failed = res->qr_iterations = 0;
    }
    int point_status = 0;
    OB_CUDA(cudaMemcpyAsync(&point_status, d_status.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    OB_CUDA(cudaStreamSynchronize(st));
    if (point_status != OB_OK)
        fail(OB_ERR_NALGEBRA, "Nalgebra error: Failed to estimate a sufficient number of quantile regressions.");      // :238-242
    };   // run_batches
    agree_on_status(rr.shard_reps ? ctx->comm.get() : nullptr, st, run_batches, "another rank of the replicate-sharded run failed");
    if (res->point_stats) OB_CUDA(cudaMemcpyAsync(res->point_stats, d_stats.p, sizeof(double) * S, cudaMemcpyDeviceToHost, st));
    const int64_t reps_all = rr.nrep;      // (mode R: every rank has computed the effects of all passes)
    const double* stats_rows = d_stats.as<double>() + S;
    const int* status_rows = d_status.as<int>() + 1;
    if (!o->skip_reduce) {
        double* dst[5] = {res->std_err, res->p_value, res->ci_lower, res->ci_upper, res->t_stat};
        reduce_to_host(st, stats_rows, status_rows, reps_all, S, d_stats.as<double>(), dst, &res->n_ok, &res->ms_reduce);
        res->gpu_launches += 1;
    }
    if (reps_all > 0) {
        if (res->rep_stats) OB_CUDA(cudaMemcpyAsync(res->rep_stats, stats_rows, sizeof(double) * (size_t)reps_all * S, cudaMemcpyDeviceToHost, st));
        if (res->rep_status) OB_CUDA(cudaMemcpyAsync(res->rep_status, status_rows, sizeof(int) * (size_t)reps_all, cudaMemcpyDeviceToHost, st));
    }
    t_total.stop();
    OB_CUDA(cudaStreamSynchronize(st));
    t_total.collect();
}

}  // namespace

extern "C" {

ob_status ob_mm_run(ob_ctx* ctx, const ob_design* d, const ob_mm_opts* o, ob_mm_result* res) {
    if (!ctx || !d || !o || !res) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        if (d->cl_strata != OB_CLUSTER_NONE)
            fail(OB_ERR_UNSUPPORTED, "Machado-Mata on a clustered design: its row draws assume constant group sizes (detach the clusters)");
        mm_run(ctx, d, o, res);
    });
}

// ob_bootstrap_run, and with a cache ob_bootstrap_run_cached: the batch loop contracts the full Gram (no cache, or a
// cache that is (re)filled), only its outcome columns (OB_CACHE_OUTCOME_ONLY: X'WX comes from the cache) or nothing
// (OB_CACHE_SOLVE_ONLY: the whole Gram comes from the cache, no multiplicities are generated)
// bayes: the Bayesian bootstrap (ob_bootstrap_run_bayes; bo null or null streams = the native stream)
static void bootstrap_body(ob_ctx* ctx, const ob_design* d, const ob_boot_opts* o, ob_gram_cache* cache, ob_result* res,
                           bool bayes = false, const ob_bayes_opts* bo = nullptr) {
        design_alive(d);
        const bool bayes_explicit = bayes && bo && (bo->wt_a || bo->wt_b);
        if (bayes) {
            if (d->cl_strata != OB_CLUSTER_NONE)
                fail(OB_ERR_UNSUPPORTED, "Bayesian bootstrap on a clustered design: cluster weights are not built (detach the clusters)");
            if (d->K1 > 0)
                fail(OB_ERR_UNSUPPORTED, "Bayesian bootstrap on a design with a selection equation: the Heckman estimator is not built for it");
            if (o->idx_a || o->idx_b)
                fail(OB_ERR_INVALID_ARG, "the Bayesian bootstrap takes no index stream (idx_a / idx_b must be NULL; explicit weights go in ob_bayes_opts)");
            if (o->count_bits != 0) fail(OB_ERR_INVALID_ARG, "the Bayesian bootstrap has fp32 weights: count_bits must be 0");
            if (!gram_fits(d->ldx, 4))
                fail(OB_ERR_UNSUPPORTED, "design too wide for the Bayesian bootstrap: K + outcomes <= 236 with fp32 weights");
            if (cache && bayes_explicit)
                fail(OB_ERR_UNSUPPORTED, "a Gram cache needs the native weight stream (explicit weight streams cannot be keyed)");
        }
        if (cache && d->K1 > 0) fail(OB_ERR_UNSUPPORTED, "a Gram cache does not apply to designs with a selection equation (Heckman)");
        if (cache && (o->idx_a || o->idx_b)) fail(OB_ERR_UNSUPPORTED, "a Gram cache needs the native resampling stream (explicit index streams cannot be keyed)");
        if (d->K1 > 0) {                 // a selection equation is attached: the Heckman two-step estimator per replicate
            design_ready(d);
            heckman_run(ctx, d, o, res);
            return;
        }
        cudaStream_t st = ctx->stream;
        const int K = d->K, T = d->T;
        const bool clustered = d->cl_strata != OB_CLUSTER_NONE;
        if (clustered && d->world > 1)
            fail(OB_ERR_UNSUPPORTED, "clusters on a row-sharded design (mode N): a unit's rows may sit on several ranks");
        if (o->ref_kind < 0 || o->ref_kind > 3) fail(OB_ERR_INVALID_ARG, "ref_kind out of range");
        if (o->n_norm < 0) fail(OB_ERR_INVALID_ARG, "negative n_norm");
        RepRange rr = replicate_range(ctx, d, o);
        if (o->shard_replicates && d->world > 1) fail(OB_ERR_INVALID_ARG, "shard_replicates on a row-sharded design (its communicator shards rows)");
        // mode R inside the library: this rank's contiguous share of the global replicate ids
        if (rr.shard_reps) { ob_replicate_shard(o->reps, ctx->comm->world, ctx->comm->rank, &rr.rb, &rr.re); rr.nrep = rr.re - rr.rb; }
        // builder.rs:431-435 (either group empty)
        if (d->g[0].shard.n_global == 0 || d->g[1].shard.n_global == 0) fail(OB_ERR_INVALID_GROUP, "Invalid group variable: One group has no data");
        // mode N: this design is one row shard; the context must carry the matching communicator
        Comm* comm = d->world > 1 ? ctx->comm.get() : nullptr;
        if (d->world > 1 && (!comm || comm->world != d->world || comm->rank != d->rank))
            fail(OB_ERR_NCCL, "row-sharded design needs ob_comm_init_* on this context with the same world/rank");
        const int world = d->world;
        int n_base = 0, n_idx = 0;
        // ---- Gram cache: what of this run the cache already holds ----
        int mode = OB_CACHE_NONE;
        const int rep_world = rr.shard_reps ? ctx->comm->world : 1, rep_rank = rr.shard_reps ? ctx->comm->rank : 0;
        if (cache) {
            const bool xx_hit = cache->xx_ok && cache->design_id == d->id && cache->x_gen == d->x_gen && cache->seed == o->seed &&
                                cache->reps == o->reps && cache->rep_begin == rr.rb && cache->rep_end == rr.re &&
                                cache->shard_reps == (rr.shard_reps ? 1 : 0) && cache->rep_world == rep_world && cache->rep_rank == rep_rank &&
                                cache->row_world == d->world && cache->row_rank == d->rank && cache->K == d->K && cache->bayes == bayes &&
                                !(o->count_bits == 8 && cache->count_bytes == 2);   // that run saturates 8-bit counts: let it fail
            mode = !xx_hit ? OB_CACHE_FILLED : (cache->y_ok && cache->y_gen == d->y_gen && cache->T == d->T) ? OB_CACHE_SOLVE_ONLY
                                                                                                           : OB_CACHE_OUTCOME_ONLY;
            // sharded runs: every rank must run the same collectives -- all take the least reuse any rank can do
            if (Comm* ac = rr.shard_reps ? ctx->comm.get() : comm) mode = allreduce_scalar(ac, mode, CommOp::MIN, st);
        }
        const bool solve_only = mode == OB_CACHE_SOLVE_ONLY, outcome_only = mode == OB_CACHE_OUTCOME_ONLY;
        for (int v = 0; v < o->n_norm; ++v) {
            n_base += o->norm_has_base[v] ? 1 : 0;
            if (o->norm_off[v + 1] < o->norm_off[v]) fail(OB_ERR_INVALID_ARG, "norm_off not monotone");
        }
        if (o->n_norm) n_idx = o->norm_off[o->n_norm];
        for (int t = 0; t < n_idx; ++t)
            if (o->norm_idx[t] < 0 || o->norm_idx[t] >= K) fail(OB_ERR_INVALID_ARG, "norm_idx outside the design");
        const int D = K + n_base, S = 5 + 2 * D;
        const int SE = T * S, KE = T * K;     // per slot: T outcomes (a quantile sweep) x S statistics / K coefficients
        int count_bytes = bayes ? 4 : rr.count_bytes;                                // fp32 weights: 4 bytes a cell
        if (outcome_only && o->count_bits == 0) count_bytes = cache->count_bytes;   // start where the fill ended
        if (bayes && rr.nrep > 0 && bayes_explicit && (!bo->wt_a || !bo->wt_b))
            fail(OB_ERR_INVALID_ARG, "an explicit weight stream needs both wt_a and wt_b");

        res->ms_counts = res->ms_gram = res->ms_solve = res->ms_reduce = res->ms_total = res->ms_gram_kernel = res->ms_comm = 0.0;
        res->gpu_launches = 0;
        res->n_ok = 0;
        Timer t_total(st, &res->ms_total);
        Trace tr;

        // ---- normalisation spec on the device ----
        const int nn = std::max(o->n_norm, 1);
        DevBuf d_nm(sizeof(int) * nn), d_noff(sizeof(int) * (nn + 1)), d_nidx(sizeof(int) * std::max(n_idx, 1)), d_nhb(sizeof(int) * nn);
        if (o->n_norm) {
            OB_CUDA(cudaMemcpyAsync(d_nm.p, o->norm_m, sizeof(int) * o->n_norm, cudaMemcpyHostToDevice, st));
            OB_CUDA(cudaMemcpyAsync(d_noff.p, o->norm_off, sizeof(int) * (o->n_norm + 1), cudaMemcpyHostToDevice, st));
            if (n_idx) OB_CUDA(cudaMemcpyAsync(d_nidx.p, o->norm_idx, sizeof(int) * n_idx, cudaMemcpyHostToDevice, st));
            OB_CUDA(cudaMemcpyAsync(d_nhb.p, o->norm_has_base, sizeof(int) * o->n_norm, cudaMemcpyHostToDevice, st));
        }

        // ---- outputs over all slots of this shard (slot 0 = point estimate) ----
        const int64_t slots = 1 + rr.nrep;
        const bool want_beta = res->rep_beta_a || res->rep_beta_b || res->beta_a || res->beta_b;
        DevBuf d_stats(sizeof(double) * (size_t)slots * SE), d_status(sizeof(int) * (size_t)slots);
        DevBuf d_ba(want_beta ? sizeof(double) * (size_t)slots * KE : 0), d_bb(want_beta ? sizeof(double) * (size_t)slots * KE : 0);
        const size_t PE = 5 * (size_t)K + 1;           // point_extra per outcome
        DevBuf d_point(sizeof(double) * PE * T);
        DevBuf d_flags(sizeof(int) * 4);

        // ---- cache storage: allocated by the filling call (and counted in its workspace budget) ----
        const int nx = gram_cache_xx_cells(K), ny = gram_cache_y_cells(K, T);
        size_t cache_new_bytes = 0;
        if (mode == OB_CACHE_FILLED) {
            cache_release_device(cache);
            cache->xx_bytes = sizeof(double) * 2 * (size_t)slots * nx;
            OB_CUDA(cudaMallocFromPoolAsync((void**)&cache->xx, cache->xx_bytes, ctx->pool_design, st));
            cache_new_bytes += cache->xx_bytes;
            if (clustered) {
                cache->rows_bytes = sizeof(long long) * 2 * (size_t)slots;
                OB_CUDA(cudaMallocFromPoolAsync((void**)&cache->rows, cache->rows_bytes, ctx->pool_design, st));
                cache_new_bytes += cache->rows_bytes;
            }
            if (bayes) {
                cache->esum_bytes = sizeof(double) * 2 * (size_t)slots;
                OB_CUDA(cudaMallocFromPoolAsync((void**)&cache->esum, cache->esum_bytes, ctx->pool_design, st));
                cache_new_bytes += cache->esum_bytes;
            }
        }
        if (mode == OB_CACHE_FILLED || outcome_only) {
            cache->y_ok = false;
            const size_t yb = sizeof(double) * 2 * (size_t)slots * ny;
            if (cache->yy_bytes != yb) {          // T changed
                if (cache->yy) cudaFreeAsync(cache->yy, st);
                cache->yy = nullptr; cache->yy_bytes = yb;
                OB_CUDA(cudaMallocFromPoolAsync((void**)&cache->yy, yb, ctx->pool_design, st));
                cache_new_bytes += yb;
            }
        }

        // ---- batch the multiplicity matrix by panels under the workspace budget ----
        const GramColumns gcols = solve_only ? GramColumns() : outcome_only ? gram_outcome_columns(K, T)
                                                                              : gram_columns(K, T, d->n_cont, d->cat_levels);
        const int ntiles = gcols.ntiles;
        const int Pld = gram_pld(K, T);
        const int64_t panels_total = (slots + BM - 1) / BM;
        const int64_t n_pad[2] = {d->g[0].n_pad, d->g[1].n_pad};
        const int64_t n_glob[2] = {d->g[0].shard.n_global, d->g[1].shard.n_global};
        // clustered: the unit matrices (padded like row matrices) and the lengths of an explicit stream, which draws units
        const int mats = clustered ? unit_mats(d) : 0;
        int64_t u_pad_all = 0;
        for (int m = 0; m < mats; ++m) u_pad_all += pad_rows(d->cl_units[m]);
        const int64_t idx_len = clustered ? d->cl_units[0] + (mats == 2 ? d->cl_units[1] : 0) : n_glob[0] + n_glob[1];
        int ranks_with_rows[2];
        for (int g = 0; g < 2; ++g)
            ranks_with_rows[g] = (d->g[g].shard.segs + d->g[g].shard.leaf_span - 1) / d->g[g].shard.leaf_span;
        const int64_t local_leaves = (int64_t)(d->g[0].shard.leaf_hi - d->g[0].shard.leaf_lo) +
                                     (d->g[1].shard.leaf_hi - d->g[1].shard.leaf_lo);
        // workspace of one panel: multiplicities (+ index stream), reduced Gram (+ the mode-N exchange), partial tiles, column
        // sums; a run that only solves needs the reduced Gram alone
        // (clustered: + the unit matrices and the per-slot row counts)
        // (Bayesian: + the per-slot weight sums, their leaf partials and mode-N exchange, and an explicit stream's upload)
        auto per_panel_bytes = [&](int cb) {
            double cl = clustered ? (solve_only ? 0.0 : (double)u_pad_all * BM * cb) + 2.0 * BM * 8.0 : 0.0;
            if (bayes)
                cl = 2.0 * BM * 8.0 + (solve_only ? 0.0 : (double)local_leaves * BM * 8.0 + (comm ? world + 1 : 0) * 2.0 * BM * 8.0 +
                                                          (bayes_explicit ? (double)(n_glob[0] + n_glob[1]) * BM * 4.0 : 0.0));
            if (solve_only) return 2.0 * BM * Pld * 8.0 + cl;
            return (double)(n_pad[0] + n_pad[1]) * BM * cb + (rr.index_mode ? (double)idx_len * BM * 4.0 : 0.0) +
                   2.0 * BM * Pld * 8.0 * (comm ? world + 2 : 1) + (double)local_leaves * ntiles * (BM * BN * 8.0) + 2.0 * BM * 8.0 + cl;
        };
        double budget = (double)o->max_workspace_bytes - (double)cache_new_bytes;
        if (o->max_workspace_bytes <= 0) {
            // Steady state (the same problem again): the context's pool already holds the whole workspace -> no device
            // query at all.  cudaMemGetInfo takes the driver's global lock and stalls for milliseconds whenever another
            // thread (NVML monitoring, for one) holds it.
            const double idle = (double)pool_idle_bytes(ctx);
            const double need_all = per_panel_bytes(count_bytes) * (double)panels_total;
            if (idle >= 1.02 * need_all) budget = 1.01 * need_all;      // every panel in one batch, from memory the pool holds
            else {
                size_t free_b = 0, total_b = 0;
                OB_CUDA(cudaMemGetInfo(&free_b, &total_b));
                budget = 0.6 * ((double)free_b + idle) - (double)cache_new_bytes;
            }
        }
        DevBuf d_lut(2 * counts_lut_bytes());

        std::vector<double> point(PE * T);
        cudaEvent_t ev_point = nullptr;          // recorded on st once the point estimate's coefficients are on the device
        struct EvGuard { cudaEvent_t& e; ~EvGuard() { if (e) cudaEventDestroy(e); } } ev_point_guard{ev_point};
        OB_CUDA(cudaEventCreateWithFlags(&ev_point, cudaEventDisableTiming));
        auto run_batches = [&] {
        for (int attempt = 0; attempt < 2; ++attempt) {  // second attempt only widens uint8 -> uint16 after saturation
            const double per_panel = per_panel_bytes(count_bytes);
            int64_t ppb = (int64_t)std::floor(budget / per_panel);
            ppb = std::max<int64_t>(1, std::min<int64_t>(ppb, panels_total));
            // every rank must cut the same batches: the collectives run once per batch
            if (comm) ppb = allreduce_scalar(comm, (long long)ppb, CommOp::MIN, st);
            tr.mark("setup", st, true);
            DevBuf d_C[2], d_idx[2], d_colsum, d_gram, d_gram_local, d_gathered, d_rows;
            ClusterWork cw;
            BayesWork bw;
            bw.ranks_with_rows[0] = ranks_with_rows[0]; bw.ranks_with_rows[1] = ranks_with_rows[1];
            const size_t gram_elems = 2 * (size_t)ppb * BM * Pld;      // [2][slots_pad][Pld]
            bool saturated = false;
            GramPlan plan; int64_t plan_panels = -1;
            DevBuf d_partials, d_pairs, d_colmap, d_cmap;
            auto allocate_workspace = [&] {
                if (!solve_only) {
                    if (!bayes) d_colsum.alloc(sizeof(long long) * 2 * (size_t)ppb * BM);
                    for (int g = 0; g < 2; ++g) d_C[g].alloc((size_t)ppb * n_pad[g] * BM * count_bytes);
                    for (int m = 0; m < mats; ++m) cw.U[m].alloc((size_t)ppb * pad_rows(d->cl_units[m]) * BM * count_bytes);
                }
                if (clustered) { d_rows.alloc(sizeof(long long) * 2 * (size_t)ppb * BM); cw.rows = d_rows.as<long long>(); }
                if (bayes) {
                    bw.esum.alloc(sizeof(double) * 2 * (size_t)ppb * BM);
                    if (!solve_only) bw.part.alloc(sizeof(double) * (size_t)std::max<int64_t>(local_leaves, 1) * ppb * BM);
                    if (!solve_only && comm) { bw.esum_local.alloc(sizeof(double) * 2 * (size_t)ppb * BM); bw.gathered.alloc(sizeof(double) * 2 * (size_t)ppb * BM * world); }
                }
                d_gram.alloc(sizeof(double) * gram_elems);
                if (cache) {
                    const std::vector<int32_t> cmap = gram_cache_map(K, T);
                    d_cmap.alloc(sizeof(int32_t) * cmap.size());
                    OB_CUDA(cudaMemcpyAsync(d_cmap.p, cmap.data(), sizeof(int32_t) * cmap.size(), cudaMemcpyHostToDevice, st));
                }
                if (solve_only) { OB_CUDA(cudaStreamSynchronize(st)); return; }
                if (comm) { d_gram_local.alloc(sizeof(double) * gram_elems); d_gathered.alloc(sizeof(double) * gram_elems * world); }
                plan = gram_make_plan(K, T, d->ldx, (int)std::min<int64_t>(ppb, panels_total), d->g, count_bytes, ctx->num_sms, gcols);
                plan_panels = plan.panels;
                d_partials.alloc(sizeof(double) * (size_t)std::max<int64_t>(plan.num_partials, 1) * BM * BN);
                d_pairs.alloc(sizeof(uint16_t) * gcols.pairs.size());
                d_colmap.alloc(sizeof(int32_t) * gcols.colmap.size());
                OB_CUDA(cudaMemcpyAsync(d_pairs.p, gcols.pairs.data(), sizeof(uint16_t) * gcols.pairs.size(), cudaMemcpyHostToDevice, st));
                OB_CUDA(cudaMemcpyAsync(d_colmap.p, gcols.colmap.data(), sizeof(int32_t) * gcols.colmap.size(), cudaMemcpyHostToDevice, st));
                OB_CUDA(cudaStreamSynchronize(st));
            };
            // row shards: a rank whose workspace cannot be had (its GPU is shared, say) must not leave its peers waiting in the
            // first collective of the batch loop -- all ranks agree on the outcome of the allocation phase
            agree_on_status(comm, st, allocate_workspace, "another rank of the row-sharded run could not allocate its workspace");

            tr.mark("workspace + pair table", st, true);
            for (int64_t p0 = 0; p0 < panels_total && !saturated; p0 += ppb) {
                const Batch b(p0, ppb, panels_total, slots, rr.rb);
                const int64_t pn = b.pn, bslots = b.bslots;
                OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));

                // (2) replicate generation (none when the cache holds every Gram cell of these slots)
                Timer t_counts(st, &res->ms_counts);
                if (!solve_only && bayes)
                    res->gpu_launches += generate_weights(d, o, bo, b, d_C, bw, d_flags.as<int>(), comm, &res->ms_comm, st);
                else if (!solve_only)
                    res->gpu_launches += generate_counts(d, o, b, count_bytes, ppb, d_C, d_idx, d_colsum, d_lut, d_flags.as<int>(), comm,
                                                         &res->ms_comm, st, clustered ? &cw : nullptr);
                t_counts.stop();
                tr.mark("counts", st, true);

                // (3) Gram / cross-product contraction
                if (!solve_only && plan_panels != pn) {
                    plan = gram_make_plan(K, T, d->ldx, (int)pn, d->g, count_bytes, ctx->num_sms, gcols);
                    plan_panels = pn;
                    d_partials.alloc(sizeof(double) * (size_t)std::max<int64_t>(plan.num_partials, 1) * BM * BN);
                }
                Timer t_gram(st, &res->ms_gram);
                GramArgs ga;
                for (int g = 0; g < 2; ++g) { ga.X[g] = d->g[g].gram_operand(); ga.C[g] = d_C[g].p; }
                ga.count_bytes = count_bytes; ga.partials = d_partials.as<double>();
                ga.d_pairs = d_pairs.as<uint16_t>(); ga.d_colmap = d_colmap.as<int32_t>();
                ga.gram = comm ? d_gram_local.as<double>() : d_gram.as<double>();
                ga.tail_mi = b.tail_mi();
                struct EventPair {   // RAII: an error thrown further down must not leak the events
                    cudaEvent_t a = nullptr, b = nullptr;
                    EventPair() { OB_CUDA(cudaEventCreate(&a)); OB_CUDA(cudaEventCreate(&b)); }
                    ~EventPair() { if (a) cudaEventDestroy(a); if (b) cudaEventDestroy(b); }
                } ev;
                ob_design* dm = const_cast<ob_design*>(d);
                if (solve_only) {
                    OB_CUDA(cudaEventRecord(ev.a, st));
                    OB_CUDA(cudaMemsetAsync(d_gram.p, 0, sizeof(double) * 2 * (size_t)pn * BM * Pld, st));
                    OB_CUDA(cudaEventRecord(ev.b, st));
                } else if (PendingPack* P = dm->pending) {
                    // the design's upload is still in flight (ob_design_pack_async / _row_shard_async): contract the leaves
                    // whose rows the first chunk delivered, then -- once everything has arrived (row shards: once the rows
                    // owned by other ranks have been exchanged) -- the rest.  Same partial tiles, same fixed-tree sums as
                    // one launch.
                    int la[2] = {0, 0}, na[2] = {0, 0};
                    const bool split = P->chunk_done.size() > 1;
                    for (int g = 0; g < 2; ++g) {
                        if (!split || plan.segs[g] == 0) continue;
                        const int64_t sr = plan.seg_rows[g];
                        const int64_t lo = (P->ready_lo[g] + sr - 1) / sr, hi = std::min<int64_t>(plan.segs[g], P->rows_ready[g][0] / sr);
                        if (hi > lo) { la[g] = (int)lo; na[g] = (int)(hi - lo); }
                    }
                    EventPair evA, evB;        // OBBOOT_TRACE: where the launches sit relative to the upload
                    OB_CUDA(cudaEventRecord(ev.a, st));
                    if (na[0] + na[1] > 0) {
                        OB_CUDA(cudaStreamWaitEvent(st, P->chunk_done.front(), 0));
                        if (tr.on) OB_CUDA(cudaEventRecord(evA.a, st));
                        gram_launch_leaves(plan, ga, la, na, st);
                        if (tr.on) OB_CUDA(cudaEventRecord(evA.b, st));
                        res->gpu_launches += 1;
                    }
                    OB_CUDA(cudaStreamWaitEvent(st, P->chunk_done.back(), 0));
                    pending_exchange(dm);      // row shards: import the rows other ranks uploaded (a collective, on st)
                    if (tr.on) OB_CUDA(cudaEventRecord(evB.a, st));
                    {   // the leaves before and after the first launch's range
                        int lo0[2] = {0, 0}, n0[2] = {na[0] ? la[0] : 0, na[1] ? la[1] : 0};
                        int lo1[2] = {la[0] + na[0], la[1] + na[1]}, n1[2] = {plan.segs[0] - lo1[0], plan.segs[1] - lo1[1]};
                        if (n0[0] + n0[1] > 0) { gram_launch_leaves(plan, ga, lo0, n0, st); res->gpu_launches += 1; }
                        gram_launch_leaves(plan, ga, lo1, n1, st);
                    }
                    OB_CUDA(cudaEventRecord(ev.b, st));
                    gram_reduce_launch(plan, ga, st);
                    res->gpu_launches += 2;
                    if (tr.on) {
                        OB_CUDA(cudaEventSynchronize(ev.b));
                        auto rel = [&](cudaEvent_t e) { float ms = -1.f; if (cudaEventElapsedTime(&ms, P->ev_begin, e) != cudaSuccess) { cudaGetLastError(); ms = -1.f; } return ms; };
                        fprintf(stderr, "[obboot] async pack (ms after its start): chunk 0 packed %.1f, upload done %.1f, all packed %.1f | "
                                        "first gram launch %.1f..%.1f (leaves %d+%d of %d+%d), rest %.1f..%.1f\n",
                                rel(P->chunk_done.front()), rel(P->ev_h2d_end), rel(P->chunk_done.back()), rel(evA.a), rel(evA.b), na[0], na[1],
                                plan.segs[0], plan.segs[1], rel(evB.a), rel(ev.b));
                    }
                    pending_finish(dm);       // host: waits for the copy stream, releases the staging, raises deferred errors
                } else {
                    gram_launch(plan, ga, st, ev.a, ev.b);
                    res->gpu_launches += 2;
                }
                t_gram.stop();
                tr.mark("gram", st, true);
                if (comm && !solve_only) {
                    // every rank's subtree sums -> all ranks; the top of the summation tree is then evaluated in fixed
                    // order on each rank (bit-identical to the single-GPU reduction)
                    Timer t_c(st, &res->ms_comm);
                    const size_t batch_elems = 2 * (size_t)pn * BM * Pld;
                    comm->allgather(d_gram_local.p, d_gathered.p, sizeof(double) * batch_elems, st);
                    gram_combine_launch(d_gathered.as<double>(), world, ranks_with_rows, (int64_t)pn * BM * Pld, d_gram.as<double>(), st);
                    res->gpu_launches += 1;
                    t_c.stop(); OB_CUDA(cudaStreamSynchronize(st)); t_c.collect();
                }
                if (cache) {
                    // the reduced Gram of these slots is complete (the reduce / combine zeroed it first): fill the cells the
                    // contraction skipped from the cache, keep the ones it computed
                    Timer t_cc(st, &res->ms_gram);
                    GramCacheCopy cc{d_gram.as<double>(), pn * BM, Pld, b.slot_lo, bslots, cache->xx, cache->yy, slots,
                                     d_cmap.as<int32_t>(), nx, ny, 0, nx + ny};
                    // clustered: the per-slot row counts travel with the cells (a SOLVE_ONLY run draws no multiplicities)
                    for (int g = 0; clustered && g < 2 && (mode == OB_CACHE_FILLED || solve_only); ++g) {
                        long long* batch_rows = d_rows.as<long long>() + (size_t)g * pn * BM;
                        long long* kept = cache->rows + (size_t)g * slots + b.slot_lo;
                        OB_CUDA(cudaMemcpyAsync(solve_only ? batch_rows : kept, solve_only ? kept : batch_rows, sizeof(long long) * (size_t)bslots,
                                                cudaMemcpyDeviceToDevice, st));
                    }
                    // Bayesian: so do the per-slot weight sums
                    for (int g = 0; bayes && g < 2 && (mode == OB_CACHE_FILLED || solve_only); ++g) {
                        double* batch_esum = bw.esum.as<double>() + (size_t)g * pn * BM;
                        double* kept = cache->esum + (size_t)g * slots + b.slot_lo;
                        OB_CUDA(cudaMemcpyAsync(solve_only ? batch_esum : kept, solve_only ? kept : batch_esum, sizeof(double) * (size_t)bslots,
                                                cudaMemcpyDeviceToDevice, st));
                    }
                    if (mode == OB_CACHE_FILLED) gram_cache_extract_launch(cc, st);
                    else if (solve_only) gram_cache_assemble_launch(cc, st);
                    else {
                        cc.c_hi = nx; gram_cache_assemble_launch(cc, st);
                        cc.c_lo = nx; cc.c_hi = nx + ny; gram_cache_extract_launch(cc, st);
                        res->gpu_launches += 1;
                    }
                    res->gpu_launches += 1;
                    t_cc.stop(); OB_CUDA(cudaStreamSynchronize(st)); t_cc.collect();
                }

                // (4) solves + decomposition epilogue
                Timer t_solve(st, &res->ms_solve);
                SolveArgs sa;
                sa.gram = d_gram.as<double>(); sa.slots_pad = pn * BM; sa.Pld = Pld; sa.slots = bslots;
                sa.K = K; sa.n_cont = d->n_cont; sa.ref_kind = o->ref_kind; sa.T = T;
                sa.n_norm = o->n_norm; sa.d_norm_m = d_nm.as<int>(); sa.d_norm_off = d_noff.as<int>();
                sa.d_norm_idx = d_nidx.as<int>(); sa.d_norm_has_base = d_nhb.as<int>();
                sa.n_base = n_base; sa.S = S; sa.weighted = d->weighted ? 1 : 0;
                sa.na = (double)n_glob[0]; sa.nb = (double)n_glob[1];
                sa.rows = clustered ? d_rows.as<long long>() : nullptr;     // [2][pn * BM]
                sa.esum = bayes ? bw.esum.as<double>() : nullptr;           // [2][pn * BM]
                sa.stats = d_stats.as<double>() + (size_t)b.slot_lo * SE;
                sa.status = d_status.as<int>() + b.slot_lo;
                sa.beta_a = want_beta ? d_ba.as<double>() + (size_t)b.slot_lo * KE : nullptr;
                sa.beta_b = want_beta ? d_bb.as<double>() + (size_t)b.slot_lo * KE : nullptr;
                sa.point_extra = (p0 == 0) ? d_point.as<double>() : nullptr;
                DevBuf d_solve_scratch(solve_scratch_bytes(K, o->ref_kind == OB_REF_POOLED, o->n_norm, T, bslots));   // wide designs only
                sa.scratch = d_solve_scratch.as<double>();
                solve_launch(sa, st);
                res->gpu_launches += 1;
                t_solve.stop();

                if (comm) comm->allreduce(d_flags.p, 4, CommDType::I32, CommOp::MAX, st);   // all ranks take the same exit
                int flags[4];
                OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
                OB_CUDA(cudaStreamSynchronize(st));
                tr.mark("solve + flags", st, false);
                t_counts.collect(); t_gram.collect(); t_solve.collect();
                { float ms = 0; cudaEventElapsedTime(&ms, ev.a, ev.b); res->ms_gram_kernel += ms; }
                saturated = check_batch_flags(flags, count_bytes, o->count_bits, d->ldx);
            }
            if (!saturated) break;
            count_bytes = 2;  // widen and redo
            res->ms_counts = res->ms_gram = res->ms_solve = res->ms_gram_kernel = res->ms_comm = 0.0;
        }

        tr.mark("batches done (buffers freed)", st, true);
        // ---- point estimate (builder.rs:810-811): a failure here is a hard error ----
        int point_status = 0;
        OB_CUDA(cudaMemcpyAsync(&point_status, d_status.p, sizeof(int), cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaMemcpyAsync(point.data(), d_point.p, sizeof(double) * point.size(), cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        if (point_status != OB_OK) fail((ob_status)point_status, status_text(point_status));
        };   // run_batches

        // mode R: a rank that failed must not leave its peers waiting inside the gather
        agree_on_status(rr.shard_reps ? ctx->comm.get() : nullptr, st, run_batches, "another rank of the replicate-sharded run failed");
        if (cache) {
            if (mode == OB_CACHE_FILLED) {
                cache->design_id = d->id; cache->x_gen = d->x_gen; cache->seed = o->seed;
                cache->reps = o->reps; cache->rep_begin = rr.rb; cache->rep_end = rr.re; cache->slots = slots;
                cache->shard_reps = rr.shard_reps ? 1 : 0; cache->rep_world = rep_world; cache->rep_rank = rep_rank;
                cache->row_world = d->world; cache->row_rank = d->rank; cache->K = K; cache->count_bytes = count_bytes;
                cache->bayes = bayes;
                cache->xx_ok = true;
            }
            if (!solve_only) { cache->y_gen = d->y_gen; cache->T = T; cache->y_ok = true; }
            cache->last_use = mode;
        }
        res->total_gap = point[5 * K];
        if (res->xa_mean) memcpy(res->xa_mean, point.data(), sizeof(double) * K);
        if (res->xb_mean) memcpy(res->xb_mean, point.data() + K, sizeof(double) * K);
        for (int t = 0; t < T; ++t) {
            if (res->beta_star) memcpy(res->beta_star + (size_t)t * K, point.data() + t * PE + 2 * K, sizeof(double) * K);
            if (res->total_gap_multi) res->total_gap_multi[t] = point[t * PE + 5 * K];
        }

        // OaxacaResults.residuals (builder.rs:946: raw residuals of group B under its un-normalised fit) on the side
        // stream: the kernel and its 8 n_b byte D2H overlap the gather and the reduction below.  A page-locked
        // destination (ob_host_alloc / ob_host_register) takes the DMA directly.
        DevBuf d_res;
        struct SideJoin { cudaStream_t s; bool armed = false; ~SideJoin() { if (armed) cudaStreamSynchronize(s); } } side_join{ctx->stream_side};
        if (res->residuals_b) {
            side_join.armed = true;      // an error further down must not release d_res under the side stream
            d_res.alloc(sizeof(double) * (size_t)std::max<int64_t>(d->g[1].n, 1) * T);
            cudaStream_t s2 = ctx->stream_side;
            OB_CUDA(cudaEventRecord(ev_point, st));            // orders the allocation, too
            OB_CUDA(cudaStreamWaitEvent(s2, ev_point, 0));
            for (int t = 0; t < T; ++t)     // outcome t sits in design column K + t
                residuals_launch(d->g[1], K, K + t, d->ldx, d_point.as<double>() + t * PE + 4 * K, d_res.as<double>() + (size_t)t * d->g[1].n, s2);
            res->gpu_launches += T;
            if (d->g[1].n) OB_CUDA(cudaMemcpyAsync(res->residuals_b, d_res.p, sizeof(double) * (size_t)d->g[1].n * T, cudaMemcpyDeviceToHost, s2));
        }
        if (res->point_stats) OB_CUDA(cudaMemcpyAsync(res->point_stats, d_stats.p, sizeof(double) * SE, cudaMemcpyDeviceToHost, st));
        if (res->beta_a) OB_CUDA(cudaMemcpyAsync(res->beta_a, d_ba.p, sizeof(double) * KE, cudaMemcpyDeviceToHost, st));
        if (res->beta_b) OB_CUDA(cudaMemcpyAsync(res->beta_b, d_bb.p, sizeof(double) * KE, cudaMemcpyDeviceToHost, st));
        tr.mark("point + residuals queued", st, false);

        // ---- mode R: replicate rows of all ranks, device to device, into global replicate order ----
        const int64_t reps_all = rr.shard_reps ? o->reps : rr.nrep;
        DevBuf d_gstats, d_gstatus, d_gba, d_gbb;
        const double* stats_rows = d_stats.as<double>() + SE;     // [reps_all][T][S]
        const int* status_rows = d_status.as<int>() + 1;
        const double* ba_rows = want_beta ? d_ba.as<double>() + KE : nullptr;
        const double* bb_rows = want_beta ? d_bb.as<double>() + KE : nullptr;
        if (rr.shard_reps) {
            Timer t_c(st, &res->ms_comm);
            Comm* cm = ctx->comm.get();
            stats_rows = allgather_shards(cm, o->reps, SE, stats_rows, d_gstats, st);
            status_rows = allgather_shards(cm, o->reps, 1, status_rows, d_gstatus, st);
            if (res->rep_beta_a) ba_rows = allgather_shards(cm, o->reps, KE, ba_rows, d_gba, st);
            if (res->rep_beta_b) bb_rows = allgather_shards(cm, o->reps, KE, bb_rows, d_gbb, st);
            t_c.stop(); OB_CUDA(cudaStreamSynchronize(st)); t_c.collect();
            tr.mark("replicate all-gather", st, false);
        }

        // ---- (5) reduction to standard errors / p-values / percentile CIs ----
        if (!o->skip_reduce) {
            // the T x S statistics of a slot reduce independently: one launch over T*S columns; outputs are [T][S]
            double* dst[5] = {res->std_err, res->p_value, res->ci_lower, res->ci_upper, res->t_stat};
            reduce_to_host(st, stats_rows, status_rows, reps_all, SE, d_stats.as<double>(), dst, &res->n_ok, &res->ms_reduce);
            res->gpu_launches += 1;
        }
        if (reps_all > 0) {
            if (res->rep_stats) OB_CUDA(cudaMemcpyAsync(res->rep_stats, stats_rows, sizeof(double) * (size_t)reps_all * SE, cudaMemcpyDeviceToHost, st));
            if (res->rep_status) OB_CUDA(cudaMemcpyAsync(res->rep_status, status_rows, sizeof(int) * (size_t)reps_all, cudaMemcpyDeviceToHost, st));
            if (res->rep_beta_a) OB_CUDA(cudaMemcpyAsync(res->rep_beta_a, ba_rows, sizeof(double) * (size_t)reps_all * KE, cudaMemcpyDeviceToHost, st));
            if (res->rep_beta_b) OB_CUDA(cudaMemcpyAsync(res->rep_beta_b, bb_rows, sizeof(double) * (size_t)reps_all * KE, cudaMemcpyDeviceToHost, st));
        }
        if (res->residuals_b) {   // the side stream rejoins before the call's end (and before d_res is released on st)
            OB_CUDA(cudaEventRecord(ev_point, ctx->stream_side));
            OB_CUDA(cudaStreamWaitEvent(st, ev_point, 0));
        }
        t_total.stop();
        OB_CUDA(cudaStreamSynchronize(st));
        t_total.collect();
        tr.mark("reduce + replicate D2H", st, false);
}

ob_status ob_bootstrap_run(ob_ctx* ctx, const ob_design* d, const ob_boot_opts* o, ob_result* res) {
    if (!ctx || !d || !o || !res) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] { bootstrap_body(ctx, d, o, nullptr, res); });
}

ob_status ob_gram_cache_create(ob_ctx* ctx, ob_gram_cache** out) {
    if (!ctx || !out) return OB_ERR_INVALID_ARG;
    auto* c = new ob_gram_cache;
    c->owner = ctx; c->device = ctx->device;
    {
        std::lock_guard<std::mutex> lk(ctx->designs_mu);
        ctx->caches.insert(c);
    }
    *out = c;
    return OB_OK;
}

void ob_gram_cache_destroy(ob_gram_cache* c) {
    if (!c) return;
    if (ob_ctx* ctx = c->owner) {      // an orphaned cache (context already destroyed) holds no device memory any more
        int prev = -1;
        cudaGetDevice(&prev);
        cudaSetDevice(c->device);
        {
            std::lock_guard<std::mutex> lk(ctx->designs_mu);
            ctx->caches.erase(c);
        }
        cache_release_device(c);
        if (prev >= 0 && prev != c->device) cudaSetDevice(prev);
    }
    delete c;
}

ob_status ob_gram_cache_last_use(const ob_gram_cache* c, int32_t* use, int64_t* bytes) {
    if (!c) return OB_ERR_INVALID_ARG;
    if (use) *use = c->last_use;
    if (bytes) *bytes = (int64_t)(c->xx_bytes + c->yy_bytes + c->rows_bytes + c->esum_bytes);
    return OB_OK;
}

ob_status ob_bootstrap_run_cached(ob_ctx* ctx, const ob_design* d, const ob_boot_opts* o, ob_gram_cache* cache, ob_result* res) {
    if (!ctx || !d || !o || !cache || !res) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        if (cache->owner != ctx) fail(OB_ERR_INVALID_ARG, "this Gram cache belongs to another context");
        try {
            bootstrap_body(ctx, d, o, cache, res);
        } catch (...) {          // whatever failed, the next call fills the cache anew
            cache_release_device(cache);
            cache->last_use = OB_CACHE_NONE;
            throw;
        }
    });
}

ob_status ob_bootstrap_run_bayes(ob_ctx* ctx, const ob_design* d, const ob_boot_opts* o, const ob_bayes_opts* bo,
                                 ob_gram_cache* cache, ob_result* res) {
    if (!ctx || !d || !o || !res) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        if (!cache) { bootstrap_body(ctx, d, o, nullptr, res, true, bo); return; }
        if (cache->owner != ctx) fail(OB_ERR_INVALID_ARG, "this Gram cache belongs to another context");
        try {
            bootstrap_body(ctx, d, o, cache, res, true, bo);
        } catch (...) {          // whatever failed, the next call fills the cache anew
            cache_release_device(cache);
            cache->last_use = OB_CACHE_NONE;
            throw;
        }
    });
}

ob_status ob_reduce_stats(ob_ctx* ctx, const double* rep_stats, const int32_t* rep_status, int64_t reps, int32_t S,
                          const double* point_stats, int64_t* n_ok, double* std_err, double* p_value,
                          double* ci_lower, double* ci_upper, double* t_stat) {
    if (!ctx || S < 1 || reps < 0 || !point_stats || (reps && (!rep_stats || !rep_status))) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        cudaStream_t st = ctx->stream;
        DevBuf d_stats(sizeof(double) * (size_t)std::max<int64_t>(reps, 1) * S), d_status(sizeof(int) * (size_t)std::max<int64_t>(reps, 1));
        DevBuf d_point(sizeof(double) * S);
        if (reps) {
            OB_CUDA(cudaMemcpyAsync(d_stats.p, rep_stats, sizeof(double) * (size_t)reps * S, cudaMemcpyHostToDevice, st));
            OB_CUDA(cudaMemcpyAsync(d_status.p, rep_status, sizeof(int) * (size_t)reps, cudaMemcpyHostToDevice, st));
        }
        OB_CUDA(cudaMemcpyAsync(d_point.p, point_stats, sizeof(double) * S, cudaMemcpyHostToDevice, st));
        double* dst[5] = {std_err, p_value, ci_lower, ci_upper, t_stat};
        reduce_to_host(st, d_stats.as<double>(), d_status.as<int>(), reps, S, d_point.as<double>(), dst, n_ok, nullptr);
    });
}

// Host-only: the columns the Gram contraction computes (gram_columns), for the CPU tests.
int64_t ob_debug_gram_columns(int32_t K, int32_t T, int32_t n_cont, const int32_t* cat_levels, int32_t n_cat,
                              uint16_t* pairs_out, int32_t* colmap_out, int64_t cap, int32_t* tiling_out) {
    if (K < 1 || T < 1 || n_cont < 0 || n_cat < 0 || (n_cat > 0 && !cat_levels) || K + T > 65535) return -1;
    const GramColumns gc = gram_columns(K, T, n_cont, std::vector<int>(cat_levels, cat_levels + n_cat));
    const int64_t len = (int64_t)gc.colmap.size();
    for (int64_t c = 0; c < len && c < cap; ++c) {
        if (pairs_out) { pairs_out[2 * c] = gc.pairs[2 * (size_t)c]; pairs_out[2 * c + 1] = gc.pairs[2 * (size_t)c + 1]; }
        if (colmap_out) colmap_out[c] = gc.colmap[(size_t)c];
    }
    if (tiling_out) { tiling_out[0] = gc.Pc; tiling_out[1] = gc.nfull; tiling_out[2] = gc.tail_q; }
    return len;
}

int64_t ob_debug_gram_outcome_columns(int32_t K, int32_t T, uint16_t* pairs_out, int32_t* colmap_out, int64_t cap,
                                      int32_t* tiling_out) {
    if (K < 1 || T < 1 || K + T > 65535) return -1;
    const GramColumns gc = gram_outcome_columns(K, T);
    const int64_t len = (int64_t)gc.colmap.size();
    for (int64_t c = 0; c < len && c < cap; ++c) {
        if (pairs_out) { pairs_out[2 * c] = gc.pairs[2 * (size_t)c]; pairs_out[2 * c + 1] = gc.pairs[2 * (size_t)c + 1]; }
        if (colmap_out) colmap_out[c] = gc.colmap[(size_t)c];
    }
    if (tiling_out) { tiling_out[0] = gc.Pc; tiling_out[1] = gc.nfull; tiling_out[2] = gc.tail_q; }
    return len;
}

// Host-only: the unit schedule of the Gram kernel for a problem shape (no device needed; CPU tests).  out8 receives up to
// cap rows of (cta, group, panel, tile, segment, stages, slot groups, tail quanta); returns the number of units.
int64_t ob_debug_gram_schedule(int32_t K, int64_t n_a, int64_t n_b, int64_t slots, int32_t world, int32_t rank, int32_t grid,
                               int64_t* out8, int64_t cap) {
    if (K < 1 || n_a < 0 || n_b < 0 || slots < 1 || world < 1 || (world & (world - 1)) || world > MAX_WORLD || rank < 0 ||
        rank >= world || grid < 1) return -1;
    GroupData gd[2];
    const int64_t ns[2] = {n_a, n_b};
    for (int g = 0; g < 2; ++g) {
        gd[g].shard = row_shard(ns[g], rank, world);
        gd[g].n = gd[g].shard.n_local; gd[g].n_pad = pad_rows(gd[g].n);
    }
    const int64_t panels = (slots + BM - 1) / BM;
    return gram_schedule_debug(K, (int)panels, slots - (panels - 1) * BM, gd, grid, out8, cap);
}

ob_status ob_debug_counts(ob_ctx* ctx, const ob_design* d, uint64_t seed, int64_t rep, int32_t group,
                          uint16_t* counts_out) {
    if (!ctx || !d || !counts_out || group < 0 || group > 1 || rep < 0) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        cudaStream_t st = ctx->stream;
        const GroupData& G = d->g[group];
        DevBuf d_C((size_t)G.n_pad * BM * 2), d_colsum(sizeof(long long) * BM), d_flags(sizeof(int) * 4), d_lut(counts_lut_bytes());
        OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
        CountsArgs ca;
        ca.C = d_C.p; ca.count_bytes = 2; ca.n = G.n; ca.n_pad = G.n_pad; ca.panels = 1; ca.slots = 2;
        ca.first_slot = 1; ca.rep0 = rep - 1; ca.group = group; ca.seed = seed;
        ca.n_global = G.shard.n_global; ca.row_begin = G.shard.row_begin;
        if (d->world > 1) fail(OB_ERR_UNSUPPORTED, "ob_debug_counts on a row-sharded design");
        DevBuf d_U, d_rows;
        const int m = d->cl_strata == OB_CLUSTER_JOINT ? 0 : group;
        if (d->cl_strata != OB_CLUSTER_NONE) {      // the unit counts of the replicate, expanded to the group's rows below
            const int64_t M = d->cl_units[m];
            d_U.alloc((size_t)pad_rows(M) * BM * 2);
            d_rows.alloc(sizeof(long long) * 2 * BM);
            ca.C = d_U.p; ca.n = ca.n_global = M; ca.n_pad = pad_rows(M); ca.row_begin = 0;
            ca.group = d->cl_strata == OB_CLUSTER_JOINT ? 2 : group;
        }
        OB_CUDA(cudaMemsetAsync(d_colsum.p, 0, d_colsum.bytes, st));
        counts_philox_body_launch(ca, d_colsum.as<long long>(), d_lut.as<unsigned char>(), st);
        counts_philox_fixup_launch(ca, d_colsum.as<long long>(), d_flags.as<int>(), st);
        if (d->cl_strata != OB_CLUSTER_NONE) {
            OB_CUDA(cudaMemsetAsync(d_rows.p, 0, d_rows.bytes, st));
            ExpandArgs ea{d_C.p, d_U.p, G.uid, 2, G.n, G.n_pad, ca.n_pad, 1, 2, d_rows.as<long long>()};
            counts_expand_launch(ea, st);
        }
        // slot 1 column of the single panel
        OB_CUDA(cudaMemcpy2DAsync(counts_out, sizeof(uint16_t), d_C.as<uint16_t>() + 1, sizeof(uint16_t) * BM,
                                  sizeof(uint16_t), (size_t)G.n, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
    });
}

// The native Bayesian-bootstrap weights E of one replicate of one group, read back (the production kernel, one panel).
ob_status ob_debug_bayes_weights(ob_ctx* ctx, const ob_design* d, uint64_t seed, int64_t rep, int32_t group, float* out) {
    if (!ctx || !d || !out || group < 0 || group > 1 || rep < 0) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        if (d->world > 1) fail(OB_ERR_UNSUPPORTED, "ob_debug_bayes_weights on a row-sharded design");
        cudaStream_t st = ctx->stream;
        const GroupData& G = d->g[group];
        const int segs = G.shard.leaf_hi - G.shard.leaf_lo;
        DevBuf d_C((size_t)G.n_pad * BM * sizeof(float)), d_part(sizeof(double) * (size_t)std::max(segs, 1) * BM);
        BayesArgs a;
        a.C = d_C.as<float>(); a.n = G.n; a.n_pad = G.n_pad; a.panels = 1;
        a.n_global = G.shard.n_global; a.row_begin = G.shard.row_begin;
        a.slots = 2; a.first_slot = 1; a.rep0 = rep - 1; a.group = group; a.seed = seed;
        a.segs = segs; a.seg_rows = G.shard.seg_rows; a.wt = nullptr; a.part = d_part.as<double>();
        bayes_weights_launch(a, st);
        OB_CUDA(cudaMemcpy2DAsync(out, sizeof(float), d_C.as<float>() + 1, sizeof(float) * BM, sizeof(float), (size_t)G.n,
                                  cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
    });
}

// The multiplicity matrix ob_bootstrap_run builds from an explicit index stream, read back (tests: np.bincount parity).
ob_status ob_debug_counts_from_indices(ob_ctx* ctx, const ob_design* d, int32_t group, const uint32_t* idx, int64_t reps,
                                       int32_t count_bits, uint16_t* counts_out, int32_t* flags_out) {
    if (!ctx || !d || !counts_out || group < 0 || group > 1 || reps < 0 || (reps && !idx) || (count_bits != 8 && count_bits != 16))
        return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        design_ready(d);
        cudaStream_t st = ctx->stream;
        const GroupData& G = d->g[group];
        const int cb = count_bits / 8;
        const int64_t slots = 1 + reps, panels = (slots + BM - 1) / BM;
        const int64_t n_glob = G.shard.n_global;
        DevBuf d_C((size_t)panels * G.n_pad * BM * cb), d_flags(sizeof(int) * 4);
        DevBuf d_idx(sizeof(uint32_t) * (size_t)std::max<int64_t>(reps * n_glob, 1));
        OB_CUDA(cudaMemsetAsync(d_flags.p, 0, sizeof(int) * 4, st));
        if (reps) OB_CUDA(cudaMemcpyAsync(d_idx.p, idx, sizeof(uint32_t) * (size_t)reps * n_glob, cudaMemcpyHostToDevice, st));
        CountsArgs ca;
        ca.C = d_C.p; ca.count_bytes = cb; ca.n = G.n; ca.n_pad = G.n_pad; ca.panels = (int)panels; ca.slots = slots;
        ca.first_slot = 1; ca.rep0 = -1; ca.group = group; ca.seed = 0;
        ca.n_global = n_glob; ca.row_begin = G.shard.row_begin;
        counts_from_indices(ca, d_idx.as<uint32_t>(), d_flags.as<int>(), st);   // the production kernel
        std::vector<uint8_t> h((size_t)panels * G.n_pad * BM * cb);
        int flags[4];
        OB_CUDA(cudaMemcpyAsync(h.data(), d_C.p, h.size(), cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaMemcpyAsync(flags, d_flags.p, sizeof flags, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
        for (int64_t r = 0; r < reps; ++r) {
            const int64_t slot = 1 + r, panel = slot / BM, col = slot % BM;
            for (int64_t i = 0; i < G.n; ++i) {
                const size_t e = (size_t)(panel * G.n_pad + i) * BM + col;
                counts_out[r * G.n + i] = cb == 1 ? (uint16_t)h[e] : reinterpret_cast<const uint16_t*>(h.data())[e];
            }
        }
        // the point-estimate slot must hold exactly one of every valid row and nothing on the padding
        for (int64_t i = 0; i < G.n_pad; ++i) {
            const size_t e = (size_t)i * BM;
            const unsigned v = cb == 1 ? h[e] : reinterpret_cast<const uint16_t*>(h.data())[e];
            if (v != (i < G.n ? 1u : 0u)) fail(OB_ERR_CUDA, "point-estimate slot of the multiplicity matrix is not all ones");
        }
        if (flags_out) *flags_out = (flags[1] ? 1 : 0) | (flags[2] ? 2 : 0);   // 1 = a count saturated, 2 = index out of range
    });
}

// The reduced Gram cells a cached run left in its cache, read back (tests: cell-by-cell checks of the contraction).
ob_status ob_debug_gram_cache_read(ob_ctx* ctx, const ob_gram_cache* c, int64_t* shape_out, double* xx_out, double* yy_out,
                                   int64_t* rows_out) {
    if (!ctx || !c) return OB_ERR_INVALID_ARG;
    return guarded(ctx, [&] {
        if (c->owner != ctx) fail(OB_ERR_INVALID_ARG, "this Gram cache belongs to another context");
        if (!c->xx || !c->yy || !c->xx_ok || !c->y_ok) fail(OB_ERR_INVALID_ARG, "the Gram cache is empty");
        if (shape_out) {
            shape_out[0] = c->slots; shape_out[1] = c->K; shape_out[2] = c->T;
            shape_out[3] = c->count_bytes; shape_out[4] = c->rows ? 1 : 0;
        }
        cudaStream_t st = ctx->stream;
        if (xx_out) OB_CUDA(cudaMemcpyAsync(xx_out, c->xx, c->xx_bytes, cudaMemcpyDeviceToHost, st));
        if (yy_out) OB_CUDA(cudaMemcpyAsync(yy_out, c->yy, c->yy_bytes, cudaMemcpyDeviceToHost, st));
        if (rows_out && c->rows) OB_CUDA(cudaMemcpyAsync(rows_out, c->rows, c->rows_bytes, cudaMemcpyDeviceToHost, st));
        OB_CUDA(cudaStreamSynchronize(st));
    });
}

}  // extern "C"
