// comm.cu -- multi-GPU plumbing behind the C ABI: one process (one nhp_ctx) per GPU, NCCL over NVLink / NVSwitch.
//
// SURVEY.md section 8e: the hot path shards by contiguous time ranges (log-likelihood, parent sweep, statistics) and by
// child column (adjacency sampler); the only exchanges are an all-reduce of the per-pair sufficient statistics and of
// the scalar log-likelihood shares, and an all-gather of the owned adjacency columns.  The host (Julia / Python) only
// distributes the 128-byte NCCL id (MPI, Distributed.jl, a file, torch.distributed -- anything) and calls
// nhp_comm_init; every collective then runs on the context's stream, ordered with the library's kernels.
// NCCL is loaded at run time (dlopen of libnccl.so.2: the copy already mapped by the host process if there is one), so
// libnhp.so itself has no link-time dependency on it and single-GPU users never touch it.
#include "nhp_internal.cuh"
#include <dlfcn.h>
#include <nccl.h>
#include <string.h>
#include <algorithm>
#include <vector>

struct NcclApi {
    void *lib = nullptr;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*Broadcast)(const void *, void *, size_t, ncclDataType_t, int, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*GroupStart)() = nullptr;
    ncclResult_t (*GroupEnd)() = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
};
static NcclApi g_nccl;

static int nccl_load(nhp_ctx *ctx) {
    if (g_nccl.lib) return NHP_OK;
    void *h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD | RTLD_GLOBAL);  // the host process's own copy first (torch, NCCL_jll)
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
    if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
    if (!h) return nhp_fail(ctx, NHP_ERR_UNSUPPORTED, "nhp_comm: cannot load libnccl.so.2 (%s)", dlerror());
    NcclApi a;
    a.lib = h;
    a.GetUniqueId = (decltype(a.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    a.CommInitRank = (decltype(a.CommInitRank))dlsym(h, "ncclCommInitRank");
    a.CommDestroy = (decltype(a.CommDestroy))dlsym(h, "ncclCommDestroy");
    a.AllReduce = (decltype(a.AllReduce))dlsym(h, "ncclAllReduce");
    a.AllGather = (decltype(a.AllGather))dlsym(h, "ncclAllGather");
    a.GetErrorString = (decltype(a.GetErrorString))dlsym(h, "ncclGetErrorString");
    a.Broadcast = (decltype(a.Broadcast))dlsym(h, "ncclBroadcast");
    a.GroupStart = (decltype(a.GroupStart))dlsym(h, "ncclGroupStart");
    a.GroupEnd = (decltype(a.GroupEnd))dlsym(h, "ncclGroupEnd");
    if (!a.GetUniqueId || !a.CommInitRank || !a.CommDestroy || !a.AllReduce || !a.AllGather || !a.GetErrorString || !a.Broadcast || !a.GroupStart || !a.GroupEnd)
        return nhp_fail(ctx, NHP_ERR_UNSUPPORTED, "nhp_comm: libnccl.so.2 lacks a required symbol");
    g_nccl = a;
    return NHP_OK;
}

#define NHP_NCCL(ctx, call)                                                                                             \
    do {                                                                                                                \
        ncclResult_t r__ = (call);                                                                                      \
        if (r__ != ncclSuccess) return nhp_fail((ctx), NHP_ERR_CUDA, "%s failed: %s", #call, g_nccl.GetErrorString(r__)); \
    } while (0)

extern "C" int nhp_comm_unique_id(void *id128) {
    if (!id128) return nhp_fail(nullptr, NHP_ERR_INVALID, "nhp_comm_unique_id: NULL buffer");
    NHP_TRY(nccl_load(nullptr));
    static_assert(sizeof(ncclUniqueId) == 128, "NCCL unique id is 128 bytes");
    ncclUniqueId id;
    ncclResult_t r = g_nccl.GetUniqueId(&id);
    if (r != ncclSuccess) return nhp_fail(nullptr, NHP_ERR_CUDA, "ncclGetUniqueId failed: %s", g_nccl.GetErrorString(r));
    memcpy(id128, &id, sizeof(id));
    return NHP_OK;
}

extern "C" int nhp_comm_init(nhp_ctx *ctx, const void *id128, int rank, int nranks) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, id128 != nullptr && nranks >= 1 && rank >= 0 && rank < nranks, NHP_ERR_INVALID, "nhp_comm_init: need 0 <= rank < nranks and an id");
    NHP_CHECK(ctx, ctx->comm == nullptr, NHP_ERR_STATE, "nhp_comm_init: this context already has a communicator");
    NHP_TRY(nccl_load(ctx));
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    ncclUniqueId id;
    memcpy(&id, id128, sizeof(id));
    ncclComm_t comm = nullptr;
    NHP_NCCL(ctx, g_nccl.CommInitRank(&comm, nranks, id, rank));
    ctx->comm = comm; ctx->rank = rank; ctx->nranks = nranks;
    return NHP_OK;
}

extern "C" int nhp_comm_destroy(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    if (!ctx->comm) return NHP_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    g_nccl.CommDestroy((ncclComm_t)ctx->comm);
    ctx->comm = nullptr; ctx->rank = 0; ctx->nranks = 1;
    cudaFree(ctx->d_comm_buf); ctx->d_comm_buf = nullptr; ctx->comm_buf_cap = 0;
    return NHP_OK;
}

extern "C" int nhp_comm_rank(const nhp_ctx *ctx, int *rank, int *nranks) {
    if (!ctx) return NHP_ERR_INVALID;
    if (rank) *rank = ctx->rank;
    if (nranks) *nranks = ctx->nranks;
    return NHP_OK;
}

static int comm_buf(nhp_ctx *ctx, size_t doubles, double **out) {
    if (doubles > ctx->comm_buf_cap) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_comm_buf);
        ctx->d_comm_buf = nullptr; ctx->comm_buf_cap = 0;
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_comm_buf, doubles * sizeof(double)));
        ctx->comm_buf_cap = doubles;
    }
    *out = ctx->d_comm_buf;
    return NHP_OK;
}

// all-reduce (sum) of a statistics buffer, in place, on the context's stream; no host synchronisation.
// Single-rank contexts (no communicator): no-op, so the same call sequence serves 1..N GPUs.
extern "C" int nhp_comm_allreduce_stats(nhp_ctx *ctx, int phase) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CHECK(ctx, phase == 0 || phase == 1, NHP_ERR_INVALID, "nhp_comm_allreduce_stats: phase must be 0 or 1");
    if (!ctx->comm || ctx->nranks == 1) return NHP_OK;
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const StatsLayout sl{ctx->K};
    double *buf = phase == 0 ? ctx->d_stats0 : ctx->d_stats1;
    const size_t cnt = phase == 0 ? (size_t)sl.total() : (size_t)(ctx->K * ctx->K);
    NHP_NCCL(ctx, g_nccl.AllReduce(buf, buf, cnt, ncclFloat64, ncclSum, (ncclComm_t)ctx->comm, ctx->stream));
    return NHP_OK;
}

// all-reduce (sum) of a device vector, in place on the context's stream (the per-node sums of the curves' slice update)
int nhp_comm_allreduce_dev(nhp_ctx *ctx, double *buf, int64_t n) {
    if (!ctx->comm || ctx->nranks == 1) return NHP_OK;
    NHP_NCCL(ctx, g_nccl.AllReduce(buf, buf, (size_t)n, ncclFloat64, ncclSum, (ncclComm_t)ctx->comm, ctx->stream));
    return NHP_OK;
}

// all-reduce (sum) of a small host vector (log-likelihood shares, gradient norms, ...): staged through the device
extern "C" int nhp_comm_allreduce_host(nhp_ctx *ctx, double *inout, int64_t n) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, inout != nullptr && n >= 1, NHP_ERR_INVALID, "nhp_comm_allreduce_host: bad argument");
    if (!ctx->comm || ctx->nranks == 1) return NHP_OK;
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    double *buf;
    NHP_TRY(comm_buf(ctx, (size_t)n, &buf));
    NHP_CUDA(ctx, cudaMemcpyAsync(buf, inout, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    NHP_NCCL(ctx, g_nccl.AllReduce(buf, buf, (size_t)n, ncclFloat64, ncclSum, (ncclComm_t)ctx->comm, ctx->stream));
    NHP_CUDA(ctx, cudaMemcpyAsync(inout, buf, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

// owned columns (c % R == r) of the parent-major matrix A[p + K c] <-> a dense [ncols_max][K] block
__global__ void k_adj_pack(const double *__restrict__ A, int K, int r, int R, int ncm, double *__restrict__ out) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)ncm * K) return;
    const int j = (int)(e / K), p = (int)(e % K), c = r + j * R;
    out[e] = c < K ? A[p + (int64_t)K * c] : 0.0;
}
__global__ void k_adj_unpack(double *__restrict__ A, int K, int R, int ncm, const double *__restrict__ in) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)R * ncm * K) return;
    const int q = (int)(e / ((int64_t)ncm * K)), rem = (int)(e % ((int64_t)ncm * K));
    const int j = rem / K, p = rem % K, c = q + j * R;
    if (c < K) A[p + (int64_t)K * c] = in[e];
}

// After nhp_cont_resample_adjacency_dev(..., col_begin = rank, col_stride = nranks, commit = 0): every rank receives the
// columns the other ranks resampled (ncclAllGather of K^2 / nranks doubles per rank), then the masked tables are rebuilt.
extern "C" int nhp_comm_allgather_adjacency(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set && ctx->has_A, NHP_ERR_STATE, "nhp_comm_allgather_adjacency: no network process parameters on the device");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->comm && ctx->nranks > 1) {
        const int K = (int)ctx->K, R = ctx->nranks, r = ctx->rank, ncm = (K + R - 1) / R;
        const size_t blk = (size_t)ncm * K;
        double *buf;
        NHP_TRY(comm_buf(ctx, blk * (size_t)(R + 1), &buf));
        double *send = buf, *recv = buf + blk;
        k_adj_pack<<<(unsigned)((blk + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_A, K, r, R, ncm, send);
        NHP_LAUNCHED(ctx);
        NHP_NCCL(ctx, g_nccl.AllGather(send, recv, blk, ncclFloat64, (ncclComm_t)ctx->comm, ctx->stream));
        k_adj_unpack<<<(unsigned)((blk * R + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_A, K, R, ncm, recv);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
    }
    return nhp_cont_adjacency_commit(ctx);
}

// The replicated stream of the adjacency sweep from the time shards: every rank has uploaded its own shard (events_upload with
// n_halo / index_base), the shards' own events travel over NVLink (one ncclBroadcast per rank and array, grouped) instead of
// every rank pulling the whole stream through PCIe.  The result is an ordinary unsharded events handle on every rank.
int nhp_events_from_device(nhp_ctx *ctx, const double *d_t, const int *d_c, int64_t n, double duration, int64_t K, nhp_events **out);  // nhp_context.cu
extern "C" int nhp_comm_allgather_events(nhp_ctx *ctx, nhp_events *ev_shard, nhp_events **out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev_shard != nullptr && out != nullptr, NHP_ERR_INVALID, "nhp_comm_allgather_events: NULL argument");
    *out = nullptr;
    NHP_CHECK(ctx, ctx->comm != nullptr && ctx->nranks > 1, NHP_ERR_STATE, "nhp_comm_allgather_events: the context has no communicator (a single GPU uses its handle as is)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int R = ctx->nranks, r = ctx->rank;
    std::vector<double> cnt((size_t)R + 1, 0.0);
    cnt[r] = (double)(ev_shard->n - ev_shard->n_halo);
    cnt[R] = r == 0 ? (double)(ev_shard->index_base + ev_shard->n_halo) : 0.0;  // index_base counts from the first passed (halo) event
    NHP_TRY(nhp_comm_allreduce_host(ctx, cnt.data(), R + 1));
    std::vector<int64_t> off((size_t)R + 1, 0);
    for (int q = 0; q < R; q++) off[q + 1] = off[q] + (int64_t)cnt[q];
    const int64_t n_total = off[R];
    NHP_CHECK(ctx, cnt[R] == 0.0 && ev_shard->index_base + ev_shard->n_halo == off[r], NHP_ERR_INVALID,
              "nhp_comm_allgather_events: the shards are not the consecutive pieces of one stream (rank %d: first own event %lld, expected %lld)", r,
              (long long)(ev_shard->index_base + ev_shard->n_halo), (long long)off[r]);
    NHP_CHECK(ctx, n_total < (int64_t)2147483000, NHP_ERR_INVALID, "nhp_comm_allgather_events: %lld events in total (limit 2^31)", (long long)n_total);
    cudaStream_t s = ctx->stream;
    double *d_t = nullptr;
    int *d_c = nullptr;
    NHP_CUDA(ctx, cudaMallocAsync(&d_t, (size_t)std::max<int64_t>(n_total, 1) * sizeof(double), s));
    if (cudaMallocAsync(&d_c, (size_t)std::max<int64_t>(n_total, 1) * sizeof(int), s) != cudaSuccess) {
        cudaFreeAsync(d_t, s);
        return nhp_fail(ctx, NHP_ERR_CUDA, "nhp_comm_allgather_events: cudaMallocAsync failed");
    }
    auto fin = [&](int rc) { cudaFreeAsync(d_t, s); cudaFreeAsync(d_c, s); return rc; };
    ncclResult_t nr = g_nccl.GroupStart();
    for (int q = 0; q < R && nr == ncclSuccess; q++) {
        const size_t m = (size_t)(off[q + 1] - off[q]);
        if (m == 0) continue;
        nr = g_nccl.Broadcast(ev_shard->d_t + ev_shard->n_halo, d_t + off[q], m, ncclFloat64, q, (ncclComm_t)ctx->comm, s);
        if (nr == ncclSuccess) nr = g_nccl.Broadcast(ev_shard->d_c + ev_shard->n_halo, d_c + off[q], m, ncclInt32, q, (ncclComm_t)ctx->comm, s);
    }
    const ncclResult_t ne = g_nccl.GroupEnd();
    if (nr != ncclSuccess || ne != ncclSuccess)
        return fin(nhp_fail(ctx, NHP_ERR_CUDA, "nhp_comm_allgather_events: NCCL broadcast failed: %s", g_nccl.GetErrorString(nr != ncclSuccess ? nr : ne)));
    return fin(nhp_events_from_device(ctx, d_t, d_c, n_total, ev_shard->duration, ev_shard->K, out));
}

// One whole Gibbs sweep of `resample!` (continuous.jl:202-208 / 350-358) on the device, for 1..N GPUs with one call
// sequence: parent sweep + fused statistics on this rank's time shard, all-reduce, second pass, all-reduce, conjugate draws
// (identical on every rank), with curves and their prior the elliptical-slice update of the curves (per-node sums all-reduced,
// identical decisions on every rank), and for a network process the adjacency sweep over this rank's columns of the replicated
// stream `ev_full`, the all-gather of the columns, the table rebuild and the Beta draw of rho.
extern "C" int nhp_cont_gibbs_sweep(nhp_ctx *ctx, nhp_events *ev_shard, nhp_events *ev_full, uint64_t seed, uint64_t counter, double duration,
                                    const double *hyper, int n_hyper, double net_alpha, double net_beta) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev_shard != nullptr, NHP_ERR_INVALID, "nhp_cont_gibbs_sweep: events handle is NULL");
    // curves with a prior (nhp_cont_baseline_prior) take their elliptical-slice update here; without a prior they move with the
    // host's slice sampler (resample_on_device_), so a network process with curves and no prior is refused before anything changes
    const bool curves = ctx->cont_set && ctx->bgrid_n > 0, prior = curves && ctx->bprior_n == ctx->bgrid_n;
    NHP_CHECK(ctx, !(ctx->cont_set && ctx->has_A && curves && !prior), NHP_ERR_UNSUPPORTED,
              "nhp_cont_gibbs_sweep: a network process with a grid baseline takes the elliptical-slice update of its curves on the host (or set their prior: nhp_cont_baseline_prior)");
    for (int i = 0; i < 8; i++) ctx->sweep_info[i] = 0.0;
    NHP_TRY(nhp_cont_resample_parents(ctx, ev_shard, seed, counter, nullptr, nullptr, nullptr));
    ctx->sweep_info[0] = ctx->last_ms;  // parent sweep + fused statistics
    NHP_TRY(nhp_comm_allreduce_stats(ctx, 0));
    NHP_TRY(nhp_cont_suffstats_second_pass(ctx, ev_shard));
    NHP_TRY(nhp_comm_allreduce_stats(ctx, 1));
    NHP_TRY(nhp_cont_resample_params(ctx, ev_shard, seed, counter, duration, hyper, n_hyper, 0));
    ctx->sweep_info[1] = ctx->last_ms;  // (all-reduces, second pass,) conjugate draws + table rebuild: everything since the parent sweep
    if (prior) {
        NHP_TRY(nhp_cont_resample_baseline(ctx, ev_shard, seed, counter, nullptr, nullptr, nullptr));
        ctx->sweep_info[3] = ctx->last_ms;  // slice update of the curves: list build + rounds + commit
        ctx->sweep_info[4] = ctx->slice_info[2];  // its rounds
    }
    if (ctx->has_A) {
        NHP_CHECK(ctx, ev_full != nullptr, NHP_ERR_INVALID, "nhp_cont_gibbs_sweep: a network process needs the unsharded stream for the adjacency sweep");
        const double rho = net_alpha > 0.0 ? -1.0 : 1.0;  // Bernoulli network: the context's rho; otherwise a dense network (link probability 1)
        NHP_TRY(nhp_cont_resample_adjacency_dev(ctx, ev_full, rho, seed, counter + (1ull << 40), ctx->rank, ctx->nranks, 0));
        ctx->sweep_info[2] = ctx->last_ms;  // adjacency sweep kernel
        NHP_TRY(nhp_comm_allgather_adjacency(ctx));
        if (net_alpha > 0.0) NHP_TRY(nhp_cont_resample_network(ctx, seed, counter, net_alpha, net_beta, nullptr));
    }
    if (ctx->trace_cap > 0 && ctx->trace_len < ctx->trace_cap) NHP_TRY(nhp_cont_trace_push(ctx));  // the sample of this sweep stays on the device
    return NHP_OK;
}

// One whole Gibbs sweep of the discrete `resample!` (discrete.jl:361-367 / 416-424) on one GPU, in the order and with the Philox keys
// of discrete.resample_on_device_: parent counts (seed, counter), conjugate draws (seed, counter) with Mn = the events per node kept
// with the data, table refresh, and for a network process the in-place adjacency sweep (seed, counter + 2^40) and the Beta draw of
// rho (seed, counter).  Only scalars cross PCIe.
extern "C" int nhp_disc_gibbs_sweep(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *hyper, int n_hyper, double net_alpha,
                                    double net_beta) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr, NHP_ERR_INVALID, "nhp_disc_gibbs_sweep: data handle is NULL");
    NHP_CHECK(ctx, dd->t_halo == 0, NHP_ERR_UNSUPPORTED, "nhp_disc_gibbs_sweep works on unsharded data");
    NHP_CHECK(ctx, !(ctx->comm && ctx->nranks > 1), NHP_ERR_UNSUPPORTED, "nhp_disc_gibbs_sweep runs on one GPU (the context has a communicator of %d ranks)", ctx->nranks);
    NHP_CHECK(ctx, ctx->disc_set, NHP_ERR_STATE, "nhp_disc_gibbs_sweep: discrete parameters not set (call nhp_disc_params_set)");
    NHP_CHECK(ctx, dd->d_conv != nullptr, NHP_ERR_STATE, "nhp_disc_gibbs_sweep: call nhp_disc_convolve first");
    NHP_CHECK(ctx, hyper != nullptr && n_hyper == 5, NHP_ERR_INVALID, "nhp_disc_gibbs_sweep: expected 5 hyper-parameters, got %d", n_hyper);
    for (int i = 0; i < n_hyper; i++) NHP_CHECK(ctx, std::isfinite(hyper[i]), NHP_ERR_INVALID, "nhp_disc_gibbs_sweep: hyper-parameter %d is not finite", i);
    const bool bern = ctx->d_has_A && net_alpha > 0.0;
    NHP_CHECK(ctx, !bern || net_beta > 0.0, NHP_ERR_INVALID, "nhp_disc_gibbs_sweep: net_beta must be positive");
    NHP_CHECK(ctx, !bern || ctx->dd_rho >= 0.0, NHP_ERR_STATE, "nhp_disc_gibbs_sweep: no link probability kept with the context (nhp_disc_network_set)");
    NHP_TRY(nhp_disc_gibbs_counts(ctx, dd, seed, counter, nullptr, 0, nullptr));
    NHP_TRY(nhp_disc_draw_params(ctx, dd, seed, counter, nhp_disc_rowsum(dd), hyper));
    NHP_TRY(nhp_disc_tables_refresh(ctx));
    if (ctx->d_has_A) {
        NHP_TRY(nhp_disc_resample_adjacency_dev(ctx, dd, bern ? -1.0 : 1.0, seed, counter + (1ull << 40)));  // Bernoulli: the context's rho; else dense (1)
        if (bern) NHP_TRY(nhp_disc_draw_network(ctx, seed, counter, net_alpha, net_beta));
    }
    if (ctx->dd_trace_cap > 0 && ctx->dd_trace_len < ctx->dd_trace_cap) NHP_TRY(nhp_disc_trace_push(ctx));  // the sample stays on the device
    return NHP_OK;
}

extern "C" int nhp_cont_sweep_info(const nhp_ctx *ctx, double *out8) {
    if (!ctx || !out8) return NHP_ERR_INVALID;
    for (int i = 0; i < 8; i++) out8[i] = ctx->sweep_info[i];
    return NHP_OK;
}
