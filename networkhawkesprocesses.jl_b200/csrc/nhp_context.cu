// nhp_context.cu -- context, error handling, continuous data upload and parameter tables.
#include "nhp_internal.cuh"
#include <stdarg.h>
#include <stdio.h>
#include <string.h>
#include <limits>

static thread_local std::string g_create_error;

int nhp_fail(nhp_ctx *ctx, int code, const char *fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    if (ctx) ctx->err = buf; else g_create_error = buf;
    return code;
}

extern "C" const char *nhp_last_error(const nhp_ctx *ctx) { return ctx ? ctx->err.c_str() : g_create_error.c_str(); }
extern "C" int nhp_version(void) { return NHP_VERSION; }
extern "C" int64_t nhp_launch_count(const nhp_ctx *ctx) { return ctx ? ctx->launches : 0; }
extern "C" double nhp_last_kernel_ms(const nhp_ctx *ctx) { return ctx ? ctx->last_ms : 0.0; }

extern "C" int nhp_create(int device, nhp_ctx **out) {
    if (!out) return nhp_fail(nullptr, NHP_ERR_INVALID, "nhp_create: out is NULL");
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return nhp_fail(nullptr, NHP_ERR_NO_DEVICE, "nhp_create: no CUDA device (%s); libnhp has no CPU path",
                        e != cudaSuccess ? cudaGetErrorString(e) : "device count 0");
    if (device < 0 || device >= ndev) return nhp_fail(nullptr, NHP_ERR_INVALID, "nhp_create: device %d out of range [0,%d)", device, ndev);
    cudaDeviceProp prop;
    e = cudaGetDeviceProperties(&prop, device);
    if (e != cudaSuccess) return nhp_fail(nullptr, NHP_ERR_CUDA, "cudaGetDeviceProperties: %s", cudaGetErrorString(e));
    if (prop.major != 10)
        return nhp_fail(nullptr, NHP_ERR_NO_DEVICE, "nhp_create: device %d is sm_%d%d; libnhp is built for sm_100a only", device, prop.major, prop.minor);
    nhp_ctx *ctx = new nhp_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = (int)prop.sharedMemPerBlockOptin;
    if (cudaSetDevice(device) != cudaSuccess || cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreate(&ctx->ev0) != cudaSuccess || cudaEventCreate(&ctx->ev1) != cudaSuccess ||
        cudaMalloc(&ctx->d_flag, sizeof(int)) != cudaSuccess || cudaMalloc(&ctx->d_winstat, 2 * sizeof(int64_t)) != cudaSuccess) {
        int rc = nhp_fail(nullptr, NHP_ERR_CUDA, "nhp_create: %s", cudaGetErrorString(cudaGetLastError()));
        delete ctx;
        return rc;
    }
    ctx->own_stream = ctx->stream;
    {   // keep freed event buffers in the device's stream-ordered pool: mle!/mcmc! drivers (and the e2e bench) upload
        // data sets of the same size over and over, and cudaFree of multi-GB buffers costs tens of milliseconds
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
    }
    cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), ctx->stream);
    *out = ctx;
    return NHP_OK;
}

static void free_cont(nhp_ctx *ctx) {
    cudaFree(ctx->d_lambda0); cudaFree(ctx->d_W); cudaFree(ctx->d_A); cudaFree(ctx->d_p1); cudaFree(ctx->d_p2);
    cudaFree(ctx->d_table); cudaFree(ctx->d_rowsum); cudaFree(ctx->d_rowsum_w); cudaFree(ctx->d_abits);
    cudaFree(ctx->d_stats0); cudaFree(ctx->d_stats1); cudaFree(ctx->d_xbar);
    cudaFree(ctx->d_adj_tw); cudaFree(ctx->d_adj_dec); ctx->d_adj_dec = nullptr; cudaFree(ctx->d_adj_rho); cudaFree(ctx->d_adj_u); cudaFree(ctx->d_adj_A); cudaFree(ctx->d_save);
    ctx->d_save = nullptr;
    ctx->d_adj_tw = nullptr; ctx->d_adj_rho = ctx->d_adj_u = ctx->d_adj_A = nullptr;
    ctx->d_lambda0 = ctx->d_W = ctx->d_A = ctx->d_p1 = ctx->d_p2 = ctx->d_rowsum = ctx->d_rowsum_w = nullptr;
    ctx->d_table = nullptr; ctx->d_abits = nullptr; ctx->d_stats0 = ctx->d_stats1 = ctx->d_xbar = nullptr;
    ctx->cap_K = 0;
}

extern "C" int nhp_destroy(nhp_ctx *ctx) {
    if (!ctx) return NHP_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    nhp_comm_destroy(ctx);
    nhp_cont_trace_free(ctx);
    nhp_disc_trace_free(ctx);
    nhp_disc_vb_trace_free(ctx);
    cudaFree(ctx->dv_q);
    nhp_big_flush(ctx);
    free_cont(ctx);
    cudaFree(ctx->d_partials); cudaFree(ctx->d_scratch); cudaFree(ctx->d_flag); cudaFree(ctx->d_winstat);
    cudaFree(ctx->dd_lambda0); cudaFree(ctx->dd_W); cudaFree(ctx->dd_A); cudaFree(ctx->dd_theta); cudaFree(ctx->dd_bump);
    cudaFree(ctx->dd_klist); cudaFree(ctx->dd_kptr); cudaFree(ctx->dd_btc); cudaFree(ctx->dd_counts); cudaFree(ctx->dd_kcnt); cudaFree(ctx->dd_ksum);
    cudaFree(ctx->d_bgrid_x); cudaFree(ctx->d_bgrid_v); cudaFree(ctx->d_bprior_L); cudaFree(ctx->d_slice);
    cudaFree(ctx->d_adj_ctl); cudaFree(ctx->d_adj_stat);
    cudaEventDestroy(ctx->ev0); cudaEventDestroy(ctx->ev1);
    cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return NHP_OK;
}

extern "C" int nhp_set_stream(nhp_ctx *ctx, void *cuda_stream) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->stream = cuda_stream ? (cudaStream_t)cuda_stream : ctx->own_stream;
    return NHP_OK;
}

extern "C" int nhp_set_option(nhp_ctx *ctx, int option, int64_t value) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    switch (option) {
        case NHP_OPT_SWEEP_LOGLIK: ctx->opt_sweep_ll = value != 0; ctx->sweep_ll_valid = false; return NHP_OK;
        default: return nhp_fail(ctx, NHP_ERR_INVALID, "nhp_set_option: unknown option %d", option);
    }
}

int nhp_scratch(nhp_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->scratch_cap) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_scratch);
        ctx->d_scratch = nullptr; ctx->scratch_cap = 0;
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_scratch, bytes));
        ctx->scratch_cap = bytes;
    }
    *out = ctx->d_scratch;
    return NHP_OK;
}

int nhp_partials(nhp_ctx *ctx, int64_t count, double **out) {
    if (count > ctx->partials_cap) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_partials);
        ctx->d_partials = nullptr; ctx->partials_cap = 0;
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_partials, (size_t)count * sizeof(double)));
        ctx->partials_cap = count;
    }
    *out = ctx->d_partials;
    return NHP_OK;
}

int nhp_timer_begin(nhp_ctx *ctx) {
    NHP_CUDA(ctx, cudaEventRecord(ctx->ev0, ctx->stream));
    return NHP_OK;
}
int nhp_timer_end(nhp_ctx *ctx) {
    NHP_CUDA(ctx, cudaEventRecord(ctx->ev1, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    float ms = 0.f;
    NHP_CUDA(ctx, cudaEventElapsedTime(&ms, ctx->ev0, ctx->ev1));
    ctx->last_ms = ms;
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// continuous data upload
// ---------------------------------------------------------------------------------------
// nodes Int64 1-based -> int32 0-based, validating range and ascending times.
__global__ void k_ingest_nodes(const int64_t *__restrict__ nodes64, const double *__restrict__ t, int *__restrict__ c, int64_t n, int64_t K, int *flag) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t v = nodes64[i];
    if (v < 1 || v > K) atomicOr(flag, 1);
    c[i] = (int)(v - 1);
    double ti = t[i];
    if (!(ti >= 0.0)) atomicOr(flag, 4);           // intensity(::HomogeneousProcess) throws for time < 0 (baselines.jl:111,116)
    if (i + 1 < n && !(t[i + 1] >= ti)) atomicOr(flag, 2);
}

// own-event counts per node (node_counts(nodes, K), parents.jl:61-68), block-privatised
__global__ void k_node_counts(const int *__restrict__ c, int64_t first, int64_t n, int K, double *__restrict__ Mn) {
    extern __shared__ int s_hist[];
    bool priv = K <= 8192;
    if (priv) {
        for (int k = threadIdx.x; k < K; k += blockDim.x) s_hist[k] = 0;
        __syncthreads();
    }
    for (int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        if (priv) atomicAdd(&s_hist[c[i]], 1);
        else atomicAdd(&Mn[c[i]], 1.0);
    }
    if (priv) {
        __syncthreads();
        for (int k = threadIdx.x; k < K; k += blockDim.x)
            if (s_hist[k]) atomicAdd(&Mn[k], (double)s_hist[k]);
    }
}

extern "C" int nhp_events_upload(nhp_ctx *ctx, const double *times, const int64_t *nodes, int64_t n, double duration, int64_t K,
                                 int64_t n_halo, int64_t index_base, int flags, nhp_events **out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "nhp_events_upload: ctx is NULL");
    NHP_CHECK(ctx, out != nullptr, NHP_ERR_INVALID, "nhp_events_upload: out is NULL");
    *out = nullptr;
    NHP_CHECK(ctx, n >= 0 && n < (int64_t)2147483000, NHP_ERR_INVALID, "nhp_events_upload: n=%lld outside [0, 2^31)", (long long)n);
    NHP_CHECK(ctx, K >= 1 && K <= 65536, NHP_ERR_INVALID, "nhp_events_upload: K=%lld outside [1, 65536]", (long long)K);
    NHP_CHECK(ctx, n_halo >= 0 && n_halo <= n, NHP_ERR_INVALID, "nhp_events_upload: n_halo=%lld outside [0, n]", (long long)n_halo);
    NHP_CHECK(ctx, index_base >= 0, NHP_ERR_INVALID, "nhp_events_upload: index_base < 0");
    NHP_CHECK(ctx, duration >= 0.0, NHP_ERR_INVALID, "nhp_events_upload: duration must be non-negative (baselines.jl:100)");
    NHP_CHECK(ctx, n == 0 || (times && nodes), NHP_ERR_INVALID, "nhp_events_upload: NULL times/nodes");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    nhp_events *ev = new nhp_events();
    ev->n = n; ev->n_halo = n_halo; ev->index_base = index_base; ev->flags = flags; ev->duration = duration; ev->K = K;
    const int64_t pad = 64;
    int rc = NHP_OK;
    auto cleanup = [&](int code) { nhp_events_free(ctx, ev); return code; };
    cudaStream_t as = ctx->stream;
    if (cudaMallocAsync(&ev->d_t, (size_t)(n + pad) * sizeof(double), as) != cudaSuccess || cudaMallocAsync(&ev->d_c, (size_t)(n + pad) * sizeof(int), as) != cudaSuccess ||
        cudaMallocAsync(&ev->d_poff, (size_t)(n + pad) * sizeof(int), as) != cudaSuccess || cudaMallocAsync(&ev->d_Mn, (size_t)K * sizeof(double), as) != cudaSuccess)
        return cleanup(nhp_fail(ctx, NHP_ERR_CUDA, "nhp_events_upload: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError())));
    cudaMemsetAsync(ev->d_t + n, 0, pad * sizeof(double), ctx->stream);
    cudaMemsetAsync(ev->d_c + n, 0, pad * sizeof(int), ctx->stream);
    cudaMemsetAsync(ev->d_poff, 0xFF, (size_t)(n + pad) * sizeof(int), ctx->stream);
    cudaMemsetAsync(ev->d_Mn, 0, (size_t)K * sizeof(double), ctx->stream);
    cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), ctx->stream);
    if (n > 0) {
        void *scratch = nullptr;
        rc = nhp_scratch(ctx, (size_t)n * sizeof(int64_t), &scratch);
        if (rc != NHP_OK) return cleanup(rc);
        if (cudaMemcpyAsync(ev->d_t, times, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess ||
            cudaMemcpyAsync(scratch, nodes, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream) != cudaSuccess)
            return cleanup(nhp_fail(ctx, NHP_ERR_CUDA, "nhp_events_upload: H2D copy failed: %s", cudaGetErrorString(cudaGetLastError())));
        int threads = 256;
        int64_t blocks = (n + threads - 1) / threads;
        k_ingest_nodes<<<(unsigned)blocks, threads, 0, ctx->stream>>>((const int64_t *)scratch, ev->d_t, ev->d_c, n, K, ctx->d_flag);
        NHP_LAUNCHED(ctx);
        if (n > n_halo) {
            int hb = (int)std::min<int64_t>((n - n_halo + 255) / 256, (int64_t)ctx->sm_count * 8);
            size_t sm = K <= 8192 ? (size_t)K * sizeof(int) : 0;
            k_node_counts<<<hb, 256, sm, ctx->stream>>>(ev->d_c, n_halo, n, (int)K, ev->d_Mn);
            NHP_LAUNCHED(ctx);
        }
    }
    int flag = 0;
    if (cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream) != cudaSuccess ||
        cudaStreamSynchronize(ctx->stream) != cudaSuccess)
        return cleanup(nhp_fail(ctx, NHP_ERR_CUDA, "nhp_events_upload: %s", cudaGetErrorString(cudaGetLastError())));
    if (flag & 1) return cleanup(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_events_upload: node outside 1..K"));
    if (flag & 2) return cleanup(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_events_upload: event times are not ascending"));
    if (flag & 4) return cleanup(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_events_upload: negative or NaN event time (baselines.jl:116)"));
    int64_t z = 0;
    while (z < n && times[z] == 0.0) z++;
    ev->n_t0 = z;
    *out = ev;
    return NHP_OK;
}

// An events handle around device-resident (times, 0-based nodes) arrays, e.g. the sample of nhp_cont_rand: the arrays are copied
// (device to device) into the handle's own padded buffers; times must be ascending and non-negative (validated).
__global__ void k_validate_sorted(const double *__restrict__ t, const int *__restrict__ c, int64_t n, int64_t K, int *flag, unsigned long long *n_t0) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double ti = t[i];
    if (c[i] < 0 || c[i] >= K) atomicOr(flag, 1);
    if (!(ti >= 0.0)) atomicOr(flag, 4);
    if (i + 1 < n && !(t[i + 1] >= ti)) atomicOr(flag, 2);
    if (ti == 0.0) atomicAdd(n_t0, 1ull);
}
int nhp_events_from_device(nhp_ctx *ctx, const double *d_t, const int *d_c, int64_t n, double duration, int64_t K, nhp_events **out) {
    *out = nullptr;
    NHP_CHECK(ctx, n >= 0 && n < (int64_t)2147483000, NHP_ERR_INVALID, "events: n=%lld outside [0, 2^31)", (long long)n);
    nhp_events *ev = new nhp_events();
    ev->n = n; ev->n_halo = 0; ev->index_base = 0; ev->flags = 1; ev->duration = duration; ev->K = K;
    const int64_t pad = 64;
    cudaStream_t as = ctx->stream;
    auto cleanup = [&](int code) { nhp_events_free(ctx, ev); return code; };
    if (cudaMallocAsync(&ev->d_t, (size_t)(n + pad) * sizeof(double), as) != cudaSuccess || cudaMallocAsync(&ev->d_c, (size_t)(n + pad) * sizeof(int), as) != cudaSuccess ||
        cudaMallocAsync(&ev->d_poff, (size_t)(n + pad) * sizeof(int), as) != cudaSuccess || cudaMallocAsync(&ev->d_Mn, (size_t)K * sizeof(double), as) != cudaSuccess)
        return cleanup(nhp_fail(ctx, NHP_ERR_CUDA, "events: cudaMalloc failed: %s", cudaGetErrorString(cudaGetLastError())));
    cudaMemsetAsync(ev->d_t + n, 0, pad * sizeof(double), as);
    cudaMemsetAsync(ev->d_c + n, 0, pad * sizeof(int), as);
    cudaMemsetAsync(ev->d_poff, 0xFF, (size_t)(n + pad) * sizeof(int), as);
    cudaMemsetAsync(ev->d_Mn, 0, (size_t)K * sizeof(double), as);
    cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), as);
    cudaMemsetAsync(ctx->d_winstat, 0, 2 * sizeof(int64_t), as);
    if (n > 0) {
        cudaMemcpyAsync(ev->d_t, d_t, (size_t)n * sizeof(double), cudaMemcpyDeviceToDevice, as);
        cudaMemcpyAsync(ev->d_c, d_c, (size_t)n * sizeof(int), cudaMemcpyDeviceToDevice, as);
        k_validate_sorted<<<(unsigned)((n + 255) / 256), 256, 0, as>>>(ev->d_t, ev->d_c, n, K, ctx->d_flag, (unsigned long long *)ctx->d_winstat);
        NHP_LAUNCHED(ctx);
        int hb = (int)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 8);
        size_t sm = K <= 8192 ? (size_t)K * sizeof(int) : 0;
        k_node_counts<<<hb, 256, sm, as>>>(ev->d_c, 0, n, (int)K, ev->d_Mn);
        NHP_LAUNCHED(ctx);
    }
    int flag = 0;
    unsigned long long nt0 = 0;
    if (cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, as) != cudaSuccess ||
        cudaMemcpyAsync(&nt0, ctx->d_winstat, sizeof(nt0), cudaMemcpyDeviceToHost, as) != cudaSuccess || cudaStreamSynchronize(as) != cudaSuccess)
        return cleanup(nhp_fail(ctx, NHP_ERR_CUDA, "events: %s", cudaGetErrorString(cudaGetLastError())));
    if (flag & 1) return cleanup(nhp_fail(ctx, NHP_ERR_INVALID, "events: node outside 1..K"));
    if (flag & 2) return cleanup(nhp_fail(ctx, NHP_ERR_INVALID, "events: event times are not ascending"));
    if (flag & 4) return cleanup(nhp_fail(ctx, NHP_ERR_INVALID, "events: negative or NaN event time (baselines.jl:116)"));
    ev->n_t0 = (int64_t)nt0;  // ascending times: the events at exactly t = 0 lead (quirk Q6)
    *out = ev;
    return NHP_OK;
}

// cached structure of the adjacency sampler (cont_adjacency.cu)
void *nhp_big_alloc(nhp_ctx *ctx, size_t bytes) {
    // the smallest cached block that holds the request without wasting more than half of itself
    int best = -1;
    for (int k = 0; k < (int)ctx->big_cache.size(); k++) {
        const size_t b = ctx->big_cache[k].second;
        if (b >= bytes && b <= bytes + bytes / 2 + (1u << 20) && (best < 0 || b < ctx->big_cache[best].second)) best = k;
    }
    if (best >= 0) {
        void *p = ctx->big_cache[best].first;
        ctx->big_cache.erase(ctx->big_cache.begin() + best);
        return p;
    }
    void *p = nullptr;
    if (cudaMalloc(&p, bytes) == cudaSuccess) return p;
    cudaGetLastError();
    nhp_big_flush(ctx);  // the cache itself may be what is in the way
    if (cudaMalloc(&p, bytes) == cudaSuccess) return p;
    cudaGetLastError();
    return nullptr;
}
void nhp_big_free(nhp_ctx *ctx, void *p, size_t bytes) {
    if (!p) return;
    if (!ctx || bytes == 0 || ctx->big_cache.size() >= 8) { cudaFree(p); return; }
    ctx->big_cache.emplace_back(p, bytes);  // kernels that still use it run on the context's stream, as will its next user
}
size_t nhp_big_cached_bytes(const nhp_ctx *ctx) {
    size_t t = 0;
    for (const auto &b : ctx->big_cache) t += b.second;
    return t;
}
void nhp_big_flush(nhp_ctx *ctx) {
    if (ctx->big_cache.empty()) return;
    cudaStreamSynchronize(ctx->stream);
    for (auto &b : ctx->big_cache) cudaFree(b.first);
    ctx->big_cache.clear();
}

void nhp_events_free_adjacency(nhp_ctx *ctx, nhp_events *ev, cudaStream_t s) {
    // the two entry arrays (up to 100+ GB) go to the context's block cache, the rest back to the stream-ordered pool: no device-wide
    // synchronisation, and the next structure of a similar size starts from warm memory
    nhp_big_free(ctx, ev->d_adj_i, ev->adj_bytes_i); nhp_big_free(ctx, ev->d_adj_dt, ev->adj_bytes_dt);
    ev->adj_bytes_i = ev->adj_bytes_dt = 0;
    void *blocks[] = {ev->d_adj_vstart, ev->d_adj_vnode, ev->d_adj_vbase, ev->d_adj_boff, ev->d_adj_lam, ev->d_adj_corder};
    ev->d_adj_corder = nullptr;
    for (void *b : blocks) if (b) cudaFreeAsync(b, s);
    ev->d_adj_vstart = ev->d_adj_vnode = ev->d_adj_boff = nullptr; ev->d_adj_vbase = nullptr; ev->d_adj_i = nullptr;
    ev->d_adj_dt = ev->d_adj_q = ev->d_adj_lam = nullptr;
    ev->adj_horizon = -1.0; ev->adj_impulse = -1; ev->adj_D = 0.0; ev->adj_total = 0; ev->adj_nv = 0;
}

extern "C" int nhp_events_free(nhp_ctx *ctx, nhp_events *ev) {
    if (!ev) return NHP_OK;
    if (ctx) {
        cudaSetDevice(ctx->device);
        cudaStream_t as = ctx->stream;  // stream-ordered: no device synchronisation, the blocks go back to the pool
        if (ev->d_t) cudaFreeAsync(ev->d_t, as);
        if (ev->d_c) cudaFreeAsync(ev->d_c, as);
        if (ev->d_poff) cudaFreeAsync(ev->d_poff, as);
        if (ev->d_Mn) cudaFreeAsync(ev->d_Mn, as);
        if (ev->d_tile_lo) cudaFreeAsync(ev->d_tile_lo, as);
        if (ev->d_wlen) cudaFreeAsync(ev->d_wlen, as);
    } else {
        cudaFree(ev->d_t); cudaFree(ev->d_c); cudaFree(ev->d_poff); cudaFree(ev->d_Mn); cudaFree(ev->d_tile_lo); cudaFree(ev->d_wlen);
    }
    {
        cudaStream_t as = ctx ? ctx->stream : nullptr;
        void *blocks[] = {ev->d_order, ev->d_node_ptr, ev->d_item_node, ev->d_item_e0, ev->d_lam0ev, ev->d_lam0bn, ev->d_lam0min,
                          ev->d_sl_g, ev->d_sl_item, ev->d_sl_t, ev->d_sl_part};
        for (void *b : blocks) if (b) cudaFreeAsync(b, as);
    }
    nhp_events_free_adjacency(ctx, ev, ctx ? ctx->stream : nullptr);
    delete ev;
    return NHP_OK;
}

extern "C" int64_t nhp_events_count(const nhp_events *ev) { return ev ? ev->n - ev->n_halo : 0; }

// ---------------------------------------------------------------------------------------
// continuous parameter tables
// ---------------------------------------------------------------------------------------
__global__ void k_build_table_ln(int K, const double *__restrict__ W, const double *__restrict__ A, const double *__restrict__ mu,
                                 const double *__restrict__ tau, double D, EntryLN *__restrict__ table, uint32_t *__restrict__ abits, int words) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)K * K) return;
    int c = (int)(e / K), p = (int)(e % K);
    int64_t src = p + (int64_t)K * c;
    double w = W[src];
    double a = A ? A[src] : 1.0;
    double t = tau[src];
    EntryLN en;
    en.cf = a * w * sqrt(t) * NHP_INVSQRT2PI * (D * D);
    en.mu = mu[src];
    en.h = 0.5 * t;
    en.pad = 0.0;
    table[e] = en;
    if (en.cf != 0.0) atomicOr(&abits[(int64_t)c * words + (p >> 5)], 1u << (p & 31));
}

__global__ void k_build_table_ex(int K, const double *__restrict__ W, const double *__restrict__ A, const double *__restrict__ theta,
                                 EntryEX *__restrict__ table, uint32_t *__restrict__ abits, int words) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)K * K) return;
    int c = (int)(e / K), p = (int)(e % K);
    int64_t src = p + (int64_t)K * c;
    double a = A ? A[src] : 1.0;
    EntryEX en;
    en.theta = theta[src];
    en.wt = a * W[src] * en.theta;
    table[e] = en;
    if (en.wt != 0.0) atomicOr(&abits[(int64_t)c * words + (p >> 5)], 1u << (p & 31));
}

// rowsum[p] = sum_c [A]W[p,c] in child order (continuous.jl:219-221 / 368-371); rowsum_w without A (Q3)
__global__ void k_rowsums(int K, const double *__restrict__ W, const double *__restrict__ A, double *__restrict__ rs, double *__restrict__ rsw) {
    int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= K) return;
    double s = 0.0, sw = 0.0;
    for (int c = 0; c < K; c++) {
        double w = W[p + (int64_t)K * c];
        sw += w;
        s += A ? A[p + (int64_t)K * c] * w : w;
    }
    rs[p] = s;
    rsw[p] = sw;
}

// masked parameter table, adjacency bit rows and row sums from the device-resident raw parameters (stream-ordered)
int nhp_cont_derive_tables(nhp_ctx *ctx) {
    const int64_t K = ctx->K, KK = K * K;
    cudaStream_t s = ctx->stream;
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_abits, 0, (size_t)(K * ctx->abits_words) * sizeof(uint32_t), s));
    unsigned blocks = (unsigned)((KK + 255) / 256);
    const double *dA = ctx->has_A ? ctx->d_A : nullptr;
    if (ctx->kind == NHP_LOGITNORMAL)
        k_build_table_ln<<<blocks, 256, 0, s>>>((int)K, ctx->d_W, dA, ctx->d_p1, ctx->d_p2, ctx->dtmax, (EntryLN *)ctx->d_table, ctx->d_abits, (int)ctx->abits_words);
    else
        k_build_table_ex<<<blocks, 256, 0, s>>>((int)K, ctx->d_W, dA, ctx->d_p1, (EntryEX *)ctx->d_table, ctx->d_abits, (int)ctx->abits_words);
    NHP_LAUNCHED(ctx);
    k_rowsums<<<(unsigned)((K + 127) / 128), 128, 0, s>>>((int)K, ctx->d_W, dA, ctx->d_rowsum, ctx->d_rowsum_w);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

extern "C" int nhp_cont_params_set(nhp_ctx *ctx, int kind, int64_t K, const double *lambda0, const double *W, const double *A,
                                   const double *p1, const double *p2, double dtmax) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "nhp_cont_params_set: ctx is NULL");
    NHP_CHECK(ctx, kind == NHP_EXPONENTIAL || kind == NHP_LOGITNORMAL, NHP_ERR_INVALID, "nhp_cont_params_set: unknown impulse kind %d", kind);
    NHP_CHECK(ctx, K >= 1 && K <= 65536, NHP_ERR_INVALID, "nhp_cont_params_set: K=%lld outside [1, 65536]", (long long)K);
    NHP_CHECK(ctx, lambda0 && W && p1, NHP_ERR_INVALID, "nhp_cont_params_set: NULL parameter array");
    NHP_CHECK(ctx, kind == NHP_EXPONENTIAL || p2 != nullptr, NHP_ERR_INVALID, "nhp_cont_params_set: LogitNormal needs tau (p2)");
    NHP_CHECK(ctx, dtmax > 0.0, NHP_ERR_INVALID, "nhp_cont_params_set: dtmax must be positive");
    if (ctx->bgrid_n > 0) { ctx->bgrid_n = 0; ctx->bgrid_version++; }  // a new parameter set starts from its homogeneous lambda0; curves are re-applied with nhp_cont_baseline_grid
    ctx->bprior_n = 0;  // and their prior with nhp_cont_baseline_prior
    NHP_CHECK(ctx, kind == NHP_EXPONENTIAL || std::isfinite(dtmax), NHP_ERR_INVALID, "nhp_cont_params_set: LogitNormal needs a finite dtmax");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t KK = K * K;
    // host-side scan: validation (baselines.jl:32) + horizon inputs + density
    double l0min = std::numeric_limits<double>::infinity(), l0sum = 0.0;
    for (int64_t k = 0; k < K; k++) {
        NHP_CHECK(ctx, lambda0[k] >= 0.0, NHP_ERR_INVALID, "HomogeneousProcess: intensity parameter lambda must be non-negative (baselines.jl:32)");
        l0min = std::min(l0min, lambda0[k]);
        l0sum += lambda0[k];
    }
    double thmin = std::numeric_limits<double>::infinity(), wtmax = 0.0, thmin_all = thmin, wtmax_all = 0.0;
    int64_t nnz = 0;
    for (int64_t e = 0; e < KK; e++) {
        double w = A ? A[e] * W[e] : W[e];
        if (w != 0.0) {
            nnz++;
            if (kind == NHP_EXPONENTIAL) { thmin = std::min(thmin, p1[e]); wtmax = std::max(wtmax, fabs(w * p1[e])); }
        }
        // the adjacency sampler also evaluates the links that are currently off (continuous.jl:477-483)
        if (kind == NHP_EXPONENTIAL && W[e] != 0.0) { thmin_all = std::min(thmin_all, p1[e]); wtmax_all = std::max(wtmax_all, fabs(W[e] * p1[e])); }
    }
    if (ctx->cap_K != K) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        free_cont(ctx);
        StatsLayout sl{K};
        int64_t words = (((K + 31) / 32) + 7) & ~(int64_t)7;  // bit rows padded to 32 bytes (256-bit gathers)
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_lambda0, (size_t)K * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_W, (size_t)KK * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_A, (size_t)KK * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_p1, (size_t)KK * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_p2, (size_t)KK * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_table, (size_t)KK * sizeof(EntryLN)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_rowsum, (size_t)K * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_rowsum_w, (size_t)K * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_abits, (size_t)(K * words) * sizeof(uint32_t)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_stats0, (size_t)sl.total() * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_stats1, (size_t)KK * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_xbar, (size_t)KK * sizeof(double)));
        NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats0, 0, (size_t)sl.total() * sizeof(double), ctx->stream));
        NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats1, 0, (size_t)KK * sizeof(double), ctx->stream));
        ctx->abits_words = words;
        ctx->cap_K = K;
    }
    ctx->cont_set = false;
    ctx->sweep_ll_valid = false;
    ctx->kind = kind; ctx->K = K; ctx->dtmax = dtmax; ctx->has_A = (A != nullptr);
    ctx->density = (double)nnz / (double)KK;
    ctx->theta_min = thmin; ctx->wt_max = wtmax; ctx->lambda0_min = l0min; ctx->lambda0_sum = l0sum;
    ctx->theta_min_all = thmin_all; ctx->wt_max_all = wtmax_all;
    { double as = 0.0; if (A) for (int64_t e = 0; e < KK; e++) as += A[e]; ctx->a_sum = A ? as : (double)KK; }
    cudaStream_t s = ctx->stream;
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_lambda0, lambda0, (size_t)K * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_W, W, (size_t)KK * sizeof(double), cudaMemcpyHostToDevice, s));
    if (A) NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_A, A, (size_t)KK * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_p1, p1, (size_t)KK * sizeof(double), cudaMemcpyHostToDevice, s));
    if (p2) NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_p2, p2, (size_t)KK * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_TRY(nhp_cont_derive_tables(ctx));
    NHP_CUDA(ctx, cudaStreamSynchronize(s)); // host arrays may be reused by the caller after return
    ctx->cont_set = true;
    return NHP_OK;
}
