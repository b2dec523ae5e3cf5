// cont_rand.cu -- rand(process::ContinuousHawkesProcess, duration)  (continuous.jl:16-37, 131-142, 335-348) on the device.
//
// The reference simulates the cluster (branching) representation recursively: baseline events per node from a
// homogeneous Poisson process (baselines.jl:67-70), and every event on node p spawns, on every child node c with
// A[p,c] = 1, Poisson(W[p,c]) children (weights.jl:25-27) at lags drawn from the impulse response (impulses.jl:63-66,
// 196-202); events beyond the duration are dropped.  Here the recursion becomes a breadth-first loop over generations:
//   generation 0  n_k ~ Poisson(lambda0_k T) per node, times uniform on [0, T]; with LogGaussianCox curves set
//                 (nhp_cont_baseline_grid) an inhomogeneous Poisson process per node instead, drawn cell by cell of the grid
//                 (Poisson count of the trapezoid area, times by the exact inverse CDF of the linear rate on the cell);
//   generation g+1  every event of generation g draws its TOTAL number of children m ~ Poisson(sum_c A W[p,c]) and then each
//                   child's node from Categorical(A W[p,:] / sum) -- by Poisson superposition / thinning exactly the law of
//                   independent Poisson(W[p,c]) counts per child node -- and its lag from the (p, c) impulse response;
// a prefix sum over the child counts places every generation behind the previous one in one buffer, and a final radix
// sort by time (the bit pattern of a non-negative double is order preserving) gives the (events, nodes) stream, which
// is left device resident as an events handle: 1e8-event true Hawkes samples for benchmarks and chain tests without
// a host round trip.  Random numbers: Philox4x32-10 keyed (seed ^ "RANDHAWK"; element, generation | draw, 0).
// Parity with the reference is distributional (Julia's own samplers are not reproducible from uniforms).
#include "rand_stream.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <vector>

__global__ void k_rand_base_counts(int K, const double *__restrict__ lambda0, double T, uint64_t seed, long long *__restrict__ counts) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= K) return;
    RandStream r(seed, (uint64_t)k, 0x80000000u);
    counts[k] = r.poisson(lambda0[k] * T);
}
// first event index of every node -> (time, node) of generation 0
__global__ void k_rand_base_emit(int K, const long long *__restrict__ off, double T, uint64_t seed, double *__restrict__ t, int *__restrict__ c, long long n0) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n0) return;
    int lo = 0, hi = K;  // node k with off[k] <= e < off[k+1]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= e) lo = mid; else hi = mid; }
    RandStream r(seed, (uint64_t)e, 0u);
    t[e] = r.uniform() * T;
    c[e] = lo;
}
// Generation 0 of a LogGaussianCox baseline: an inhomogeneous Poisson process with the piecewise-linear rate of the sweeps
// (cont_baseline.cu).  Cell i = (k, g), k = i / (G-1), is grid interval g of node k clipped to [0, T]; the rate is linear on it,
// from a at its left end to b at its right end (the interpolation formula of grid_interp, interpolation.jl:31).
__device__ __forceinline__ void rand_curve_cell(const double *__restrict__ x, const double *__restrict__ v, int G, long long i, double T, double *lo, double *hi,
                                                double *a, double *b) {
    const int k = (int)(i / (G - 1)), g = (int)(i - (long long)k * (G - 1));
    const double x0 = x[g], x1 = x[g + 1], y0 = v[(int64_t)k * G + g], y1 = v[(int64_t)k * G + g + 1];
    const double l = fmax(x0, 0.0), r = fmin(x1, T);
    *lo = l; *hi = r;
    *a = (y1 * (l - x0) + y0 * (x1 - l)) / (x1 - x0);
    *b = (y1 * (r - x0) + y0 * (x1 - r)) / (x1 - x0);
}
// per cell: Poisson(trapezoid area of the clipped cell)
__global__ void k_rand_curve_counts(long long ncell, int G, const double *__restrict__ x, const double *__restrict__ v, double T, uint64_t seed,
                                    long long *__restrict__ counts) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ncell) return;
    double lo, hi, a, b;
    rand_curve_cell(x, v, G, i, T, &lo, &hi, &a, &b);
    RandStream r(seed, (uint64_t)i, 0x80000001u);
    counts[i] = hi > lo ? r.poisson(0.5 * (a + b) * (hi - lo)) : 0;
}
// first event index of every cell -> (time, node): the inverse CDF of the linear density on the cell,
//   s = h u (a + b) / (a + sqrt(a^2 + u (b^2 - a^2))),   exact for a = 0, b = 0 and a = b alike (a cell with a = b = 0 has no events)
__global__ void k_rand_curve_emit(long long ncell, int G, const long long *__restrict__ off, const double *__restrict__ x, const double *__restrict__ v, double T,
                                  uint64_t seed, double *__restrict__ t, int *__restrict__ c, long long n0) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n0) return;
    long long lo = 0, hi = ncell;  // cell i with off[i] <= e < off[i+1]
    while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (off[mid] <= e) lo = mid; else hi = mid; }
    double l, rt, a, b;
    rand_curve_cell(x, v, G, lo, T, &l, &rt, &a, &b);
    RandStream r(seed, (uint64_t)e, 0x80000002u);
    const double u = r.uniform();
    const double sd = (rt - l) * u * (a + b) / (a + sqrt(a * a + u * (b * b - a * a)));
    t[e] = fmin(l + sd, rt);
    c[e] = (int)(lo / (G - 1));
}
// number of children of every event of the current generation
__global__ void k_rand_child_counts(const double *__restrict__ t, const int *__restrict__ c, long long g0, long long ng, const double *__restrict__ rowsum, double T,
                                    uint64_t seed, uint32_t gen, long long *__restrict__ counts) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ng) return;
    const int p = c[g0 + i];
    long long m = 0;
    if (p >= 0 && t[g0 + i] <= T) {
        RandStream r(seed, (uint64_t)(g0 + i), gen * 2u + 1u);
        m = r.poisson(rowsum[p]);
    }
    counts[i] = m;
}
template <int KIND>
__global__ void k_rand_child_emit(double *__restrict__ t, int *__restrict__ c, long long g0, long long ng, const long long *__restrict__ off, long long total,
                                  long long out0, int K, const int *__restrict__ row_n, const int *__restrict__ row_c, const double *__restrict__ row_cum,
                                  const double *__restrict__ p1, const double *__restrict__ p2, double D, double T, uint64_t seed, uint32_t gen) {
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= total) return;
    long long lo = 0, hi = ng;  // parent i with off[i] <= s < off[i+1]
    while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (off[mid] <= s) lo = mid; else hi = mid; }
    const double tp = t[g0 + lo];
    const int p = c[g0 + lo];
    RandStream r(seed, (uint64_t)(out0 + s), gen * 2u + 2u);
    // child node: Categorical(A W[p,:] / rowsum) by inversion on the row's running sums
    const int nr = row_n[p];
    const double *cum = row_cum + (int64_t)p * K;
    const double target = r.uniform() * cum[nr - 1];
    int a = 0, b = nr - 1;
    while (a < b) { const int mid = (a + b) >> 1; if (cum[mid] > target) b = mid; else a = mid + 1; }
    const int cc = row_c[(int64_t)p * K + a];
    const int64_t kk = p + (int64_t)K * cc;
    double dt;
    if (KIND == NHP_EXPONENTIAL) dt = -log(r.uniform()) / p1[kk];                    // rand(Exponential(1/theta))        impulses.jl:63-66
    else dt = D / (1.0 + exp(-(p1[kk] + r.normal() / sqrt(p2[kk]))));                 // dtmax * rand(LogitNormal(mu, sigma)) impulses.jl:196-202
    const double tc = tp + dt;
    t[out0 + s] = tc;
    c[out0 + s] = tc <= T ? cc : -1;  // truncate(childevents, duration)   continuous.jl:39-48
}
// sort key: the time's bit pattern; dropped events get the largest key and are counted
__global__ void k_rand_keys(const double *__restrict__ t, const int *__restrict__ c, long long n, unsigned long long *__restrict__ keys, unsigned long long *__restrict__ ndrop) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const bool drop = c[i] < 0;
    keys[i] = drop ? ~0ull : (unsigned long long)__double_as_longlong(t[i]);
    if (drop) atomicAdd(ndrop, 1ull);
}
__global__ void k_rand_unkey(const unsigned long long *__restrict__ keys, long long n, double *__restrict__ t) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) t[i] = __longlong_as_double((long long)keys[i]);
}

#define R_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fin(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__)); } while (0)

extern "C" int nhp_cont_rand(nhp_ctx *ctx, double duration, uint64_t seed, int64_t max_events, nhp_events **out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, out != nullptr, NHP_ERR_INVALID, "nhp_cont_rand: out is NULL");
    *out = nullptr;
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set (call nhp_cont_params_set)");
    NHP_CHECK(ctx, duration > 0.0 && std::isfinite(duration), NHP_ERR_INVALID, "nhp_cont_rand: duration must be positive and finite");
    NHP_CHECK(ctx, max_events >= 1 && max_events < (int64_t)2147483000, NHP_ERR_INVALID, "nhp_cont_rand: max_events outside [1, 2^31)");
    const bool curves = ctx->bgrid_n > 0;
    NHP_CHECK(ctx, !curves || (ctx->bgrid_lo <= 0.0 && ctx->bgrid_hi >= duration), NHP_ERR_INVALID,
              "nhp_cont_rand: the curves' grid [%g, %g] does not cover [0, duration = %g]", ctx->bgrid_lo, ctx->bgrid_hi, duration);
    const int64_t ncell = curves ? ctx->K * (ctx->bgrid_n - 1) : 0;  // generation 0 with curves: one Poisson count per (node, grid interval)
    NHP_CHECK(ctx, ncell < (int64_t)2147483000, NHP_ERR_INVALID, "nhp_cont_rand: K (n_grid - 1) = %lld cells exceed 2^31", (long long)ncell);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int K = (int)ctx->K;
    const int64_t cap = max_events;
    cudaStream_t s = ctx->stream;
    double *d_t = nullptr, *d_t2 = nullptr, *row_cum = nullptr;
    int *d_c = nullptr, *d_c2 = nullptr, *row_n = nullptr, *row_c = nullptr;
    long long *d_cnt = nullptr, *d_off = nullptr;
    unsigned long long *d_keys = nullptr, *d_keys2 = nullptr, *d_drop = nullptr;
    void *d_tmp = nullptr;
    auto fin = [&](int rc) {
        cudaStreamSynchronize(s);
        cudaFree(d_t); cudaFree(d_t2); cudaFree(row_cum); cudaFree(d_c); cudaFree(d_c2); cudaFree(row_n); cudaFree(row_c); cudaFree(d_cnt); cudaFree(d_off);
        cudaFree(d_keys); cudaFree(d_keys2); cudaFree(d_drop); cudaFree(d_tmp);
        return rc;
    };
    R_CUDA(cudaMalloc(&d_t, (size_t)cap * sizeof(double)));
    R_CUDA(cudaMalloc(&d_c, (size_t)cap * sizeof(int)));
    R_CUDA(cudaMalloc(&row_n, (size_t)K * sizeof(int)));
    R_CUDA(cudaMalloc(&row_c, (size_t)K * K * sizeof(int)));
    R_CUDA(cudaMalloc(&row_cum, (size_t)K * K * sizeof(double)));
    R_CUDA(cudaMalloc(&d_drop, sizeof(unsigned long long)));
    k_rand_rows<<<(K + 7) / 8, 256, 0, s>>>(K, ctx->d_W, ctx->has_A ? ctx->d_A : nullptr, row_n, row_c, row_cum);
    NHP_LAUNCHED(ctx);
    // ---- generation 0
    const int64_t cnt_cap = std::max<int64_t>(K, 1 << 20);
    int64_t cnt_len = cnt_cap;
    R_CUDA(cudaMalloc(&d_cnt, (size_t)(cnt_len + 1) * sizeof(long long)));
    R_CUDA(cudaMalloc(&d_off, (size_t)(cnt_len + 1) * sizeof(long long)));
    size_t tmp_bytes = 0, need = 0;
    auto ensure_tmp = [&](size_t bytes) -> cudaError_t {
        if (bytes <= tmp_bytes) return cudaSuccess;
        cudaStreamSynchronize(s);
        cudaFree(d_tmp); d_tmp = nullptr; tmp_bytes = 0;
        cudaError_t e = cudaMalloc(&d_tmp, bytes);
        if (e == cudaSuccess) tmp_bytes = bytes;
        return e;
    };
    auto ensure_cnt = [&](int64_t len) -> cudaError_t {
        if (len <= cnt_len) return cudaSuccess;
        cudaStreamSynchronize(s);
        cudaFree(d_cnt); cudaFree(d_off); d_cnt = d_off = nullptr;
        cnt_len = len;
        cudaError_t e = cudaMalloc(&d_cnt, (size_t)(len + 1) * sizeof(long long));
        if (e == cudaSuccess) e = cudaMalloc(&d_off, (size_t)(len + 1) * sizeof(long long));
        return e;
    };
    // exclusive scan of d_cnt[0..len) into d_off[0..len]; returns the total
    auto scan_total = [&](int64_t len, long long *total) -> int {
        R_CUDA(cudaMemsetAsync(d_cnt + len, 0, sizeof(long long), s));
        cub::DeviceScan::ExclusiveSum(nullptr, need, d_cnt, d_off, (int)(len + 1), s);
        R_CUDA(ensure_tmp(need));
        R_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_cnt, d_off, (int)(len + 1), s));
        NHP_LAUNCHED(ctx);
        R_CUDA(cudaMemcpyAsync(total, d_off + len, sizeof(long long), cudaMemcpyDeviceToHost, s));
        R_CUDA(cudaStreamSynchronize(s));
        return NHP_OK;
    };
    long long n0 = 0;
    if (curves) {  // inhomogeneous: the curves of nhp_cont_baseline_grid, cell by cell
        const int G = (int)ctx->bgrid_n;
        R_CUDA(ensure_cnt(ncell));
        k_rand_curve_counts<<<(unsigned)((ncell + 255) / 256), 256, 0, s>>>(ncell, G, ctx->d_bgrid_x, ctx->d_bgrid_v, duration, seed, d_cnt);
        NHP_LAUNCHED(ctx);
        { int rc = scan_total(ncell, &n0); if (rc != NHP_OK) return rc; }
    } else {
        k_rand_base_counts<<<(K + 127) / 128, 128, 0, s>>>(K, ctx->d_lambda0, duration, seed, d_cnt);
        NHP_LAUNCHED(ctx);
        { int rc = scan_total(K, &n0); if (rc != NHP_OK) return rc; }
    }
    if (n0 > cap) return fin(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_cont_rand: the sample needs more than max_events = %lld events (generation 0 alone has %lld)", (long long)cap, n0));
    if (n0 > 0 && curves) {
        k_rand_curve_emit<<<(unsigned)((n0 + 255) / 256), 256, 0, s>>>(ncell, (int)ctx->bgrid_n, d_off, ctx->d_bgrid_x, ctx->d_bgrid_v, duration, seed, d_t, d_c, n0);
        NHP_LAUNCHED(ctx);
    } else if (n0 > 0) {
        k_rand_base_emit<<<(unsigned)((n0 + 255) / 256), 256, 0, s>>>(K, d_off, duration, seed, d_t, d_c, n0);
        NHP_LAUNCHED(ctx);
    }
    // ---- later generations
    long long g0 = 0, ng = n0, total_n = n0;
    for (uint32_t gen = 1; ng > 0 && gen < 100000u; gen++) {
        R_CUDA(ensure_cnt(ng));
        k_rand_child_counts<<<(unsigned)((ng + 255) / 256), 256, 0, s>>>(d_t, d_c, g0, ng, ctx->d_rowsum, duration, seed, gen, d_cnt);
        NHP_LAUNCHED(ctx);
        long long nchild = 0;
        { int rc = scan_total(ng, &nchild); if (rc != NHP_OK) return rc; }
        if (total_n + nchild > cap)
            return fin(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_cont_rand: the sample needs more than max_events = %lld events (is the process stable?)", (long long)cap));
        if (nchild > 0) {
            if (ctx->kind == NHP_LOGITNORMAL)
                k_rand_child_emit<NHP_LOGITNORMAL><<<(unsigned)((nchild + 255) / 256), 256, 0, s>>>(d_t, d_c, g0, ng, d_off, nchild, total_n, K, row_n, row_c, row_cum, ctx->d_p1,
                                                                                                     ctx->d_p2, ctx->dtmax, duration, seed, gen);
            else
                k_rand_child_emit<NHP_EXPONENTIAL><<<(unsigned)((nchild + 255) / 256), 256, 0, s>>>(d_t, d_c, g0, ng, d_off, nchild, total_n, K, row_n, row_c, row_cum, ctx->d_p1,
                                                                                                     nullptr, ctx->dtmax, duration, seed, gen);
            NHP_LAUNCHED(ctx);
        }
        g0 = total_n; ng = nchild; total_n += nchild;
    }
    R_CUDA(cudaGetLastError());
    // ---- drop the truncated events, sort by time
    int64_t n_keep = 0;
    if (total_n > 0) {
        R_CUDA(cudaMalloc(&d_keys, (size_t)total_n * sizeof(unsigned long long)));
        R_CUDA(cudaMalloc(&d_keys2, (size_t)total_n * sizeof(unsigned long long)));
        R_CUDA(cudaMalloc(&d_c2, (size_t)total_n * sizeof(int)));
        R_CUDA(cudaMemsetAsync(d_drop, 0, sizeof(unsigned long long), s));
        k_rand_keys<<<(unsigned)((total_n + 255) / 256), 256, 0, s>>>(d_t, d_c, total_n, d_keys, d_drop);
        NHP_LAUNCHED(ctx);
        cub::DeviceRadixSort::SortPairs(nullptr, need, d_keys, d_keys2, d_c, d_c2, (int)total_n, 0, 64, s);
        R_CUDA(ensure_tmp(need));
        R_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tmp_bytes, d_keys, d_keys2, d_c, d_c2, (int)total_n, 0, 64, s));
        NHP_LAUNCHED(ctx);
        unsigned long long nd = 0;
        R_CUDA(cudaMemcpyAsync(&nd, d_drop, sizeof(nd), cudaMemcpyDeviceToHost, s));
        R_CUDA(cudaStreamSynchronize(s));
        n_keep = total_n - (int64_t)nd;
        if (n_keep > 0) {
            k_rand_unkey<<<(unsigned)((n_keep + 255) / 256), 256, 0, s>>>(d_keys2, n_keep, d_t);
            NHP_LAUNCHED(ctx);
        }
    }
    nhp_events *ev = nullptr;
    int rc = nhp_events_from_device(ctx, d_t, d_c2, n_keep, duration, K, &ev);
    if (rc != NHP_OK) return fin(rc);
    *out = ev;
    return fin(NHP_OK);
}

// the (events, nodes) arrays of a device-resident handle, in Julia's conventions (Float64 times, 1-based Int64 nodes)
__global__ void k_nodes_to_int64(const int *__restrict__ c, int64_t n, int64_t *__restrict__ out) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = (int64_t)c[i] + 1;
}
extern "C" int nhp_events_download(nhp_ctx *ctx, nhp_events *ev, double *times, int64_t *nodes, double *duration) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "nhp_events_download: events handle is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t own = ev->n - ev->n_halo;
    if (duration) *duration = ev->duration;
    if (own == 0) return NHP_OK;
    cudaStream_t s = ctx->stream;
    if (times) NHP_CUDA(ctx, cudaMemcpyAsync(times, ev->d_t + ev->n_halo, (size_t)own * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (nodes) {
        void *scratch;
        NHP_TRY(nhp_scratch(ctx, (size_t)own * sizeof(int64_t), &scratch));
        k_nodes_to_int64<<<(unsigned)((own + 255) / 256), 256, 0, s>>>(ev->d_c + ev->n_halo, own, (int64_t *)scratch);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaMemcpyAsync(nodes, scratch, (size_t)own * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    }
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}
