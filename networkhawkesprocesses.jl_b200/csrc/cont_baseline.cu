// cont_baseline.cu -- inhomogeneous baselines inside the sweeps: LogGaussianCoxProcess (baselines.jl:187-336).
//
// The reference's LGCP baseline is lambda0_k(t) = LinearInterpolator(x, lambda[k])(t) (utils/interpolation.jl:27-36): piecewise
// linear on a grid x[0..G), y_G at t = x_G exactly, DomainError outside [x_0, x_G]; its integral is the trapezoid sum.  On the hot path
// it enters (i) the total intensity of every event (log-likelihood, parent weights "baseline last"), (ii) the compensator
// sum_k integrate(lambda0_k), and (iii) the elliptical-slice update of the curve itself, whose likelihood per node is
// -integrate(f) + sum over the events ATTRIBUTED TO THE BASELINE of log f(t) (baselines.jl:228-254: split_extract + loglikelihood).
//   * nhp_cont_baseline_grid keeps the curves on the device; the sweeps then read a per-event baseline rate (k_event_baseline, cached
//     with the events handle per curve version) instead of lambda0[node] -- one extra 8-byte stream, no grid search in the hot loops;
//   * nhp_cont_baseline_loglik evaluates the slice sampler's likelihood for all K nodes at once from the device-resident parent
//     assignment (parent offset 0 = baseline): the reference's split_extract never materialises.
#include "nhp_internal.cuh"
#include <algorithm>
#include <vector>

// value of the piecewise-linear curve (x[G], y[G]) at t; *bad is raised outside the support (the reference throws a DomainError)
__device__ __forceinline__ double grid_interp(const double *__restrict__ x, const double *__restrict__ y, int G, double t, int *bad) {
    if (!(t >= x[0]) || !(t <= x[G - 1])) { *bad = 1; return y[0]; }
    int lo = 0, hi = G - 1;  // last g with x[g] <= t
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (x[mid] <= t) lo = mid; else hi = mid; }
    if (t >= x[G - 1]) return y[G - 1];
    const double x0 = x[lo], x1 = x[lo + 1];
    return (y[lo + 1] * (t - x0) + y[lo] * (x1 - t)) / (x1 - x0);  // interpolation.jl:31
}

__global__ void k_event_baseline(const double *__restrict__ t, const int *__restrict__ c, int64_t n, const double *__restrict__ x, const double *__restrict__ v, int G,
                                 double *__restrict__ out, int *__restrict__ flag) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int bad = 0;
    out[i] = grid_interp(x, v + (int64_t)c[i] * G, G, t[i], &bad);
    if (bad) atomicOr(flag, 256);
}

// per-node slice-sampler likelihood terms: ll[k] += log f_k(t_i) for the own events of node k whose parent is the baseline
__global__ void k_baseline_loglik(const double *__restrict__ t, const int *__restrict__ c, const int *__restrict__ poff, int64_t first, int64_t n, const double *__restrict__ x,
                                  const double *__restrict__ v, int G, double *__restrict__ ll, int *__restrict__ flag) {
    for (int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
        const int po = poff[i];
        if (po < 0) atomicOr(flag, 512);  // no parent assignment on the device
        if (po != 0) continue;
        int bad = 0;
        const int k = c[i];
        const double f = grid_interp(x, v + (int64_t)k * G, G, t[i], &bad);
        if (bad) atomicOr(flag, 256);
        red_add_f64(ll + k, log(f));
    }
}

static double trapezoid(const double *x, const double *y, int64_t G) {
    double s = 0.0;
    for (int64_t g = 0; g + 1 < G; g++) s += 0.5 * (y[g] + y[g + 1]) * (x[g + 1] - x[g]);
    return s;
}

static int check_grid(nhp_ctx *ctx, int64_t G, const double *x, const double *values, int64_t K, const char *who) {
    NHP_CHECK(ctx, G >= 2 && G < (1 << 24) && x && values, NHP_ERR_INVALID, "%s: need a grid of at least two points and its values", who);
    for (int64_t g = 0; g + 1 < G; g++) NHP_CHECK(ctx, x[g + 1] > x[g], NHP_ERR_INVALID, "%s: the grid must be strictly increasing", who);
    for (int64_t e = 0; e < K * G; e++) NHP_CHECK(ctx, values[e] >= 0.0 && values[e] <= 1.7976931348623157e308, NHP_ERR_INVALID, "%s: baseline values must be finite and non-negative", who);
    return NHP_OK;
}

extern "C" int nhp_cont_baseline_grid(nhp_ctx *ctx, int64_t n_grid, const double *x, const double *values) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "nhp_cont_baseline_grid: set the continuous parameters first (the curves replace lambda0 of that model)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    ctx->bgrid_version++;
    ctx->sweep_ll_valid = false; ctx->parents_valid = false;
    if (n_grid == 0) {  // back to the homogeneous lambda0
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
        cudaFree(ctx->d_bgrid_x); cudaFree(ctx->d_bgrid_v);
        ctx->d_bgrid_x = ctx->d_bgrid_v = nullptr; ctx->bgrid_n = 0; ctx->baseline_integral = 0.0;
        ctx->bprior_n = 0;
        return NHP_OK;
    }
    const int64_t K = ctx->K;
    NHP_TRY(check_grid(ctx, n_grid, x, values, K, "nhp_cont_baseline_grid"));
    if (ctx->bgrid_n != n_grid) {
        ctx->bprior_n = 0;  // a prior of another grid size does not apply
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
        cudaFree(ctx->d_bgrid_x); cudaFree(ctx->d_bgrid_v);
        ctx->d_bgrid_x = ctx->d_bgrid_v = nullptr; ctx->bgrid_n = 0;
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_bgrid_x, (size_t)n_grid * sizeof(double)));
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_bgrid_v, (size_t)(K * n_grid) * sizeof(double)));
    }
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bgrid_x, x, (size_t)n_grid * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bgrid_v, values, (size_t)(K * n_grid) * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->bgrid_n = n_grid;
    double tot = 0.0, mn = 1.7976931348623157e308;
    for (int64_t k = 0; k < K; k++) tot += trapezoid(x, values + k * n_grid, n_grid);  // integrated_intensity(p::LogGaussianCoxProcess, duration), baselines.jl:336
    for (int64_t e = 0; e < K * n_grid; e++) mn = std::min(mn, values[e]);
    ctx->baseline_integral = tot;
    ctx->bgrid_min = mn;
    ctx->lambda0_min = mn;  // the Exponential cut-off horizon measures the omitted tail against the smallest baseline rate
    return NHP_OK;
}

// the per-event baseline rates of `ev` for the context's current curves (NULL: homogeneous baseline)
int nhp_cont_event_baseline(nhp_ctx *ctx, nhp_events *ev, const double **lam0ev) {
    *lam0ev = nullptr;
    if (ctx->bgrid_n == 0) return NHP_OK;
    if (ev->d_lam0ev && ev->lam0ev_version == ctx->bgrid_version) { *lam0ev = ev->d_lam0ev; return NHP_OK; }
    cudaStream_t s = ctx->stream;
    if (!ev->d_lam0ev) NHP_CUDA(ctx, cudaMallocAsync(&ev->d_lam0ev, (size_t)std::max<int64_t>(ev->n, 1) * sizeof(double), s));
    if (ev->n > 0) {
        NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
        k_event_baseline<<<(unsigned)((ev->n + 255) / 256), 256, 0, s>>>(ev->d_t, ev->d_c, ev->n, ctx->d_bgrid_x, ctx->d_bgrid_v, (int)ctx->bgrid_n, ev->d_lam0ev, ctx->d_flag);
        NHP_LAUNCHED(ctx);
        int flag = 0;
        NHP_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
        NHP_CHECK(ctx, !(flag & 256), NHP_ERR_INVALID, "baseline: an event time is outside the interpolation support of the grid (interpolation.jl:29)");
    }
    ev->lam0ev_version = ctx->bgrid_version;
    *lam0ev = ev->d_lam0ev;
    return NHP_OK;
}

// one CTA per node: its events' rates in the by-node order, and their minimum
__global__ void k_event_baseline_bynode(const double *__restrict__ lam0ev, const int *__restrict__ order, const int *__restrict__ node_ptr, int K,
                                        double *__restrict__ bynode, double *__restrict__ colmin) {
    __shared__ double s_min[32];
    for (int c = blockIdx.x; c < K; c += gridDim.x) {
        double m = INFINITY;
        for (int e = node_ptr[c] + threadIdx.x; e < node_ptr[c + 1]; e += blockDim.x) {
            const double v = lam0ev[order[e]];
            bynode[e] = v;
            m = fmin(m, v);
        }
        for (int d = 16; d > 0; d >>= 1) m = fmin(m, __shfl_xor_sync(0xffffffffu, m, d));
        if ((threadIdx.x & 31) == 0) s_min[threadIdx.x >> 5] = m;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); w++) m = fmin(m, s_min[w]);
            colmin[c] = m;
        }
        __syncthreads();
    }
}

// The adjacency sampler's view of the curves: the per-event rates in the by-node order of the handle (a column chunk's initial
// intensities are one contiguous read) and their minimum per node, the lower bound of every intensity of the column without any
// parent's share (certification bound and floor of the sweep).  Rebuilt with the per-event rates, for the same curve version.
int nhp_cont_event_baseline_bynode(nhp_ctx *ctx, nhp_events *ev, const double **lam0bn, const double **lam0min) {
    *lam0bn = *lam0min = nullptr;
    if (ctx->bgrid_n == 0) return NHP_OK;
    const double *lam0ev = nullptr;
    NHP_TRY(nhp_cont_event_baseline(ctx, ev, &lam0ev));
    if (!(ev->d_lam0bn && ev->lam0bn_version == ctx->bgrid_version)) {
        NHP_TRY(nhp_events_build_node_index(ctx, ev));
        cudaStream_t s = ctx->stream;
        const int64_t K = ev->K, own = ev->n - ev->n_halo;
        if (!ev->d_lam0bn) NHP_CUDA(ctx, cudaMallocAsync(&ev->d_lam0bn, (size_t)std::max<int64_t>(own, 1) * sizeof(double), s));
        if (!ev->d_lam0min) NHP_CUDA(ctx, cudaMallocAsync(&ev->d_lam0min, (size_t)K * sizeof(double), s));
        k_event_baseline_bynode<<<(unsigned)std::min<int64_t>(K, (int64_t)ctx->sm_count * 8), 256, 0, s>>>(lam0ev, ev->d_order, ev->d_node_ptr, (int)K, ev->d_lam0bn,
                                                                                                         ev->d_lam0min);
        NHP_LAUNCHED(ctx);
        ev->lam0min.resize((size_t)K);
        NHP_CUDA(ctx, cudaMemcpyAsync(ev->lam0min.data(), ev->d_lam0min, (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
        ev->lam0bn_version = ctx->bgrid_version;
    }
    *lam0bn = ev->d_lam0bn;
    *lam0min = ev->d_lam0min;
    return NHP_OK;
}

double nhp_cont_baseline_term(const nhp_ctx *ctx, const nhp_events *ev) {
    if (!(ev->flags & 1)) return 0.0;  // exactly one shard adds the baseline integral
    return ctx->bgrid_n > 0 ? ctx->baseline_integral : ctx->lambda0_sum * ev->duration;
}

// loglikelihood(process::LogGaussianCoxProcess, data, node, y) for every node at once (baselines.jl:247-254), with data =
// split_extract(data, parents, nnodes) read off the device-resident parent assignment of the last parent sweep:
//   ll[k] = -integrate(f_k) + sum_{i on k, parent(i) = baseline} log f_k(t_i),   f_k = LinearInterpolator(x, values[k])
// For a time shard the sums cover the shard's own events and the integral is added on the shard with flags bit 0.
extern "C" int nhp_cont_baseline_loglik(nhp_ctx *ctx, nhp_events *ev, int64_t n_grid, const double *x, const double *values, double *ll) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev != nullptr && ll != nullptr, NHP_ERR_INVALID, "nhp_cont_baseline_loglik: NULL argument");
    NHP_CHECK(ctx, ctx->cont_set && ev->K == ctx->K, NHP_ERR_STATE, "nhp_cont_baseline_loglik: parameters not set for this data");
    NHP_CHECK(ctx, ctx->parents_valid, NHP_ERR_STATE, "nhp_cont_baseline_loglik: no parent assignment on the device (run nhp_cont_resample_parents first)");
    const int64_t K = ctx->K;
    NHP_TRY(check_grid(ctx, n_grid, x, values, K, "nhp_cont_baseline_loglik"));
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    void *scratch = nullptr;
    NHP_TRY(nhp_scratch(ctx, (size_t)(n_grid + K * n_grid + K) * sizeof(double), &scratch));
    double *dx = (double *)scratch, *dv = dx + n_grid, *dll = dv + K * n_grid;
    NHP_CUDA(ctx, cudaMemcpyAsync(dx, x, (size_t)n_grid * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(dv, values, (size_t)(K * n_grid) * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaMemsetAsync(dll, 0, (size_t)K * sizeof(double), s));
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
    NHP_TRY(nhp_timer_begin(ctx));
    const int64_t own = ev->n - ev->n_halo;
    if (own > 0) {
        const int grid = (int)std::min<int64_t>((own + 255) / 256, (int64_t)ctx->sm_count * 16);
        k_baseline_loglik<<<grid, 256, 0, s>>>(ev->d_t, ev->d_c, ev->d_poff, ev->n_halo, ev->n, dx, dv, (int)n_grid, dll, ctx->d_flag);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
    }
    int flag = 0;
    NHP_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ll, dll, (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_TRY(nhp_timer_end(ctx));
    NHP_CHECK(ctx, !(flag & 256), NHP_ERR_INVALID, "baseline: an event time is outside the interpolation support of the grid (interpolation.jl:29)");
    NHP_CHECK(ctx, !(flag & 512), NHP_ERR_STATE, "nhp_cont_baseline_loglik: events without a parent assignment");
    if (ev->flags & 1) for (int64_t k = 0; k < K; k++) ll[k] -= trapezoid(x, values + k * n_grid, n_grid);
    return NHP_OK;
}
