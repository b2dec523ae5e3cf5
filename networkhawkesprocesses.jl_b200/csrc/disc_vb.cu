// disc_vb.cu -- the discrete mean-field VB step on the device (`update!`, discrete.jl:369-375; `vb!`, inference.jl:153-181).
//
// The state q is the reference's variational_params vector (discrete.jl:204-209) kept with the context:
//   q = [alphav(N); betav(N); gammav(N^2 B); kappav(N^2); nuv(N^2)],  gammav[p + N(c + N b)], kappav[p + N c], nuv[p + N c].
// One step: k_vb_expect turns q into the exp-expectations e0[c] and ET[c][p*B + b] (the statistics kernels' layout, so there is no
// transpose), nhp_disc_vb_reduce runs the responsibilities and reductions of nhp_disc_vb_stats, k_vb_update writes the new q in place
// and reduces the largest relative change.  Only that scalar crosses PCIe.
//
// Stochastic VI (Hoffman et al. 2013; the reference's `svi!` is an empty stub) runs the same step on a window of n of the T bins,
// (t_begin + j) mod T for j < n: the statistics of the window only, scaled by s = T / n, give the target q*, and q moves to
// (1 - step) q + step q*.  The VB step is the window of all T bins with (s, step) = (1, 1), which is the plain update bit for bit.
#include "nhp_internal.cuh"
#include <algorithm>
#include <cmath>

static size_t vb_q_doubles(int64_t N, int64_t B) { return (size_t)(2 * N) + (size_t)(N * N) * (size_t)(B + 2); }

// one thread per (p, c), e = p + N c: B + 2 digammas; threads e < N also write e0[e]
//   e0[c]             = exp(psi(alphav[c]) - log betav[c])                                       baselines.jl:454-456
//   ET[c][p*B + b]    = exp((psi(gammav[p,c,b]) - psi(sum_b gammav[p,c,:])) + (psi(kappav[p,c]) - log nuv[p,c]))
//                                                                       impulses.jl:373-375 + weights.jl:95-97, summed as update_ does
__global__ void __launch_bounds__(256) k_vb_expect(const double *__restrict__ q, int N, int B, double *__restrict__ e0, double *__restrict__ ET) {
    const int64_t NN = (int64_t)N * N;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= NN) return;
    const double *gv = q + 2 * N, *kv = gv + NN * B, *nv = kv + NN;
    if (e < N) e0[e] = exp(nhp_digamma(q[e]) - log(q[N + e]));
    double S = 0.0;
    for (int b = 0; b < B; b++) S += gv[e + NN * b];
    const double psiS = nhp_digamma(S), lw = nhp_digamma(kv[e]) - log(nv[e]);
    double *out = ET + e * B;  // c*N*B + p*B = (p + N c) * B
    for (int b = 0; b < B; b++) out[b] = exp((nhp_digamma(gv[e + NN * b]) - psiS) + lw);
}

__device__ __forceinline__ double rel_change(double nw, double old) { return fabs(nw - old) / old; }

__device__ __forceinline__ double blend(double old, double target, double step) { return (1.0 - step) * old + step * target; }

// in place, one thread per (p, c) (+ alphav, betav for e < N), the targets
//   gammav* = gamma + s g,  kappav* = kappa + s sum_b g (b = 0 .. B-1, as k_vb_finish),  nuv* = nu + s events[p],
//   alphav* = alpha0 + s alpha_sum,  betav* = betav_new (1/beta0 + T dt, computed on the host, unscaled)
// blended as q = (1 - step) q + step q*;  change = max |new - old| / old over all of q (bit order of non-negative doubles is their
// numeric order: an integer atomicMax per warp)
__global__ void __launch_bounds__(256) k_vb_update(double *__restrict__ q, const double *__restrict__ gammaT, const double *__restrict__ alpha_sum,
                                                   const double *__restrict__ events, int N, int B, double alpha0, double betav_new, double kappa,
                                                   double nu, double gamma, double s, double step, unsigned long long *__restrict__ change) {
    const int64_t NN = (int64_t)N * N;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double mx = 0.0;
    if (e < NN) {
        double *gv = q + 2 * N, *kv = gv + NN * B, *nv = kv + NN;
        const double *g = gammaT + e * B;
        double ks = 0.0;
#pragma unroll 1  // unrolled, the divisions' slow-path calls make ptxas spill
        for (int b = 0; b < B; b++) {
            const double gb = g[b];
            ks += gb;
            const double old = gv[e + NN * b], nw = blend(old, gamma + s * gb, step);
            mx = fmax(mx, rel_change(nw, old));
            gv[e + NN * b] = nw;
        }
        const double kn = blend(kv[e], kappa + s * ks, step), nn = blend(nv[e], nu + s * events[e % N], step);
        mx = fmax(mx, fmax(rel_change(kn, kv[e]), rel_change(nn, nv[e])));
        kv[e] = kn;
        nv[e] = nn;
        if (e < N) {
            const double an = blend(q[e], alpha0 + s * alpha_sum[e], step), bn = blend(q[N + e], betav_new, step);
            mx = fmax(mx, fmax(rel_change(an, q[e]), rel_change(bn, q[N + e])));
            q[e] = an;
            q[N + e] = bn;
        }
    }
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, d));
    if ((threadIdx.x & 31) == 0 && mx > 0.0) atomicMax(change, (unsigned long long)__double_as_longlong(mx));
}

extern "C" int nhp_disc_vb_set(nhp_ctx *ctx, int64_t N, int64_t B, double dt, const double *hyper, int n_hyper, const double *q) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, N >= 1 && N <= 32768 && B >= 1, NHP_ERR_INVALID, "nhp_disc_vb_set: bad dimensions N=%lld B=%lld", (long long)N, (long long)B);
    NHP_CHECK(ctx, hyper != nullptr && q != nullptr, NHP_ERR_INVALID, "nhp_disc_vb_set: NULL argument");
    NHP_CHECK(ctx, n_hyper == 5, NHP_ERR_INVALID, "nhp_disc_vb_set: expected 5 hyper-parameters, got %d", n_hyper);
    NHP_CHECK(ctx, dt > 0.0 && std::isfinite(dt), NHP_ERR_INVALID, "nhp_disc_vb_set: dt must be positive and finite");
    for (int i = 0; i < n_hyper; i++)
        NHP_CHECK(ctx, hyper[i] > 0.0 && std::isfinite(hyper[i]), NHP_ERR_INVALID, "nhp_disc_vb_set: hyper-parameter %d must be positive and finite", i);
    const size_t n = vb_q_doubles(N, B);
    for (size_t i = 0; i < n; i++)
        NHP_CHECK(ctx, q[i] > 0.0 && std::isfinite(q[i]), NHP_ERR_INVALID, "nhp_disc_vb_set: q[%zu] = %g is not positive and finite", i, q[i]);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->dv_cap < n) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->dv_q); ctx->dv_q = nullptr; ctx->dv_cap = 0; ctx->dv_set = false;
        NHP_CUDA(ctx, cudaMalloc(&ctx->dv_q, n * sizeof(double)));
        ctx->dv_cap = n;
    }
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->dv_q, q, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the caller may reuse q after return
    ctx->dv_N = N; ctx->dv_B = B; ctx->dv_dt = dt;
    for (int i = 0; i < 5; i++) ctx->dv_hyper[i] = hyper[i];
    ctx->dv_set = true;
    return NHP_OK;
}

extern "C" int nhp_disc_vb_get(nhp_ctx *ctx, double *q) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->dv_set, NHP_ERR_STATE, "nhp_disc_vb_get: no VB state (call nhp_disc_vb_set)");
    NHP_CHECK(ctx, q != nullptr, NHP_ERR_INVALID, "nhp_disc_vb_get: NULL argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CUDA(ctx, cudaMemcpyAsync(q, ctx->dv_q, vb_q_doubles(ctx->dv_N, ctx->dv_B) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

// One step over the window (t_begin + j) mod T, j < n_bins, blended with `step`; the refusals come before anything changes.  The window
// of all T bins uses the events per node kept with the data, a shorter one counts them in its ranges.
static int vb_window_step(nhp_ctx *ctx, nhp_disc *dd, const char *fn, int64_t t_begin, int64_t n_bins, double step, double *change) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr, NHP_ERR_INVALID, "%s: data handle is NULL", fn);
    NHP_CHECK(ctx, dd->t_halo == 0, NHP_ERR_UNSUPPORTED, "%s works on unsharded data", fn);
    NHP_CHECK(ctx, !(ctx->comm && ctx->nranks > 1), NHP_ERR_UNSUPPORTED, "%s runs on one GPU (the context has a communicator of %d ranks)", fn, ctx->nranks);
    NHP_CHECK(ctx, ctx->dv_set, NHP_ERR_STATE, "%s: no VB state (call nhp_disc_vb_set)", fn);
    NHP_CHECK(ctx, dd->d_conv != nullptr, NHP_ERR_STATE, "%s: call nhp_disc_convolve first", fn);
    const int64_t N = ctx->dv_N, B = ctx->dv_B, NN = N * N, NB = N * B, T = dd->T;
    NHP_CHECK(ctx, dd->N == N && dd->B == B, NHP_ERR_INVALID, "%s: the VB state has N=%lld B=%lld, the data N=%lld B=%lld", fn, (long long)N,
              (long long)B, (long long)dd->N, (long long)dd->B);
    NHP_CHECK(ctx, ctx->dv_trace_cap == 0 || (ctx->dv_trace_N == N && ctx->dv_trace_B == B), NHP_ERR_STATE,
              "%s: the open VB trace was begun for N=%lld B=%lld", fn, (long long)ctx->dv_trace_N, (long long)ctx->dv_trace_B);
    NHP_CHECK(ctx, t_begin >= 0 && t_begin < T && n_bins >= 1 && n_bins <= T, NHP_ERR_INVALID,
              "%s: window (t_begin=%lld, n_bins=%lld) outside 0 <= t_begin < T, 1 <= n_bins <= T (T=%lld)", fn, (long long)t_begin, (long long)n_bins, (long long)T);
    NHP_CHECK(ctx, step > 0.0 && step <= 1.0, NHP_ERR_INVALID, "%s: step=%g outside (0, 1]", fn, step);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    void *scratch;
    // layout: e0[N] | ET[N*NB] | gammaT[N*NB] | alpha_sum[N] | events[N] | change (the last four zeroed together)
    NHP_TRY(nhp_scratch(ctx, (size_t)(3 * N + 2 * NB * N + 1) * sizeof(double), &scratch));
    double *d_e0 = (double *)scratch, *d_ET = d_e0 + N, *d_gT = d_ET + NB * N, *d_alpha = d_gT + NB * N, *d_events = d_alpha + N, *d_change = d_events + N;
    NHP_CUDA(ctx, cudaMemsetAsync(d_gT, 0, (size_t)(NB * N + 2 * N + 1) * sizeof(double), s));
    const unsigned blocks = (unsigned)((NN + 255) / 256);
    k_vb_expect<<<blocks, 256, 0, s>>>(ctx->dv_q, (int)N, (int)B, d_e0, d_ET);
    NHP_LAUNCHED(ctx);
    // the window as at most two ranges [t_begin, end) and, when it wraps, [0, t_begin + n_bins - T)
    const int64_t end = std::min(t_begin + n_bins, T), wrap = t_begin + n_bins - end;
    NHP_TRY(nhp_disc_vb_reduce(ctx, dd, t_begin, end, d_e0, d_ET, d_alpha, d_gT));
    NHP_TRY(nhp_disc_vb_reduce(ctx, dd, 0, wrap, d_e0, d_ET, d_alpha, d_gT));
    const double *events = nhp_disc_rowsum(dd);
    if (n_bins < T) {
        NHP_TRY(nhp_disc_range_events(ctx, dd, t_begin, end, d_events));
        NHP_TRY(nhp_disc_range_events(ctx, dd, 0, wrap, d_events));
        events = d_events;
    }
    const double *h = ctx->dv_hyper;
    const double betav = 1.0 / h[1] + (double)T * ctx->dv_dt;  // baselines.jl:450 as written (1 / beta0, not beta0)
    const double scale = (double)T / (double)n_bins;
    k_vb_update<<<blocks, 256, 0, s>>>(ctx->dv_q, d_gT, d_alpha, events, (int)N, (int)B, h[0], betav, h[2], h[3], h[4], scale, step,
                                       (unsigned long long *)d_change);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    if (ctx->dv_trace_cap > 0 && ctx->dv_trace_len < ctx->dv_trace_cap) {  // the state of this step stays on the device
        const size_t n = vb_q_doubles(N, B);
        NHP_CUDA(ctx, cudaMemcpyAsync(ctx->dv_trace + (size_t)ctx->dv_trace_len * n, ctx->dv_q, n * sizeof(double), cudaMemcpyDeviceToDevice, s));
        ctx->dv_trace_len++;
    }
    if (change) {
        NHP_CUDA(ctx, cudaMemcpyAsync(change, d_change, sizeof(double), cudaMemcpyDeviceToHost, s));
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
    }
    return NHP_OK;
}

extern "C" int nhp_disc_vb_step(nhp_ctx *ctx, nhp_disc *dd, double *change) {
    return vb_window_step(ctx, dd, "nhp_disc_vb_step", 0, dd ? dd->T : 1, 1.0, change);
}

extern "C" int nhp_disc_svi_step(nhp_ctx *ctx, nhp_disc *dd, int64_t t_begin, int64_t n_bins, double step, double *change) {
    return vb_window_step(ctx, dd, "nhp_disc_svi_step", t_begin, n_bins, step, change);
}

extern "C" int nhp_disc_vb_trace_free(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->dv_trace);
    ctx->dv_trace = nullptr; ctx->dv_trace_cap = ctx->dv_trace_len = 0;
    return NHP_OK;
}

extern "C" int nhp_disc_vb_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->dv_set, NHP_ERR_STATE, "nhp_disc_vb_trace_begin: no VB state (the slot size follows it; call nhp_disc_vb_set)");
    NHP_CHECK(ctx, capacity >= 1, NHP_ERR_INVALID, "nhp_disc_vb_trace_begin: capacity must be positive");
    NHP_TRY(nhp_disc_vb_trace_free(ctx));
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = vb_q_doubles(ctx->dv_N, ctx->dv_B);
    if (cudaMalloc(&ctx->dv_trace, (size_t)capacity * n * sizeof(double)) != cudaSuccess) {
        cudaGetLastError();
        ctx->dv_trace = nullptr;
        return nhp_fail(ctx, NHP_ERR_CUDA, "nhp_disc_vb_trace_begin: cannot allocate %lld slots of %.2f MB", (long long)capacity, 1e-6 * (double)(n * 8));
    }
    ctx->dv_trace_cap = capacity; ctx->dv_trace_len = 0; ctx->dv_trace_N = ctx->dv_N; ctx->dv_trace_B = ctx->dv_B;
    return NHP_OK;
}

extern "C" int nhp_disc_vb_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    if (count) *count = ctx->dv_trace_len;
    if (capacity) *capacity = ctx->dv_trace_cap;
    return NHP_OK;
}

extern "C" int nhp_disc_vb_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *q_out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, first >= 0 && count >= 0 && first + count <= ctx->dv_trace_len, NHP_ERR_INVALID, "nhp_disc_vb_trace_read: slots [%lld, %lld) outside the %lld stored",
              (long long)first, (long long)(first + count), (long long)ctx->dv_trace_len);
    if (count == 0) return NHP_OK;
    NHP_CHECK(ctx, q_out != nullptr, NHP_ERR_INVALID, "nhp_disc_vb_trace_read: NULL argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t n = vb_q_doubles(ctx->dv_trace_N, ctx->dv_trace_B);
    NHP_CUDA(ctx, cudaMemcpyAsync(q_out, ctx->dv_trace + (size_t)first * n, (size_t)count * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}
