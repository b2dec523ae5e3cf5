// disc_vb.cu -- the discrete mean-field VB step on the device (`update!`, discrete.jl:369-375; `vb!`, inference.jl:153-181).
//
// The state q is the reference's variational_params vector (discrete.jl:204-209) kept with the context (ctx->dvb, a VbState:
// vb_state.cu holds its upload, read-back and trace):
//   q = [alphav(N); betav(N); gammav(N^2 B); kappav(N^2); nuv(N^2)],  gammav[p + N(c + N b)], kappav[p + N c], nuv[p + N c].
// One step: k_dvb_expect turns q into the exp-expectations e0[c] and ET[c][p*B + b] (the statistics kernels' layout, so there is no
// transpose), nhp_disc_vb_reduce runs the responsibilities and reductions of nhp_disc_vb_stats, k_dvb_update writes the new q in place
// and reduces the largest relative change.  Only that scalar crosses PCIe.
//
// Stochastic VI (Hoffman et al. 2013; the reference's `svi!` is an empty stub) runs the same step on a window of n of the T bins,
// (t_begin + j) mod T for j < n: the statistics of the window only, scaled by s = T / n, give the target q*, and q moves to
// (1 - step) q + step q*.  The VB step is the window of all T bins with (s, step) = (1, 1), which is the plain update bit for bit.
//
// A network state (nhp_disc_vb_network_set) fits the Gamma mixture W | A=1 ~ Gamma(kappa, nu), W | A=0 ~ Gamma(kappa0, nu0),
// A ~ Bernoulli(rho), rho ~ Beta(alpha_rho, beta_rho) with the factors q(W | A=1) = Gamma(kappav, nuv), q(W | A=0) = Gamma(kappa0v,
// nu0v), q(A=1) = pv, q(rho) = Beta(alpharhov, betarhov) appended to q.  The step reuses nhp_disc_vb_reduce as it is: the network
// instantiations of the two kernels (NET = true) add the mixture E[ln W] to the expectations and write the per-link targets and block
// sums of the new q(A=1), and k_vbn_finish adds those sums in a fixed order into q(rho).
#include "vb_network.cuh"  // rel_change, blend, stable_sigmoid, vb_block_reduce, k_vbn_finish
#include <algorithm>
#include <cmath>

// the standard layout; a network state appends kappa0v(N^2); nu0v(N^2); pv(N^2); alpharhov; betarhov
static size_t vb_state_doubles(int64_t N, int64_t B, bool network) {
    return (size_t)(2 * N) + (size_t)(N * N) * (size_t)(B + (network ? 5 : 2)) + (network ? 2 : 0);
}

// one thread per (p, c), e = p + N c: B + 2 digammas; threads e < N also write e0[e]
//   e0[c]             = exp(psi(alphav[c]) - log betav[c])                                       baselines.jl:454-456
//   ET[c][p*B + b]    = exp((psi(gammav[p,c,b]) - psi(sum_b gammav[p,c,:])) + E[ln W[p,c]])
//   E[ln W[p,c]]      = psi(kappav) - log nuv                                                    impulses.jl:373-375 + weights.jl:95-97,
//                                                                                               summed as update_ does
// NET: the mixture E[ln W[p,c]] = pv (psi(kappav) - log nuv) + (1 - pv) (psi(kappa0v) - log nu0v), and thread 0 writes
// lrho = psi(alpharhov) - psi(betarhov), the prior log-odds of a link
template <bool NET>
__global__ void __launch_bounds__(256) k_dvb_expect(const double *__restrict__ q, int N, int B, double *__restrict__ e0, double *__restrict__ ET,
                                                    double *__restrict__ lrho) {
    const int64_t NN = (int64_t)N * N;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= NN) return;
    const double *gv = q + 2 * N, *kv = gv + NN * B, *nv = kv + NN;
    if (e < N) e0[e] = exp(nhp_digamma(q[e]) - log(q[N + e]));
    double lw = nhp_digamma(kv[e]) - log(nv[e]);
    if constexpr (NET) {
        const double *k0v = nv + NN, *n0v = k0v + NN, *pv = n0v + NN;
        if (e == 0) *lrho = nhp_digamma(pv[NN]) - nhp_digamma(pv[NN + 1]);
        const double p = pv[e];
        lw = p * lw + (1.0 - p) * (nhp_digamma(k0v[e]) - log(n0v[e]));
    }
    double S = 0.0;
    for (int b = 0; b < B; b++) S += gv[e + NN * b];
    const double psiS = nhp_digamma(S);
    double *out = ET + e * B;  // c*N*B + p*B = (p + N c) * B
    for (int b = 0; b < B; b++) out[b] = exp((nhp_digamma(gv[e + NN * b]) - psiS) + lw);
}

// in place, one thread per (p, c) (+ alphav, betav for e < N); with ks = sum_b g (b = 0 .. B-1, as k_vb_finish) and E = events[p]
//   gammav* = gamma + s g,  kappav* = kappa + s ks,  nuv* = nu + s E,  alphav* = alpha0 + s alpha_sum,
//   betav* = betav_new (1/beta0 + T dt, computed on the host, unscaled)
// blended as q = (1 - step) q + step q*;  change = max |new - old| / old over all of q (vb_block_reduce).
// NET: also kappa0v* = kappa0 + s ks,  nu0v* = nu0 + s E,
//   pv* = sigmoid(lrho + [lgamma(kappav*) - kappav* log nuv*] - [lgamma(kappa0v*) - kappa0v* log nu0v*] + cprior)
// where cprior = [kappa log nu - lgamma(kappa)] - [kappa0 log nu0 - lgamma(kappa0)] (the brackets are the log marginal likelihoods of
// the link's statistics under slab and spike); change takes |new - old| over pv, which may be exactly 0 or 1, and each block writes
// the sum of its pv* to psum[blockIdx.x]
template <bool NET>
__global__ void __launch_bounds__(256) k_dvb_update(double *__restrict__ q, const double *__restrict__ gammaT, const double *__restrict__ alpha_sum,
                                                    const double *__restrict__ events, const double *__restrict__ lrho, int N, int B, double alpha0,
                                                    double betav_new, double kappa, double nu, double gamma, double kappa0, double nu0, double cprior,
                                                    double s, double step, unsigned long long *__restrict__ change, double *__restrict__ psum) {
    const int64_t NN = (int64_t)N * N;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double mx = 0.0, pt = 0.0;
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
        const double ev = s * events[e % N], k1 = kappa + s * ks, n1 = nu + ev;
        const double kn = blend(kv[e], k1, step), nn = blend(nv[e], n1, step);
        mx = fmax(mx, fmax(rel_change(kn, kv[e]), rel_change(nn, nv[e])));
        if constexpr (NET) {
            double *k0v = nv + NN, *n0v = k0v + NN, *pv = n0v + NN;
            const double k0 = kappa0 + s * ks, n0 = nu0 + ev;
            pt = stable_sigmoid(*lrho + (lgamma(k1) - k1 * log(n1)) - (lgamma(k0) - k0 * log(n0)) + cprior);
            const double k0n = blend(k0v[e], k0, step), n0n = blend(n0v[e], n0, step), pn = blend(pv[e], pt, step);
            mx = fmax(mx, fmax(rel_change(k0n, k0v[e]), rel_change(n0n, n0v[e])));
            mx = fmax(mx, fabs(pn - pv[e]));
            k0v[e] = k0n; n0v[e] = n0n; pv[e] = pn;
        }
        kv[e] = kn;
        nv[e] = nn;
        if (e < N) {
            const double an = blend(q[e], alpha0 + s * alpha_sum[e], step), bn = blend(q[N + e], betav_new, step);
            mx = fmax(mx, fmax(rel_change(an, q[e]), rel_change(bn, q[N + e])));
            q[e] = an;
            q[N + e] = bn;
        }
    }
    vb_block_reduce<NET>(mx, pt, change, psum);
}

// the two set calls: every entry of hyper positive and finite; every entry of q positive and finite except, for a network state,
// pv (in [0, 1]); refused before anything changes
static int vb_set_state(nhp_ctx *ctx, const char *fn, bool network, int64_t N, int64_t B, double dt, const double *hyper, int n_hyper, const double *q) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, N >= 1 && N <= 32768 && B >= 1, NHP_ERR_INVALID, "%s: bad dimensions N=%lld B=%lld", fn, (long long)N, (long long)B);
    NHP_CHECK(ctx, hyper != nullptr && q != nullptr, NHP_ERR_INVALID, "%s: NULL argument", fn);
    const int want = network ? 9 : 5;
    NHP_CHECK(ctx, n_hyper == want, NHP_ERR_INVALID, "%s: expected %d hyper-parameters, got %d", fn, want, n_hyper);
    NHP_CHECK(ctx, dt > 0.0 && std::isfinite(dt), NHP_ERR_INVALID, "%s: dt must be positive and finite", fn);
    for (int i = 0; i < n_hyper; i++)
        NHP_CHECK(ctx, hyper[i] > 0.0 && std::isfinite(hyper[i]), NHP_ERR_INVALID, "%s: hyper-parameter %d must be positive and finite", fn, i);
    const size_t n = vb_state_doubles(N, B, network);
    const size_t p_lo = network ? (size_t)(2 * N) + (size_t)(N * N) * (size_t)(B + 4) : n, p_hi = network ? p_lo + (size_t)(N * N) : n;
    VbState &st = ctx->dvb;
    NHP_TRY(nhp_vb_state_set(ctx, st, fn, q, n, n, 0, 0, p_lo, p_hi, N, B, network));
    st.dt = dt;
    for (int i = 0; i < n_hyper; i++) st.hyper[i] = hyper[i];
    return NHP_OK;
}

extern "C" int nhp_disc_vb_set(nhp_ctx *ctx, int64_t N, int64_t B, double dt, const double *hyper, int n_hyper, const double *q) {
    return vb_set_state(ctx, "nhp_disc_vb_set", false, N, B, dt, hyper, n_hyper, q);
}

extern "C" int nhp_disc_vb_network_set(nhp_ctx *ctx, int64_t N, int64_t B, double dt, const double *hyper, int n_hyper, const double *q) {
    return vb_set_state(ctx, "nhp_disc_vb_network_set", true, N, B, dt, hyper, n_hyper, q);
}

extern "C" int nhp_disc_vb_get(nhp_ctx *ctx, double *q) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    return nhp_vb_state_get(ctx, ctx->dvb, "nhp_disc_vb_get", "nhp_disc_vb_set", q);
}

// One step over the window (t_begin + j) mod T, j < n_bins, blended with `step`; the refusals come before anything changes.  The window
// of all T bins uses the events per node kept with the data, a shorter one counts them in its ranges.
static int vb_window_step(nhp_ctx *ctx, nhp_disc *dd, const char *fn, int64_t t_begin, int64_t n_bins, double step, double *change) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr, NHP_ERR_INVALID, "%s: data handle is NULL", fn);
    NHP_CHECK(ctx, dd->t_halo == 0, NHP_ERR_UNSUPPORTED, "%s works on unsharded data", fn);
    NHP_CHECK(ctx, !(ctx->comm && ctx->nranks > 1), NHP_ERR_UNSUPPORTED, "%s runs on one GPU (the context has a communicator of %d ranks)", fn, ctx->nranks);
    VbState &st = ctx->dvb;
    const DeviceTrace &tr = st.trace;
    NHP_CHECK(ctx, st.set, NHP_ERR_STATE, "%s: no VB state (call nhp_disc_vb_set)", fn);
    NHP_CHECK(ctx, dd->d_conv != nullptr, NHP_ERR_STATE, "%s: call nhp_disc_convolve first", fn);
    const int64_t N = st.n, B = st.b, NN = N * N, NB = N * B, T = dd->T;
    NHP_CHECK(ctx, dd->N == N && dd->B == B, NHP_ERR_INVALID, "%s: the VB state has N=%lld B=%lld, the data N=%lld B=%lld", fn, (long long)N,
              (long long)B, (long long)dd->N, (long long)dd->B);
    NHP_CHECK(ctx, tr.cap == 0 || (tr.shape.n == N && tr.shape.b == B), NHP_ERR_STATE, "%s: the open VB trace was begun for N=%lld B=%lld", fn,
              (long long)tr.shape.n, (long long)tr.shape.b);
    NHP_CHECK(ctx, tr.cap == 0 || tr.shape.a == st.network, NHP_ERR_STATE, "%s: the open VB trace was begun for a %s state", fn,
              tr.shape.a ? "network" : "standard");
    NHP_CHECK(ctx, t_begin >= 0 && t_begin < T && n_bins >= 1 && n_bins <= T, NHP_ERR_INVALID,
              "%s: window (t_begin=%lld, n_bins=%lld) outside 0 <= t_begin < T, 1 <= n_bins <= T (T=%lld)", fn, (long long)t_begin, (long long)n_bins, (long long)T);
    NHP_CHECK(ctx, step > 0.0 && step <= 1.0, NHP_ERR_INVALID, "%s: step=%g outside (0, 1]", fn, step);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    void *scratch;
    const bool net = st.network;
    const unsigned blocks = (unsigned)((NN + 255) / 256);
    // layout: e0[N] | ET[N*NB] | gammaT[N*NB] | alpha_sum[N] | events[N] | change (the last four zeroed together), and for a network
    // state | lrho | psum[blocks]
    const size_t extra = net ? 1 + (size_t)blocks : 0;
    NHP_TRY(nhp_scratch(ctx, (size_t)(3 * N + 2 * NB * N + 1 + extra) * sizeof(double), &scratch));
    double *d_e0 = (double *)scratch, *d_ET = d_e0 + N, *d_gT = d_ET + NB * N, *d_alpha = d_gT + NB * N, *d_events = d_alpha + N, *d_change = d_events + N;
    double *d_lrho = d_change + 1, *d_psum = d_lrho + 1;
    NHP_CUDA(ctx, cudaMemsetAsync(d_gT, 0, (size_t)(NB * N + 2 * N + 1) * sizeof(double), s));
    if (net)
        k_dvb_expect<true><<<blocks, 256, 0, s>>>(st.q, (int)N, (int)B, d_e0, d_ET, d_lrho);
    else
        k_dvb_expect<false><<<blocks, 256, 0, s>>>(st.q, (int)N, (int)B, d_e0, d_ET, nullptr);
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
    const double *h = st.hyper;
    const double betav = 1.0 / h[1] + (double)T * st.dt;  // baselines.jl:450 as written (1 / beta0, not beta0)
    const double scale = (double)T / (double)n_bins;
    if (net) {
        const double cprior = (h[2] * std::log(h[3]) - std::lgamma(h[2])) - (h[5] * std::log(h[6]) - std::lgamma(h[5]));
        k_dvb_update<true><<<blocks, 256, 0, s>>>(st.q, d_gT, d_alpha, events, d_lrho, (int)N, (int)B, h[0], betav, h[2], h[3], h[4], h[5], h[6],
                                                  cprior, scale, step, (unsigned long long *)d_change, d_psum);
        NHP_LAUNCHED(ctx);
        k_vbn_finish<<<1, 256, 0, s>>>(st.q + st.doubles - 2, d_psum, (int)blocks, h[7], h[8], (double)NN, step, (unsigned long long *)d_change);
        NHP_LAUNCHED(ctx);
    } else {
        k_dvb_update<false><<<blocks, 256, 0, s>>>(st.q, d_gT, d_alpha, events, nullptr, (int)N, (int)B, h[0], betav, h[2], h[3], h[4], 0.0, 0.0, 0.0,
                                                   scale, step, (unsigned long long *)d_change, nullptr);
        NHP_LAUNCHED(ctx);
    }
    NHP_CUDA(ctx, cudaGetLastError());
    NHP_TRY(nhp_vb_trace_push(ctx, st));  // the state of this step stays on the device
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
    nhp_trace_free(ctx, ctx->dvb.trace);
    return NHP_OK;
}

extern "C" int nhp_disc_vb_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    return nhp_vb_trace_begin(ctx, ctx->dvb, "nhp_disc_vb_trace_begin", "nhp_disc_vb_set", capacity);
}

extern "C" int nhp_disc_vb_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    return nhp_trace_count(ctx->dvb.trace, count, capacity);
}

extern "C" int nhp_disc_vb_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *q_out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    return nhp_vb_trace_read(ctx, ctx->dvb, "nhp_disc_vb_trace_read", first, count, q_out);
}
