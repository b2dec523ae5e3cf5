// cont_conjugate.cu -- the conjugate parameter draws of one Gibbs sweep on the device, so that `resample!`
// (continuous.jl:202-208 / 350-358) can stay on the GPU between sweeps: the K^2 sufficient statistics never travel to
// the host and the parameter tables are rebuilt in place.  SURVEY.md section 8f ("next": device-side conjugate draws).
//   baseline  lambda0[k] ~ Gamma(alpha0 + M0[k], 1/(beta0 + T))                                     baselines.jl:72-77
//   weights   W[p,c]     ~ Gamma(kappa + Mnm[p,c], 1/(nu + Mn[p]))  (also where A == 0, quirk Q14)   weights.jl:59-64
//   Exponential   theta  ~ Gamma(alpha + Mnm, 1/(beta + Mnm Xnm)),  Mnm Xnm = S1                      impulses.jl:68-73
//   LogitNormal   tau    ~ Gamma(alpha0 + Mnm/2, 1/b),  b = S2/2 + Mnm kmu/(Mnm + kmu) (Xnm - mumu)^2/2, NaN -> beta0 (Q5)
//                 mu     ~ Normal((kmu mumu + Mnm Xnm)/(kmu + Mnm) [NaN -> mumu], 1/sqrt((kmu + Mnm) tau))   impulses.jl:204-214
// Random numbers: Philox4x32-10 with key seed ^ "CONJUGAT", counter words (element, draw block | parameter id, sweep
// counter): every rank of a multi-GPU job that holds the same (all-reduced) statistics draws the same parameters.
// Gamma: Marsaglia & Tsang (2000) with the shape < 1 boost; Normal: Box-Muller.  Parity with the reference is
// distributional (Julia's own samplers are not reproducible from uniforms): tests check the moments.
#include "nhp_internal.cuh"
#include <algorithm>
#include <cmath>
#include <vector>

struct PhiloxStream {
    uint32_t k0, k1, c0, c1, c2, c3;
    uint32_t buf[4];
    int have;
    __device__ PhiloxStream(uint64_t seed, uint32_t element, uint32_t param, uint64_t counter) {
        const uint64_t key = seed ^ 0x434F4E4A55474154ull;
        k0 = (uint32_t)key; k1 = (uint32_t)(key >> 32);
        c0 = element; c1 = param << 24; c2 = (uint32_t)counter; c3 = (uint32_t)(counter >> 32);
        have = 0;
    }
    __device__ double uniform() {  // (0, 1): 53 bits, never exactly 0
        if (have == 0) { philox4x32_10(c0, c1, c2, c3, k0, k1, buf); c1++; have = 2; }
        have--;
        const uint64_t x = (((uint64_t)buf[2 * have] << 32) | (uint64_t)buf[2 * have + 1]) >> 11;
        return ((double)x + 0.5) * 1.1102230246251565e-16;
    }
    __device__ double normal() {
        const double u1 = uniform(), u2 = uniform();
        return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    }
    __device__ double gamma(double shape, double scale) {
        if (!(shape > 0.0) || !(scale > 0.0)) return nan("");
        double boost = 1.0;
        if (shape < 1.0) { boost = pow(uniform(), 1.0 / shape); shape += 1.0; }
        const double d = shape - 1.0 / 3.0, c = 1.0 / sqrt(9.0 * d);
        for (int it = 0; it < 1000; it++) {
            const double x = normal();
            double v = 1.0 + c * x;
            if (v <= 0.0) continue;
            v = v * v * v;
            const double u = uniform();
            const double x2 = x * x;
            if (u < 1.0 - 0.0331 * x2 * x2 || log(u) < 0.5 * x2 + d * (1.0 - v + log(v))) return fmax(d * v * boost * scale, 1e-300);
        }
        return fmax(d * boost * scale, 1e-300);  // unreachable in practice (acceptance > 95 % per trial)
    }
};

struct ConjArgs {
    int K, kind;
    uint64_t seed, counter;
    double T;
    double a0l, b0l, kappa, nu;       // baseline, weights
    double h0, h1, h2, h3;            // EX: alpha, beta;  LN: mumu, kappamu, alpha0, beta0
    const double *M0, *Mn, *Mnm, *S1, *S2;
    double *lambda0, *W, *p1, *p2;
};

__global__ void k_conjugate(const ConjArgs a) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t KK = (int64_t)a.K * a.K;
    if (e < a.K) {
        PhiloxStream r(a.seed, (uint32_t)e, 0u, a.counter);
        a.lambda0[e] = r.gamma(a.a0l + a.M0[e], 1.0 / (a.b0l + a.T));
    }
    if (e >= KK) return;
    const int p = (int)(e % a.K);
    const double m = a.Mnm[e];
    {
        PhiloxStream r(a.seed, (uint32_t)e, 1u, a.counter);
        a.W[e] = r.gamma(a.kappa + m, 1.0 / (a.nu + a.Mn[p]));
    }
    PhiloxStream r(a.seed, (uint32_t)e, 2u, a.counter);
    if (a.kind == NHP_EXPONENTIAL) {
        a.p1[e] = r.gamma(a.h0 + m, 1.0 / (a.h1 + a.S1[e]));  // Mnm * Xnm = S1 (0 where Mnm == 0)
    } else {
        const double mumu = a.h0, kmu = a.h1, alpha0 = a.h2, beta0 = a.h3;
        const double X = a.S1[e] / m;  // NaN where Mnm == 0, as in the reference
        double b = 0.5 * a.S2[e] + m * kmu / (m + kmu) * (X - mumu) * (X - mumu) * 0.5;
        if (isnan(b)) b = beta0;
        const double tau = r.gamma(alpha0 + 0.5 * m, 1.0 / b);
        double mun = (kmu * mumu + m * X) / (kmu + m);
        if (isnan(mun)) mun = mumu;
        a.p2[e] = tau;
        a.p1[e] = mun + r.normal() / sqrt((kmu + m) * tau);
    }
}

// scalars the host keeps about the parameters: [lambda0 min, lambda0 sum, theta min, max |w theta|, #non-zero effective weights,
// theta min and max |W theta| over all entries with W != 0 (adjacency sampler), sum of A]; one partial row of 8 per block
constexpr int PS_BLOCKS = 128;
__global__ void __launch_bounds__(256) k_param_scan(int K, int kind, const double *__restrict__ lambda0, const double *__restrict__ W, const double *__restrict__ A,
                                                    const double *__restrict__ p1, double *__restrict__ part) {
    __shared__ double s_v[8][256];
    double l0min = INFINITY, l0sum = 0.0, tmin = INFINITY, wmax = 0.0, nnz = 0.0, tmin_all = INFINITY, wmax_all = 0.0, asum = 0.0;
    const int64_t KK = (int64_t)K * K;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < KK; e += (int64_t)gridDim.x * blockDim.x) {
        if (e < K) { l0min = fmin(l0min, lambda0[e]); l0sum += lambda0[e]; }
        const double w0 = W[e], a = A ? A[e] : 1.0;
        const double w = a * w0;
        asum += a;
        if (w != 0.0) {
            nnz += 1.0;
            if (kind == NHP_EXPONENTIAL) { tmin = fmin(tmin, p1[e]); wmax = fmax(wmax, fabs(w * p1[e])); }
        }
        if (kind == NHP_EXPONENTIAL && w0 != 0.0) { tmin_all = fmin(tmin_all, p1[e]); wmax_all = fmax(wmax_all, fabs(w0 * p1[e])); }
    }
    const int t = threadIdx.x;
    s_v[0][t] = l0min; s_v[1][t] = l0sum; s_v[2][t] = tmin; s_v[3][t] = wmax; s_v[4][t] = nnz; s_v[5][t] = tmin_all; s_v[6][t] = wmax_all; s_v[7][t] = asum;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if (t < s) {
            s_v[0][t] = fmin(s_v[0][t], s_v[0][t + s]); s_v[1][t] += s_v[1][t + s];
            s_v[2][t] = fmin(s_v[2][t], s_v[2][t + s]); s_v[3][t] = fmax(s_v[3][t], s_v[3][t + s]);
            s_v[4][t] += s_v[4][t + s];
            s_v[5][t] = fmin(s_v[5][t], s_v[5][t + s]); s_v[6][t] = fmax(s_v[6][t], s_v[6][t + s]);
            s_v[7][t] += s_v[7][t + s];
        }
        __syncthreads();
    }
    if (t < 8) part[(size_t)blockIdx.x * 8 + t] = s_v[t][0];
}
__global__ void k_param_scan_final(const double *__restrict__ part, int nb, double *__restrict__ out) {
    const int t = threadIdx.x;  // 8 threads, one per scalar; fixed order => deterministic
    if (t >= 8) return;
    const bool is_min = t == 0 || t == 2 || t == 5, is_max = t == 3 || t == 6;
    double v = is_min ? INFINITY : 0.0;
    for (int b = 0; b < nb; b++) {
        const double x = part[(size_t)b * 8 + t];
        v = is_min ? fmin(v, x) : (is_max ? fmax(v, x) : v + x);
    }
    out[t] = v;
}

int nhp_cont_derive_tables(nhp_ctx *ctx);  // nhp_context.cu: masked tables, bit rows, row sums from the device-resident raw parameters

// refresh the host-side scalars from the device-resident parameters and rebuild the derived tables
int nhp_cont_params_refresh(nhp_ctx *ctx) {
    cudaStream_t s = ctx->stream;
    const int64_t K = ctx->K;
    double *scratch;
    NHP_TRY(nhp_partials(ctx, 8 * (PS_BLOCKS + 1), &scratch));
    const int nb = (int)std::min<int64_t>(PS_BLOCKS, (K * K + 255) / 256);
    k_param_scan<<<nb, 256, 0, s>>>((int)K, ctx->kind, ctx->d_lambda0, ctx->d_W, ctx->has_A ? ctx->d_A : nullptr, ctx->d_p1, scratch + 8);
    NHP_LAUNCHED(ctx);
    k_param_scan_final<<<1, 32, 0, s>>>(scratch + 8, nb, scratch);
    NHP_LAUNCHED(ctx);
    double h[8];
    NHP_CUDA(ctx, cudaMemcpyAsync(h, scratch, sizeof(h), cudaMemcpyDeviceToHost, s));
    NHP_TRY(nhp_cont_derive_tables(ctx));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->lambda0_min = ctx->bgrid_n > 0 ? ctx->bgrid_min : h[0];  // curves on the device: the cut-off horizon keeps their minimum
    ctx->lambda0_sum = h[1]; ctx->theta_min = h[2]; ctx->wt_max = h[3];
    ctx->density = h[4] / (double)(K * K);
    ctx->theta_min_all = h[5]; ctx->wt_max_all = h[6];
    ctx->a_sum = ctx->has_A ? h[7] : (double)(K * K);
    return NHP_OK;
}

extern "C" int nhp_cont_resample_params(nhp_ctx *ctx, nhp_events *ev, uint64_t seed, uint64_t counter, double duration, const double *hyper, int n_hyper,
                                        int flags) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set (call nhp_cont_params_set)");
    NHP_CHECK(ctx, ctx->parents_valid, NHP_ERR_STATE, "nhp_cont_resample_params: no parent assignment (call nhp_cont_resample_parents first)");
    const int need = ctx->kind == NHP_LOGITNORMAL ? 8 : 6;
    NHP_CHECK(ctx, hyper != nullptr && n_hyper == need, NHP_ERR_INVALID, "nhp_cont_resample_params: expected %d hyper-parameters, got %d", need, n_hyper);
    for (int i = 0; i < n_hyper; i++) NHP_CHECK(ctx, std::isfinite(hyper[i]), NHP_ERR_INVALID, "nhp_cont_resample_params: hyper-parameter %d is not finite", i);
    NHP_CHECK(ctx, duration > 0.0, NHP_ERR_INVALID, "nhp_cont_resample_params: duration must be positive");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (flags & 1) {
        NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "nhp_cont_resample_params: events handle is NULL");
        NHP_TRY(nhp_cont_suffstats_second_pass(ctx, ev));
    }
    const int64_t K = ctx->K, KK = K * K;
    const StatsLayout sl{K};
    ConjArgs a;
    a.K = (int)K; a.kind = ctx->kind; a.seed = seed; a.counter = counter; a.T = duration;
    a.a0l = hyper[0]; a.b0l = hyper[1]; a.kappa = hyper[2]; a.nu = hyper[3];
    a.h0 = hyper[4]; a.h1 = hyper[5]; a.h2 = need == 8 ? hyper[6] : 0.0; a.h3 = need == 8 ? hyper[7] : 0.0;
    a.M0 = ctx->d_stats0 + sl.off_M0(); a.Mn = ctx->d_stats0 + sl.off_Mn(); a.Mnm = ctx->d_stats0 + sl.off_Mnm(); a.S1 = ctx->d_stats0 + sl.off_S1();
    a.S2 = ctx->d_stats1;
    a.lambda0 = ctx->d_lambda0; a.W = ctx->d_W; a.p1 = ctx->d_p1; a.p2 = ctx->d_p2;
    NHP_TRY(nhp_timer_begin(ctx));
    k_conjugate<<<(unsigned)((KK + 127) / 128), 128, 0, ctx->stream>>>(a);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    ctx->cont_set = false;
    ctx->sweep_ll_valid = false;
    NHP_TRY(nhp_cont_params_refresh(ctx));
    NHP_TRY(nhp_timer_end(ctx));
    ctx->cont_set = true;
    return NHP_OK;
}

extern "C" int nhp_cont_params_get(nhp_ctx *ctx, double *lambda0, double *W, double *A, double *p1, double *p2) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t K = ctx->K, KK = K * K;
    cudaStream_t s = ctx->stream;
    if (lambda0) NHP_CUDA(ctx, cudaMemcpyAsync(lambda0, ctx->d_lambda0, (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (W) NHP_CUDA(ctx, cudaMemcpyAsync(W, ctx->d_W, (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (A) {
        NHP_CHECK(ctx, ctx->has_A, NHP_ERR_STATE, "nhp_cont_params_get: the process has no adjacency matrix");
        NHP_CUDA(ctx, cudaMemcpyAsync(A, ctx->d_A, (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    if (p1) NHP_CUDA(ctx, cudaMemcpyAsync(p1, ctx->d_p1, (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (p2) {
        NHP_CHECK(ctx, ctx->kind == NHP_LOGITNORMAL, NHP_ERR_STATE, "nhp_cont_params_get: the Exponential impulse has no second parameter");
        NHP_CUDA(ctx, cudaMemcpyAsync(p2, ctx->d_p2, (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    }
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// rho ~ Beta(alpha + sum(A), beta + K^2 - sum(A))  (networks.jl:72-78) as a ratio of two Gamma draws, on the device so that every
// rank of a multi-GPU chain draws the same value from the same (seed, counter); out[0] = rho.  Stream ids: 3 continuous, 11 discrete.
__global__ void k_network_draw(uint64_t seed, uint64_t counter, uint32_t param, double a, double b, double *out) {
    if (threadIdx.x != 0 || blockIdx.x != 0) return;
    PhiloxStream r(seed, 0u, param, counter);
    const double x = r.gamma(a, 1.0), y = r.gamma(b, 1.0);
    out[0] = x / (x + y);
}

extern "C" int nhp_cont_resample_network(nhp_ctx *ctx, uint64_t seed, uint64_t counter, double alpha, double beta, double *rho_out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set && ctx->has_A, NHP_ERR_STATE, "nhp_cont_resample_network: no network process parameters on the device");
    NHP_CHECK(ctx, alpha > 0.0 && beta > 0.0, NHP_ERR_INVALID, "nhp_cont_resample_network: alpha and beta must be positive");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    double *scratch;
    NHP_TRY(nhp_partials(ctx, 8, &scratch));
    const double KK = (double)ctx->K * (double)ctx->K;
    k_network_draw<<<1, 32, 0, ctx->stream>>>(seed, counter, 3u, alpha + ctx->a_sum, beta + KK - ctx->a_sum, scratch);
    NHP_LAUNCHED(ctx);
    double rho = 0.0;
    NHP_CUDA(ctx, cudaMemcpyAsync(&rho, scratch, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->rho = rho;
    if (rho_out) *rho_out = rho;
    return NHP_OK;
}

extern "C" int nhp_cont_network_get(const nhp_ctx *ctx, double *rho) {
    if (!ctx || !rho) return NHP_ERR_INVALID;
    *rho = ctx->rho;
    return NHP_OK;
}

extern "C" int nhp_cont_network_set(nhp_ctx *ctx, double rho) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, rho >= 0.0 && rho <= 1.0, NHP_ERR_INVALID, "BernoulliNetworkModel: link probability must be in [0, 1]");
    ctx->rho = rho;
    return NHP_OK;
}

// ---- development hooks (include/nhp_devel.h): device-side snapshot of the parameters
extern "C" int nhp_cont_params_save(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t K = (size_t)ctx->K, KK = K * K;
    if (!ctx->d_save) NHP_CUDA(ctx, cudaMalloc(&ctx->d_save, (K + 4 * KK) * sizeof(double)));
    cudaStream_t s = ctx->stream;
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_save, ctx->d_lambda0, K * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_save + K, ctx->d_W, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_save + K + KK, ctx->d_A, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_save + K + 2 * KK, ctx->d_p1, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_save + K + 3 * KK, ctx->d_p2, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}
extern "C" int nhp_cont_params_restore(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set && ctx->d_save, NHP_ERR_STATE, "nhp_cont_params_restore: nothing saved");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t K = (size_t)ctx->K, KK = K * K;
    cudaStream_t s = ctx->stream;
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_lambda0, ctx->d_save, K * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_W, ctx->d_save + K, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_A, ctx->d_save + K + KK, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_p1, ctx->d_save + K + 2 * KK, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_p2, ctx->d_save + K + 3 * KK, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    ctx->cont_set = false;
    ctx->sweep_ll_valid = false;
    NHP_TRY(nhp_cont_params_refresh(ctx));
    ctx->cont_set = true;
    return NHP_OK;
}


// ---------------------------------------------------------------------------------------
// discrete Gibbs sweep (discrete.jl:361-367 / 416-424): conjugate draws from the counts of the last parent sweep
//   baseline  lambda0[c] ~ Gamma(alpha0 + counts[c, 0], 1 / (beta0 + T dt))          intended form of baselines.jl:413-419 (quirk Q2)
//   weights   W[p,c]     ~ Gamma(kappa + sum_b counts[c, p, b], 1 / (nu + Mn[p]))     weights.jl:59-64
//   impulses  theta[p,c,:] ~ Dirichlet(gamma + counts[c, p, :])                        impulses.jl:337-353 (normalised Gammas)
// ---------------------------------------------------------------------------------------
struct DiscConjArgs {
    int N, B;
    uint64_t seed, counter;
    double Tdt, alpha0, beta0, kappa, nu, gamma;
    const double *counts, *Mn;
    double *lambda0, *W, *theta;
};
__global__ void k_disc_conjugate(const DiscConjArgs a) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t NN = (int64_t)a.N * a.N;
    if (e < a.N) {
        PhiloxStream r(a.seed, (uint32_t)e, 8u, a.counter);
        a.lambda0[e] = r.gamma(a.alpha0 + a.counts[e], 1.0 / (a.beta0 + a.Tdt));
    }
    if (e >= NN) return;
    const int p = (int)(e % a.N), c = (int)(e / a.N);  // e = p + N c as in W
    double m = 0.0;
    for (int b = 0; b < a.B; b++) m += a.counts[c + (int64_t)a.N * (1 + p * a.B + b)];
    {
        PhiloxStream r(a.seed, (uint32_t)e, 9u, a.counter);
        a.W[e] = r.gamma(a.kappa + m, 1.0 / (a.nu + a.Mn[p]));
    }
    PhiloxStream r(a.seed, (uint32_t)e, 10u, a.counter);
    double tot = 0.0;
    for (int b = 0; b < a.B; b++) {
        const double g = r.gamma(a.gamma + a.counts[c + (int64_t)a.N * (1 + p * a.B + b)], 1.0);
        a.theta[e + NN * b] = g;  // theta[p + N (c + N b)]
        tot += g;
    }
    for (int b = 0; b < a.B; b++) a.theta[e + NN * b] /= tot;
}

// the draws in place on the context's parameters; d_Mn: events per node on the device.  The derived tables are not refreshed here.
int nhp_disc_draw_params(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *d_Mn, const double *hyper) {
    const int64_t N = ctx->dN, NN = N * N;
    DiscConjArgs a;
    a.N = (int)N; a.B = (int)ctx->dB; a.seed = seed; a.counter = counter; a.Tdt = (double)(dd->T - dd->t_halo) * ctx->ddt;
    a.alpha0 = hyper[0]; a.beta0 = hyper[1]; a.kappa = hyper[2]; a.nu = hyper[3]; a.gamma = hyper[4];
    a.counts = ctx->dd_counts; a.Mn = d_Mn; a.lambda0 = ctx->dd_lambda0; a.W = ctx->dd_W; a.theta = ctx->dd_theta;
    k_disc_conjugate<<<(unsigned)((NN + 127) / 128), 128, 0, ctx->stream>>>(a);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

extern "C" int nhp_disc_resample_params(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *Mn, const double *hyper, int n_hyper,
                                        double *lambda0, double *W, double *theta) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr && ctx->disc_set, NHP_ERR_STATE, "nhp_disc_resample_params: discrete parameters not set");
    const int64_t N = ctx->dN, B = ctx->dB, NN = N * N;
    NHP_CHECK(ctx, dd->N == N, NHP_ERR_INVALID, "nhp_disc_resample_params: the data has %lld nodes, the parameters %lld", (long long)dd->N, (long long)N);
    NHP_CHECK(ctx, ctx->dd_counts && ctx->dd_counts_N == N && ctx->dd_counts_B == B, NHP_ERR_STATE,
              "nhp_disc_resample_params: no counts of a parent sweep with these parameters on the device (call nhp_disc_gibbs_counts first)");
    NHP_CHECK(ctx, Mn && hyper && n_hyper == 5 && lambda0 && W && theta, NHP_ERR_INVALID, "nhp_disc_resample_params: need Mn[N], 5 hyper-parameters and the three outputs");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    void *scratch = nullptr;
    NHP_TRY(nhp_scratch(ctx, (size_t)N * sizeof(double), &scratch));
    NHP_CUDA(ctx, cudaMemcpyAsync(scratch, Mn, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_TRY(nhp_timer_begin(ctx));
    NHP_TRY(nhp_disc_draw_params(ctx, dd, seed, counter, (const double *)scratch, hyper));
    NHP_TRY(nhp_timer_end(ctx));
    // the derived tables (bump, sparse parent lists) follow the new parameters on the device; the parameters go to the host (they are the sample)
    const double ms = ctx->last_ms;
    NHP_TRY(nhp_disc_tables_refresh(ctx));
    ctx->last_ms = ms;
    NHP_CUDA(ctx, cudaMemcpyAsync(lambda0, ctx->dd_lambda0, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(W, ctx->dd_W, (size_t)NN * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(theta, ctx->dd_theta, (size_t)(NN * B) * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// rho of the discrete Bernoulli network from the sum of A left by the last table refresh; the value stays with the context
int nhp_disc_draw_network(nhp_ctx *ctx, uint64_t seed, uint64_t counter, double alpha, double beta) {
    double *scratch;
    NHP_TRY(nhp_partials(ctx, 8, &scratch));
    const double NN = (double)ctx->dN * (double)ctx->dN;
    k_network_draw<<<1, 32, 0, ctx->stream>>>(seed, counter, 11u, alpha + ctx->dd_a_sum, beta + NN - ctx->dd_a_sum, scratch);
    NHP_LAUNCHED(ctx);
    double rho = 0.0;
    NHP_CUDA(ctx, cudaMemcpyAsync(&rho, scratch, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->dd_rho = rho;
    return NHP_OK;
}
