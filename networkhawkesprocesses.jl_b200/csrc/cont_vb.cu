// cont_vb.cu -- mean-field VB of a continuous standard Hawkes process on the device (the reference has no `vb!` for continuous
// processes; this is the model of the Gibbs sweep, SURVEY section 10, with a factorised posterior).
//
// Priors (the hyper-parameters of nhp_cont_resample_params): lambda0_k ~ Gamma(alpha0, beta0), W[p,c] ~ Gamma(kappa, nu), Exponential
// theta ~ Gamma(alpha, beta), LogitNormal (mu, tau) ~ NormalGamma(mumu, kappamu, a0, b0); all rates.  The state q kept with the context
//   (ctx->cvb, a VbState: vb_state.cu holds its upload, read-back and trace):
//   q = [alphav(K); betav(K); kappav(K^2); nuv(K^2); atheta(K^2); btheta(K^2)]                      Exponential
//   q = [alphav(K); betav(K); kappav(K^2); nuv(K^2); mv(K^2); lambdav(K^2); av(K^2); bv(K^2)]        LogitNormal
// K^2 planes parent-major, X[p + K c].
//
// E-step.  Under q the responsibilities of the augmented likelihood are those of the parent sweep at *effective* parameters, because
// E_q[ln W + ln h(dt)] = ln W_eff + ln h(dt; theta_eff) for every lag dt:
//   lambda0_eff = exp(psi(alphav) - ln betav),  lW = psi(kappav) - ln nuv
//   Exponential:  theta_eff = atheta / btheta,  W_eff = exp(lW + psi(atheta) - ln btheta) / theta_eff      (E ln h = E ln theta - theta_eff dt)
//   LogitNormal:  mu_eff = mv, tau_eff = av / bv,  W_eff = exp(lW + (psi(av) - ln av) / 2 - 1 / (2 lambdav))
//                                                              (E[tau (y - mu)^2] = tau_eff (y - mv)^2 + 1 / lambdav)
// k_cvb_expect writes them into the context's parameters and nhp_cont_params_refresh rebuilds the tables (and the Exponential cut-off
// horizon) from them.  Sweep 1 (the ordinary intensity sweep) gives Z_i = lambda_i at those parameters; sweep 2 is the gradient's
// child-major scatter (cont_grad.cu, TERMS_VB) of u = W_eff h(dt) / Z_i: Mnm = sum u, S1 = sum u dt | sum u (y - mv), S2 = sum u (y - mv)^2
// (LogitNormal; y = logit(dt / dtmax)), and per child node sum 1 / Z_i, which times lambda0_eff is M0.  The LogitNormal sums are
// shifted about the current mv, so one sweep gives the centred second moment: S = S2 - S1^2 / Mnm.
//
// M-step (k_cvb_update, in place): alphav = alpha0 + M0, betav = beta0 + T, kappav = kappa + Mnm, nuv = nu + Mn[p],
//   Exponential  atheta = alpha + Mnm, btheta = beta + S1
//   LogitNormal  n = Mnm, d = S1 / n (0 for n = 0), ybar = mv + d, S = max(S2 - n d^2, 0):
//                lambdav = kappamu + n, mv = (kappamu mumu + n ybar) / lambdav, av = a0 + n / 2,
//                bv = b0 + S / 2 + kappamu n (ybar - mumu)^2 / (2 lambdav)
// (the textbook Normal-Gamma update; it keeps b0 where the Gibbs draw replaces it, quirk Q5).  A pair with n = 0 gets its prior.  The same
// kernel then writes the posterior means (alphav / betav, kappav / nuv, atheta / btheta | mv, av / bv) into the context's parameters,
// so a later log-likelihood, intensity or nhp_cont_params_get sees the fitted model.
//
// A network state (nhp_cont_vb_network_set) fits the Gamma mixture of the discrete network VB (disc_vb.cu): A[p,c] ~ Bernoulli(rho),
// rho ~ Beta(alpha_rho, beta_rho), W | A=1 ~ Gamma(kappa, nu) (the slab), W | A=0 ~ Gamma(kappa0, nu0) (the spike), with
//   q = [standard layout; kappa0v(K^2); nu0v(K^2); pv(K^2); alpharhov; betarhov],  pv[p + K c] = q(A[p,c] = 1).
// The E-step is the standard one with the mixture lW = pv (psi(kappav) - ln nuv) + (1 - pv) (psi(kappa0v) - ln nu0v): no link has a zero
// effective weight, so the sweeps run the process as a standard one (no adjacency mask, no cached pair structure).  The M-step is the
// standard one plus kappa0v = kappa0 + Mnm, nu0v = nu0 + Mn[p] and
//   logit pv = psi(alpharhov) - psi(betarhov) + [lgamma(kappav) - kappav ln nuv] - [lgamma(kappa0v) - kappa0v ln nu0v] + cprior
// (new kappav, nuv, kappa0v, nu0v; the old q(rho); cprior = [kappa ln nu - lgamma(kappa)] - [kappa0 ln nu0 - lgamma(kappa0)]), and
// k_vbn_finish (vb_network.cuh, shared with the discrete step) adds the per-block sums of pv in a fixed order into q(rho).  The context
// then holds the slab means kappav / nuv as W, A = [pv > 1/2] and rho = alpharhov / (alpharhov + betarhov).
#include "cont_sweep.cuh"
#include "vb_network.cuh"
#include <algorithm>
#include <cmath>

static size_t cvb_q_doubles(int kind, int64_t K) { return (size_t)(2 * K) + (size_t)(K * K) * (kind == NHP_LOGITNORMAL ? 6 : 4); }
// the network state: the standard layout, then kappa0v(K^2); nu0v(K^2); pv(K^2); alpharhov; betarhov
static size_t cvb_state_doubles(int kind, int64_t K, bool network) { return cvb_q_doubles(kind, K) + (network ? (size_t)(3 * K * K) + 2 : 0); }
// what the state's buffer holds behind q: the change slot, and for a network state lrho and the per-block sums of pv
static size_t cvb_alloc_doubles(int kind, int64_t K, bool network) {
    return cvb_state_doubles(kind, K, network) + 1 + (network ? 1 + (size_t)((K * K + 255) / 256) : 0);
}

// one thread per (p, c), e = p + K c (threads e < K also write lambda0_eff[e]): the effective parameters above; NET: lW is the mixture's
// and thread 0 writes lrho = psi(alpharhov) - psi(betarhov), the prior log-odds of a link
template <bool NET>
__global__ void __launch_bounds__(256) k_cvb_expect(const double *__restrict__ q, int K, int kind, double *__restrict__ lambda0, double *__restrict__ W,
                                                    double *__restrict__ p1, double *__restrict__ p2, double *__restrict__ lrho) {
    const int64_t KK = (int64_t)K * K;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= KK) return;
    const double *kv = q + 2 * K, *nv = kv + KK, *x1 = nv + KK, *x2 = x1 + KK;
    if (e < K) lambda0[e] = exp(nhp_digamma(q[e]) - log(q[K + e]));
    double lw = nhp_digamma(kv[e]) - log(nv[e]);
    if constexpr (NET) {
        const double *k0v = kv + KK * (kind == NHP_LOGITNORMAL ? 6 : 4), *n0v = k0v + KK, *pv = n0v + KK;
        if (e == 0) *lrho = nhp_digamma(pv[KK]) - nhp_digamma(pv[KK + 1]);
        const double p = pv[e];
        lw = p * lw + (1.0 - p) * (nhp_digamma(k0v[e]) - log(n0v[e]));
    }
    if (kind == NHP_EXPONENTIAL) {
        const double a = x1[e], b = x2[e], th = a / b;
        W[e] = exp(lw + (nhp_digamma(a) - log(b))) / th;
        p1[e] = th;
    } else {
        const double *x3 = x2 + KK, *x4 = x3 + KK;
        const double a = x3[e];
        W[e] = exp(lw + 0.5 * (nhp_digamma(a) - log(a)) - 0.5 / x2[e]);
        p1[e] = x1[e];
        p2[e] = a / x4[e];
    }
}

struct CvbArgs {
    int K, kind, update;      // update = 0: M0 and the posterior means of the unchanged q only (nhp_cont_vb_stats)
    double T;                 // duration of the data
    double h[8];              // the standard hyper-parameters of the state (ctx->cvb.hyper)
    double *q;
    double *M0;               // [K] in: sum of 1 / Z_i per node; out: M0 = lambda0_eff * that
    const double *Mn, *Mnm, *S1, *S2;
    double *lambda0, *W, *p1, *p2;  // in: the effective parameters (lambda0 read by threads e < K); out: the posterior means
    unsigned long long *change;     // max relative change (|new - old| for mv), as the bits of a non-negative double
    // network state only (behind the standard fields, which keep their offsets)
    double kappa0, nu0, cprior;     // the spike's hyper-parameters and the prior part of logit pv
    const double *lrho;             // psi(alpharhov) - psi(betarhov) of the old q(rho)
    double *A;                      // out: [pv > 1/2], the context's adjacency matrix
    double *psum;                   // out: [gridDim.x] sums of the new pv per block (fixed order)
};

// one thread per (p, c) (+ alphav, betav and M0 for e < K): the M-step above in place, then the posterior means; change and, NET, the
// block sums of pv by vb_block_reduce.  NET: also the spike, pv and A
template <bool NET>
__global__ void __launch_bounds__(256) k_cvb_update(const CvbArgs a) {
    const int K = a.K;
    const int64_t KK = (int64_t)K * K;
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double mx = 0.0;
    double pt = 0.0;  // NET: the new pv of this link
    if (e < KK) {
        double *q = a.q, *kv = q + 2 * K, *nv = kv + KK, *x1 = nv + KK, *x2 = x1 + KK, *x3 = x2 + KK, *x4 = x3 + KK;
        const bool ln = a.kind == NHP_LOGITNORMAL;
        if (e < K) {
            const double m0 = a.lambda0[e] * a.M0[e];
            a.M0[e] = m0;
            if (a.update) {
                const double an = a.h[0] + m0, bn = a.h[1] + a.T;
                mx = fmax(rel_change(an, q[e]), rel_change(bn, q[K + e]));
                q[e] = an;
                q[K + e] = bn;
            }
            a.lambda0[e] = q[e] / q[K + e];
        }
        if (a.update) {
            const double n = a.Mnm[e];
            const double kn = a.h[2] + n, nn = a.h[3] + a.Mn[e % K];
            mx = fmax(mx, fmax(rel_change(kn, kv[e]), rel_change(nn, nv[e])));
            kv[e] = kn;
            nv[e] = nn;
            if constexpr (NET) {
                double *k0v = kv + KK * (ln ? 6 : 4), *n0v = k0v + KK, *pv = n0v + KK;
                const double k0 = a.kappa0 + n, n0 = a.nu0 + a.Mn[e % K];
                const double pn = stable_sigmoid(*a.lrho + (lgamma(kn) - kn * log(nn)) - (lgamma(k0) - k0 * log(n0)) + a.cprior);
                mx = fmax(mx, fmax(rel_change(k0, k0v[e]), rel_change(n0, n0v[e])));
                mx = fmax(mx, fabs(pn - pv[e]));
                k0v[e] = k0; n0v[e] = n0; pv[e] = pn;
            }
            if (!ln) {
                const double an = a.h[4] + n, bn = a.h[5] + a.S1[e];
                mx = fmax(mx, fmax(rel_change(an, x1[e]), rel_change(bn, x2[e])));
                x1[e] = an;
                x2[e] = bn;
            } else {
                const double mumu = a.h[4], kmu = a.h[5];
                const double d = n > 0.0 ? a.S1[e] / n : 0.0;
                const double ybar = x1[e] + d, S = fmax(a.S2[e] - n * d * d, 0.0);
                const double lv = kmu + n, mv = (kmu * mumu + n * ybar) / lv, av = a.h[6] + 0.5 * n;
                const double dm = ybar - mumu;
                const double bv = a.h[7] + 0.5 * S + kmu * n * dm * dm / (2.0 * lv);
                mx = fmax(mx, fabs(mv - x1[e]));
                mx = fmax(mx, fmax(rel_change(lv, x2[e]), fmax(rel_change(av, x3[e]), rel_change(bv, x4[e]))));
                x1[e] = mv; x2[e] = lv; x3[e] = av; x4[e] = bv;
            }
        }
        a.W[e] = kv[e] / nv[e];
        if (!ln) a.p1[e] = x1[e] / x2[e];
        else { a.p1[e] = x1[e]; a.p2[e] = x3[e] / x4[e]; }
        if constexpr (NET) {
            pt = kv[KK * (ln ? 8 : 6) + e];  // pv
            a.A[e] = pt > 0.5 ? 1.0 : 0.0;
        }
    }
    vb_block_reduce<NET>(mx, pt, a.change, a.psum);
}

int nhp_cont_params_refresh(nhp_ctx *ctx);  // cont_conjugate.cu
int nhp_cont_fill_args(nhp_ctx *ctx, nhp_events *ev, int recursive, SweepArgs &a);            // cont_sweep.cu
int nhp_cont_run_event_intensity(nhp_ctx *ctx, nhp_events *ev, int recursive, double *d_out);  // cont_sweep.cu
int nhp_cont_child_scatter(nhp_ctx *ctx, nhp_events *ev, SweepArgs &a, const double *lam, int terms, double *g_l0, double *g_w, double *g_p1,
                           double *g_p2, int *grid_out);  // cont_grad.cu
constexpr int CVB_TERMS = 1;                              // TERMS_VB of cont_grad.cu

// the two set calls: every hyper-parameter positive and finite except mumu (finite); every entry of q positive and finite except mv
// (finite) and, for a network state, pv (in [0, 1]); refused before anything changes.  The buffer also holds the work slots behind q
static int cvb_set_state(nhp_ctx *ctx, const char *fn, bool network, const double *hyper, int n_hyper, const double *q) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "%s: continuous parameters not set (kind, K and dtmax come from nhp_cont_params_set)", fn);
    NHP_CHECK(ctx, hyper != nullptr && q != nullptr, NHP_ERR_INVALID, "%s: NULL argument", fn);
    const int kind = ctx->kind;
    const int64_t K = ctx->K, KK = K * K;
    const int nstd = kind == NHP_LOGITNORMAL ? 8 : 6, want = nstd + (network ? 4 : 0);
    NHP_CHECK(ctx, n_hyper == want, NHP_ERR_INVALID, "%s: expected %d hyper-parameters, got %d", fn, want, n_hyper);
    for (int i = 0; i < n_hyper; i++) {
        const bool mumu = kind == NHP_LOGITNORMAL && i == 4;  // the prior mean of mu may have any sign
        NHP_CHECK(ctx, std::isfinite(hyper[i]) && (mumu || hyper[i] > 0.0), NHP_ERR_INVALID, "%s: hyper-parameter %d must be %s", fn, i,
                  mumu ? "finite" : "positive and finite");
    }
    const size_t n = cvb_state_doubles(kind, K, network);
    const size_t mv_lo = (size_t)(2 * K + 2 * KK), mv_hi = kind == NHP_LOGITNORMAL ? mv_lo + (size_t)KK : mv_lo;
    const size_t p_lo = network ? cvb_q_doubles(kind, K) + (size_t)(2 * KK) : n, p_hi = network ? p_lo + (size_t)KK : n;
    VbState &st = ctx->cvb;
    NHP_TRY(nhp_vb_state_set(ctx, st, fn, q, n, cvb_alloc_doubles(kind, K, network), mv_lo, mv_hi, p_lo, p_hi, K, kind, network));
    for (int i = 0; i < 12; i++) st.hyper[i] = 0.0;  // [standard hyper-parameters, zero-padded to 8; kappa0, nu0, alpha_rho, beta_rho]
    for (int i = 0; i < nstd; i++) st.hyper[i] = hyper[i];
    for (int i = nstd; i < n_hyper; i++) st.hyper[8 + i - nstd] = hyper[i];
    return NHP_OK;
}

extern "C" int nhp_cont_vb_set(nhp_ctx *ctx, const double *hyper, int n_hyper, const double *q) {
    return cvb_set_state(ctx, "nhp_cont_vb_set", false, hyper, n_hyper, q);
}

extern "C" int nhp_cont_vb_network_set(nhp_ctx *ctx, const double *hyper, int n_hyper, const double *q) {
    return cvb_set_state(ctx, "nhp_cont_vb_network_set", true, hyper, n_hyper, q);
}

extern "C" int nhp_cont_vb_get(nhp_ctx *ctx, double *q) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    return nhp_vb_state_get(ctx, ctx->cvb, "nhp_cont_vb_get", "nhp_cont_vb_set", q);
}

// The E-step (and with `update` the M-step) on ev; every refusal comes before anything changes.  The statistics stay in the
// statistics buffers: M0, Mn, Mnm, S1 in phase 0, S2 in phase 1.  A network state runs the sweeps with has_A cleared (a standard
// process at the effective parameters), then sets it again with A = [pv > 1/2].
static int cvb_run(nhp_ctx *ctx, nhp_events *ev, const char *fn, bool update) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "%s: events handle is NULL", fn);
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "%s: continuous parameters not set (call nhp_cont_params_set)", fn);
    VbState &vb = ctx->cvb;
    const DeviceTrace &tr = vb.trace;
    const bool net = vb.set && vb.network;
    if (net)
        NHP_CHECK(ctx, ctx->has_A, NHP_ERR_STATE, "%s: the VB state is a network state but the parameters have no adjacency matrix", fn);
    else
        NHP_CHECK(ctx, !ctx->has_A, NHP_ERR_UNSUPPORTED, "%s runs a standard process (the parameters have an adjacency matrix)", fn);
    NHP_CHECK(ctx, ctx->bgrid_n == 0, NHP_ERR_UNSUPPORTED, "%s takes a homogeneous baseline (LogGaussianCox curves are set)", fn);
    NHP_CHECK(ctx, ev->n_halo == 0 && ev->index_base == 0, NHP_ERR_UNSUPPORTED, "%s works on unsharded events", fn);
    NHP_CHECK(ctx, !(ctx->comm && ctx->nranks > 1), NHP_ERR_UNSUPPORTED, "%s runs on one GPU (the context has a communicator of %d ranks)", fn, ctx->nranks);
    NHP_CHECK(ctx, vb.set, NHP_ERR_STATE, "%s: no VB state (call nhp_cont_vb_set)", fn);
    NHP_CHECK(ctx, vb.b == ctx->kind && vb.n == ctx->K, NHP_ERR_STATE,
              "%s: the VB state was set for kind %d, K=%lld; the parameters now have kind %d, K=%lld", fn, (int)vb.b, (long long)vb.n, ctx->kind,
              (long long)ctx->K);
    NHP_CHECK(ctx, ev->K == ctx->K, NHP_ERR_INVALID, "%s: events were uploaded with K=%lld but the VB state has K=%lld", fn, (long long)ev->K, (long long)ctx->K);
    NHP_CHECK(ctx, !update || tr.cap == 0 || (tr.shape.n == ctx->K && tr.shape.b == ctx->kind), NHP_ERR_STATE,
              "%s: the open VB trace was begun for kind %d, K=%lld", fn, (int)tr.shape.b, (long long)tr.shape.n);
    NHP_CHECK(ctx, !update || tr.cap == 0 || tr.shape.a == net, NHP_ERR_STATE, "%s: the open VB trace was begun for a %s state",
              fn, tr.shape.a ? "network" : "standard");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t K = ctx->K, KK = K * K, own = ev->n;
    const size_t nq = vb.doubles;
    const StatsLayout sl{K};
    const unsigned blocks = (unsigned)((KK + 255) / 256);
    cudaStream_t s = ctx->stream;
    double *d_change = vb.q + nq, *d_lrho = d_change + 1, *d_psum = d_lrho + 1;  // d_lrho, d_psum: network state only
    // effective parameters -> the context's parameters and tables
    if (net) {
        k_cvb_expect<true><<<blocks, 256, 0, s>>>(vb.q, (int)K, ctx->kind, ctx->d_lambda0, ctx->d_W, ctx->d_p1, ctx->d_p2, d_lrho);
        ctx->has_A = false;  // the E-step is that of a standard process: no mask, no pair structure (d_A keeps its values until the M-step)
    } else {
        k_cvb_expect<false><<<blocks, 256, 0, s>>>(vb.q, (int)K, ctx->kind, ctx->d_lambda0, ctx->d_W, ctx->d_p1, ctx->d_p2, nullptr);
    }
    NHP_LAUNCHED(ctx);
    struct RestoreA {  // a network process again on every way out of this call
        nhp_ctx *c; bool on;
        ~RestoreA() { if (on) c->has_A = true; }
    } restore{ctx, net};
    NHP_CUDA(ctx, cudaGetLastError());
    ctx->cont_set = false;
    ctx->parents_valid = false;
    ctx->sweep_ll_valid = false;
    ctx->grad_valid = false;
    NHP_TRY(nhp_cont_params_refresh(ctx));
    ctx->cont_set = true;
    double *st = ctx->d_stats0;
    NHP_CUDA(ctx, cudaMemsetAsync(st, 0, (size_t)sl.total() * sizeof(double), s));
    NHP_CUDA(ctx, cudaMemcpyAsync(st + sl.off_Mn(), ev->d_Mn, (size_t)K * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats1, 0, (size_t)KK * sizeof(double), s));
    NHP_CUDA(ctx, cudaMemsetAsync(d_change, 0, sizeof(double), s));
    if (own > 0) {
        SweepArgs a;
        NHP_TRY(nhp_cont_fill_args(ctx, ev, 0, a));
        void *scratch;  // sweep 1: Z_i (nothing else uses the scratch area until the call returns)
        NHP_TRY(nhp_scratch(ctx, (size_t)own * sizeof(double), &scratch));
        NHP_TRY(nhp_cont_run_event_intensity(ctx, ev, 0, (double *)scratch));
        int grid = 0;   // sweep 2: the expected statistics
        NHP_TRY(nhp_cont_child_scatter(ctx, ev, a, (const double *)scratch, CVB_TERMS, st + sl.off_M0(), st + sl.off_Mnm(), st + sl.off_S1(), ctx->d_stats1, &grid));
    }
    CvbArgs ca;
    ca.K = (int)K; ca.kind = ctx->kind; ca.update = update ? 1 : 0; ca.T = ev->duration;
    for (int i = 0; i < 8; i++) ca.h[i] = vb.hyper[i];
    ca.q = vb.q; ca.M0 = st + sl.off_M0(); ca.Mn = st + sl.off_Mn(); ca.Mnm = st + sl.off_Mnm(); ca.S1 = st + sl.off_S1(); ca.S2 = ctx->d_stats1;
    ca.lambda0 = ctx->d_lambda0; ca.W = ctx->d_W; ca.p1 = ctx->d_p1; ca.p2 = ctx->d_p2; ca.change = (unsigned long long *)d_change;
    double rho_q[2] = {0.0, 0.0};  // network state: q(rho) after the step
    if (net) {
        const double *hn = vb.hyper + 8, kappa = vb.hyper[2], nu = vb.hyper[3];
        ca.kappa0 = hn[0]; ca.nu0 = hn[1];
        ca.cprior = (kappa * std::log(nu) - std::lgamma(kappa)) - (hn[0] * std::log(hn[1]) - std::lgamma(hn[0]));
        ca.lrho = d_lrho; ca.A = ctx->d_A; ca.psum = d_psum;
        k_cvb_update<true><<<blocks, 256, 0, s>>>(ca);
        NHP_LAUNCHED(ctx);
        if (update) {
            k_vbn_finish<<<1, 256, 0, s>>>(vb.q + nq - 2, d_psum, (int)blocks, hn[2], hn[3], (double)KK, 1.0, (unsigned long long *)d_change);
            NHP_LAUNCHED(ctx);
        }
        NHP_CUDA(ctx, cudaMemcpyAsync(rho_q, vb.q + nq - 2, sizeof(rho_q), cudaMemcpyDeviceToHost, s));  // read after the refresh's synchronisation
    } else {
        ca.kappa0 = ca.nu0 = ca.cprior = 0.0; ca.lrho = nullptr; ca.A = nullptr; ca.psum = nullptr;
        k_cvb_update<false><<<blocks, 256, 0, s>>>(ca);
        NHP_LAUNCHED(ctx);
    }
    NHP_CUDA(ctx, cudaGetLastError());
    // the posterior means are the context's parameters from here on (a network state: with A = [pv > 1/2])
    if (net) ctx->has_A = true;
    ctx->cont_set = false;
    NHP_TRY(nhp_cont_params_refresh(ctx));
    ctx->cont_set = true;
    if (net) ctx->rho = rho_q[0] / (rho_q[0] + rho_q[1]);
    if (update) NHP_TRY(nhp_vb_trace_push(ctx, vb));  // the state of this step stays on the device
    return NHP_OK;
}

extern "C" int nhp_cont_vb_stats(nhp_ctx *ctx, nhp_events *ev, double *M0, double *Mnm, double *S1, double *S2) {
    NHP_TRY(cvb_run(ctx, ev, "nhp_cont_vb_stats", false));
    const int64_t K = ctx->K, KK = K * K;
    const StatsLayout sl{K};
    cudaStream_t s = ctx->stream;
    if (M0) NHP_CUDA(ctx, cudaMemcpyAsync(M0, ctx->d_stats0 + sl.off_M0(), (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (Mnm) NHP_CUDA(ctx, cudaMemcpyAsync(Mnm, ctx->d_stats0 + sl.off_Mnm(), (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (S1) NHP_CUDA(ctx, cudaMemcpyAsync(S1, ctx->d_stats0 + sl.off_S1(), (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (S2) NHP_CUDA(ctx, cudaMemcpyAsync(S2, ctx->d_stats1, (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

extern "C" int nhp_cont_vb_step(nhp_ctx *ctx, nhp_events *ev, double *change) {
    NHP_TRY(nhp_timer_begin(ctx));
    NHP_TRY(cvb_run(ctx, ev, "nhp_cont_vb_step", true));
    if (change)
        NHP_CUDA(ctx, cudaMemcpyAsync(change, ctx->cvb.q + ctx->cvb.doubles, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_TRY(nhp_timer_end(ctx));
    return NHP_OK;
}

extern "C" int nhp_cont_vb_trace_free(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    nhp_trace_free(ctx, ctx->cvb.trace);
    return NHP_OK;
}

extern "C" int nhp_cont_vb_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    return nhp_vb_trace_begin(ctx, ctx->cvb, "nhp_cont_vb_trace_begin", "nhp_cont_vb_set", capacity);
}

extern "C" int nhp_cont_vb_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    return nhp_trace_count(ctx->cvb.trace, count, capacity);
}

extern "C" int nhp_cont_vb_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *q_out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    return nhp_vb_trace_read(ctx, ctx->cvb, "nhp_cont_vb_trace_read", first, count, q_out);
}
