// cont_grad.cu -- analytic gradient of the continuous log-likelihood (extension for `mle!`, continuous.jl:144-198:
// the reference hands Optim a gradient-free objective, i.e. ~2P log-likelihood sweeps per finite-difference gradient;
// this file produces the same gradient from two sweeps).
//
//   ll = sum_i log lambda_i - [first shard] T sum_k lambda0_k - sum_p Mn[p] rowsum[p]           (continuous.jl:217-238)
//   lambda_i = lambda0[c_i] + sum_{j in window(i)} a[p,c] W[p,c] h_pc(dt),  p = c_j, c = c_i, dt = t_i - t_j
//
//   d ll / d lambda0[k] = sum_{i: c_i = k} 1/lambda_i - [first shard] T
//   d ll / d W[p,c]     = sum_pairs a h_pc(dt) / lambda_i - Mn[p] d rowsum[p] / d W[p,c]
//   Exponential  h = theta e^{-theta dt}:       d/d theta = sum a W e^{-theta dt} (1 - theta dt) / lambda_i
//   LogitNormal  h = pdf(LogitNormal(mu, tau^-1/2), dt/D), z = logit(dt/D):
//                d/d mu = sum v tau (z - mu) / lambda_i,   d/d tau = sum v (1/(2 tau) - (z - mu)^2 / 2) / lambda_i,   v = a W h
//   d rowsum[p] / d W[p,c] = a[p,c]  (1 under quirk Q3: recursive Exponential network, the integral term ignores A).
//
// Sweep 1 is the ordinary per-event intensity sweep (whatever family applies: sparse / child-major / time-tiled).
// Sweep 2 is child-major (see cont_child.cu): a CTA owns a child node c, keeps the K raw-parameter entries of column c
// and the K-long accumulators of dW[:,c], dp1[:,c], dp2[:,c] in shared memory, walks the child events of c with one
// warp per event and coalesced window reads, and scatters each pair's terms with shared-memory atomics; the columns
// are flushed to the K^2 planes once per child.  Pairs whose effective weight is structurally zero (a = 0) cost one
// shared-memory read.  The result lives in the statistics buffers (dlambda0 -> M0 slot, dW -> Mnm, dp1 -> S1,
// dp2 -> S2), so the multi-GPU reduction is the same two all-reduces as for the Gibbs statistics.
//
// The walk is a template over the per-pair terms it scatters: the gradient's (TERMS_GRAD), or the expected parent
// statistics of mean-field VB (TERMS_VB, cont_vb.cu): with u = W h(dt) / lambda_i the probability that the pair is the
// child's parent, (u, u dt) for Exponential and (u, u dz, u dz^2) for LogitNormal, dz = logit(dt / D) - mu.
#include "cont_sweep.cuh"
#include <algorithm>

constexpr int GR_EVENTS = 256;  // child events per work item (as the child-major sweep)

struct GEntry { double c0, w, p1, p2; };  // EX: c0 = a theta, w = a W, p1 = theta;  LN: c0 = a D^2 sqrt(tau / 2 pi), w = W, p1 = mu, p2 = tau

struct GradArgs {
    SweepArgs s;
    const int *order, *node_ptr, *item_node, *item_e0;
    int64_t nitems;
    const double *W, *A, *p1, *p2;  // raw K x K parent-major planes (A may be NULL)
    const double *lam;              // [n_own] total intensity at every own event (sweep 1)
    double *g_l0, *g_w, *g_p1, *g_p2;
    int acc_smem;                   // accumulators in shared memory (else straight to the global planes)
    const unsigned short *wlen;     // [n_own] cached window length per own event (65535 = saturated)
};

template <int KIND> __device__ __forceinline__ GEntry make_entry(const GradArgs &ga, int64_t k, double D) {
    const double a = ga.A ? ga.A[k] : 1.0, w = ga.W[k];
    GEntry e;
    if (KIND == NHP_EXPONENTIAL) { e.p1 = ga.p1[k]; e.p2 = 0.0; e.c0 = a * e.p1; e.w = a * w; }
    else { e.p1 = ga.p1[k]; e.p2 = ga.p2[k]; e.c0 = a * D * D * sqrt(e.p2 * 0.15915494309189535); e.w = w; }
    return e;
}

enum { TERMS_GRAD = 0, TERMS_VB = 1 };

// the three per-pair terms (already divided by lambda_i); returns false when the pair contributes nothing
template <int KIND, int TERMS> __device__ __forceinline__ bool pair_terms(const GEntry &en, double dt, double D, double inv, const FastTables *ft, double &tw,
                                                                         double &t1, double &t2) {
    if (en.c0 == 0.0) return false;
    if (KIND == NHP_EXPONENTIAL) {
        if (dt < 0.0) return false;
        const double x = -en.p1 * dt;
        const double ex = (__double2hiint(x) >= 0x40862800) ? exp(x) : fast_exp_c(x, ft);
        tw = en.c0 * ex * inv;
        if (TERMS == TERMS_VB) {  // u = W theta e^{-theta dt} / lambda_i, u dt
            tw *= en.w;
            t1 = tw * dt;
        } else t1 = en.w * ex * fma(-en.p1, dt, 1.0) * inv;
        t2 = 0.0;
        return true;
    }
    const double b = D - dt;
    if (!(dt > 0.0 && b > 0.0)) return false;  // pdf is zero outside 0 < x < 1
    double dz, pj;  // z - mu and the Jacobian 1 / (dt b), as pair_value(EntryLN)
    if (in_mid_range(dt) && in_mid_range(b)) {
        pj = fast_rcp_mid(dt * b);
        dz = fast_log_n(dt * dt * pj, ft) - en.p1;
    } else {
        pj = 1.0 / (dt * b);
        dz = (log(dt) - log(b)) - en.p1;
    }
    const double ex = fast_exp(-(0.5 * en.p2) * dz * dz, ft);
    const double ha = en.c0 * pj * ex * inv;  // a h / lambda_i
    const double v = en.w * ha;               // a W h / lambda_i
    if (TERMS == TERMS_VB) {                  // u, u dz, u dz^2
        tw = v;
        t1 = v * dz;
        t2 = t1 * dz;
        return true;
    }
    tw = ha;
    t1 = v * en.p2 * dz;
    t2 = v * (0.5 / en.p2 - 0.5 * dz * dz);
    return true;
}

template <int KIND, int TERMS> __global__ void __launch_bounds__(1024) k_child_grad(const GradArgs ga) {
    const SweepArgs &a = ga.s;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ FastTables s_ft;
    __shared__ double red[64];
    const int BS = blockDim.x;
    constexpr int NP = KIND == NHP_LOGITNORMAL ? 3 : 2;
    GEntry *col = reinterpret_cast<GEntry *>(smem);                                    // [K] raw parameters of column c
    double *acc = reinterpret_cast<double *>(smem + (size_t)a.K * sizeof(GEntry));    // [NP][K] when acc_smem
    fast_tables_load(&s_ft);
    const FastTables *ft = &s_ft;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t ipc = (ga.nitems + gridDim.x - 1) / gridDim.x;
    const int64_t it0 = blockIdx.x * ipc, it1 = min(ga.nitems, it0 + ipc);
    double sum_log = 0.0, sum_row = 0.0;
    int cur = -1;
    auto flush = [&](int c) {  // accumulated columns -> global planes (several CTAs may share a child)
        if (!ga.acc_smem || c < 0) return;
        __syncthreads();
        for (int k = threadIdx.x; k < a.K; k += BS) {
            const int64_t o = k + (int64_t)a.K * c;
            double v = acc[k];
            if (v != 0.0) { red_add_f64(ga.g_w + o, v); acc[k] = 0.0; }
            v = acc[a.K + k];
            if (v != 0.0) { red_add_f64(ga.g_p1 + o, v); acc[a.K + k] = 0.0; }
            if (NP == 3) {
                v = acc[2 * a.K + k];
                if (v != 0.0) { red_add_f64(ga.g_p2 + o, v); acc[2 * a.K + k] = 0.0; }
            }
        }
    };
    if (ga.acc_smem) for (int k = threadIdx.x; k < NP * a.K; k += BS) acc[k] = 0.0;
    for (int64_t item = it0; item < it1; item++) {
        const int c = ga.item_node[item];
        if (c != cur) {
            flush(cur);
            __syncthreads();
            for (int k = threadIdx.x; k < a.K; k += BS) col[k] = make_entry<KIND>(ga, k + (int64_t)a.K * c, a.D);
            cur = c;
            __syncthreads();
        }
        const int e0 = ga.item_e0[item], e1 = min(e0 + GR_EVENTS, ga.node_ptr[c + 1]);
        double inv_sum = 0.0;
        for (int e = e0 + warp; e < e1; e += BS / 32) {
            const int i = ga.order[e];
            const double ti = __ldg(a.t + i);
            const double thr = ti - a.horizon;
            const int jlo = (int)a.jmin;
            const double lam = __ldg(ga.lam + (i - a.first));
            const double inv = 1.0 / lam;
            if (lane == 0) {
                if (TERMS == TERMS_GRAD) sum_log += log(lam);
                inv_sum += inv;
            }
            const int wraw = (int)__ldg(ga.wlen + (i - a.first));
            const int w = wraw < 65535 ? min(wraw, i - jlo) : i - jlo;  // known trip count: loads of several trips in flight
#pragma unroll 2
            for (int k = lane; k < w; k += 32) {
                const int j = i - 1 - k;
                const double tj = __ldg(a.t + j);
                if (wraw >= 65535 && !(tj > thr)) break;
                const int p = __ldg(a.c + j);
                double tw, t1, t2;
                if (!pair_terms<KIND, TERMS>(col[p], ti - tj, a.D, inv, ft, tw, t1, t2)) continue;
                if (ga.acc_smem) {
                    atomicAdd(acc + p, tw);
                    atomicAdd(acc + a.K + p, t1);
                    if (NP == 3) atomicAdd(acc + 2 * a.K + p, t2);
                } else {
                    const int64_t o = p + (int64_t)a.K * c;
                    red_add_f64(ga.g_w + o, tw);
                    red_add_f64(ga.g_p1 + o, t1);
                    if (NP == 3) red_add_f64(ga.g_p2 + o, t2);
                }
            }
        }
        if (lane == 0 && inv_sum != 0.0) red_add_f64(ga.g_l0 + c, inv_sum);
    }
    flush(cur);
    block_sum2_any(sum_log, sum_row, red);
    if (threadIdx.x == 0) { a.partials[2 * (size_t)blockIdx.x] = sum_log; a.partials[2 * (size_t)blockIdx.x + 1] = 0.0; }
}

// compensator terms of this shard: dlambda0 -= T on the first shard; dW[p,c] -= Mn[p] * (A[p,c] or 1)
__global__ void k_grad_finish(int K, const double *__restrict__ Mn, const double *__restrict__ A, int ignore_A, double T_first, double *__restrict__ g_l0,
                              double *__restrict__ g_w) {
    const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < K) g_l0[k] -= T_first;
    if (k < (int64_t)K * K) {
        const int p = (int)(k % K);
        const double a = (A && !ignore_A) ? A[k] : 1.0;
        g_w[k] -= Mn[p] * a;
    }
}

int nhp_cont_fill_args(nhp_ctx *ctx, nhp_events *ev, int recursive, SweepArgs &a);                 // cont_sweep.cu
int nhp_cont_run_event_intensity(nhp_ctx *ctx, nhp_events *ev, int recursive, double *d_out);     // cont_sweep.cu
int nhp_cont_reduce_partials(nhp_ctx *ctx, nhp_events *ev, const double *partials, int grid, const double *rowsum);  // cont_sweep.cu

// Sweep 2 of the gradient and of the VB statistics: the child-major scatter of the per-pair terms (`terms`: TERMS_GRAD | TERMS_VB)
// of the context's parameters, given lam[n_own] = lambda_i of sweep 1, added into the zeroed planes g_l0[K] (sum of 1 / lambda_i per
// child node), g_w, g_p1, g_p2 [K*K].  a: nhp_cont_fill_args of this call; its `partials` receive the per-CTA log-sums (TERMS_GRAD).
// *grid_out = CTAs launched (0: no work items).
int nhp_cont_child_scatter(nhp_ctx *ctx, nhp_events *ev, SweepArgs &a, const double *lam, int terms, double *g_l0, double *g_w, double *g_p1,
                           double *g_p2, int *grid_out) {
    const int64_t K = ctx->K;
    cudaStream_t s = ctx->stream;
    *grid_out = 0;
    NHP_TRY(nhp_events_build_node_index(ctx, ev));
    NHP_CUDA(ctx, fast_tables_upload(s));
    GradArgs ga;
    ga.s = a; ga.order = ev->d_order; ga.node_ptr = ev->d_node_ptr; ga.item_node = ev->d_item_node; ga.item_e0 = ev->d_item_e0; ga.nitems = ev->n_items;
    ga.W = ctx->d_W; ga.A = ctx->has_A ? ctx->d_A : nullptr; ga.p1 = ctx->d_p1; ga.p2 = ctx->d_p2; ga.lam = lam;
    ga.g_l0 = g_l0; ga.g_w = g_w; ga.g_p1 = g_p1; ga.g_p2 = g_p2; ga.wlen = ev->d_wlen;
    const int np = ctx->kind == NHP_LOGITNORMAL ? 3 : 2;
    const size_t lim = (size_t)ctx->smem_optin - 8192;
    size_t smem = (size_t)K * (sizeof(GEntry) + np * sizeof(double));
    ga.acc_smem = smem <= lim;
    { const char *eg = getenv("NHP_GRAD_SMEM"); if (eg && atoi(eg) == 0) ga.acc_smem = 0; }  // A/B: accumulate with global RED.ADD.F64 instead
    if (!ga.acc_smem) smem = (size_t)K * sizeof(GEntry);
    NHP_CHECK(ctx, smem <= lim, NHP_ERR_INVALID, "%s: K=%lld needs %zu bytes of shared memory per CTA (limit %zu)",
              terms == TERMS_VB ? "nhp_cont_vb" : "nhp_cont_loglik_grad", (long long)K, smem, lim);
    NHP_TRY(nhp_partials(ctx, 2 * (int64_t)ctx->sm_count * 32, &a.partials));
    ga.s.partials = a.partials;
    auto launch = [&](auto kernel) -> int {
        NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
        NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int per_sm = 1;
        const int fit = (int)std::max<size_t>(1, lim / std::max<size_t>(smem, 1));
        const int block = fit >= 8 ? 256 : (fit >= 4 ? 512 : 1024);  // big columns leave room for few CTAs per SM: give them more warps
        NHP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
        const int grid = (int)std::min<int64_t>(ev->n_items, (int64_t)ctx->sm_count * std::max(per_sm, 1));
        kernel<<<grid, block, smem, s>>>(ga);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
        *grid_out = grid;
        return NHP_OK;
    };
    if (ev->n_items == 0) return NHP_OK;
    const bool ln = ctx->kind == NHP_LOGITNORMAL;
    if (terms == TERMS_VB) return ln ? launch(k_child_grad<NHP_LOGITNORMAL, TERMS_VB>) : launch(k_child_grad<NHP_EXPONENTIAL, TERMS_VB>);
    return ln ? launch(k_child_grad<NHP_LOGITNORMAL, TERMS_GRAD>) : launch(k_child_grad<NHP_EXPONENTIAL, TERMS_GRAD>);
}

extern "C" int nhp_cont_loglik_grad_dev(nhp_ctx *ctx, nhp_events *ev, int recursive) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    SweepArgs a;
    NHP_TRY(nhp_cont_fill_args(ctx, ev, recursive, a));
    NHP_CHECK(ctx, a.lam0ev == nullptr, NHP_ERR_UNSUPPORTED, "the analytic gradient takes a homogeneous baseline");
    const int64_t K = ctx->K, own = ev->n - ev->n_halo;
    const StatsLayout sl{K};
    cudaStream_t s = ctx->stream;
    ctx->parents_valid = false;
    ctx->sweep_ll_valid = false;
    // gradient planes live in the statistics buffers: dlambda0 -> M0, dW -> Mnm, dp1 -> S1, dp2 -> S2
    double *g_l0 = ctx->d_stats0 + sl.off_M0(), *g_w = ctx->d_stats0 + sl.off_Mnm(), *g_p1 = ctx->d_stats0 + sl.off_S1(), *g_p2 = ctx->d_stats1;
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats0, 0, (size_t)sl.total() * sizeof(double), s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_stats0 + sl.off_Mn(), ev->d_Mn, (size_t)K * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats1, 0, (size_t)(K * K) * sizeof(double), s));
    const bool rec = recursive && ctx->kind == NHP_EXPONENTIAL;
    NHP_TRY(nhp_timer_begin(ctx));
    if (own > 0) {
        // sweep 1: lambda_i (scratch holds it; nothing else uses the scratch area until the call returns)
        void *scratch;
        NHP_TRY(nhp_scratch(ctx, (size_t)own * sizeof(double), &scratch));
        NHP_TRY(nhp_cont_run_event_intensity(ctx, ev, recursive, (double *)scratch));
        // sweep 2: child-major scatter of the per-pair terms
        int grid = 0;
        NHP_TRY(nhp_cont_child_scatter(ctx, ev, a, (const double *)scratch, TERMS_GRAD, g_l0, g_w, g_p1, g_p2, &grid));
        if (grid > 0) NHP_TRY(nhp_cont_reduce_partials(ctx, ev, a.partials, grid, a.rowsum));
    }
    const double T_first = (ev->flags & 1) ? ev->duration : 0.0;
    k_grad_finish<<<(unsigned)((K * K + 255) / 256), 256, 0, s>>>((int)K, ev->d_Mn, ctx->has_A ? ctx->d_A : nullptr, rec && ctx->has_A ? 1 : 0, T_first, g_l0, g_w);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    NHP_TRY(nhp_timer_end(ctx));
    ctx->grad_valid = true;
    return NHP_OK;
}

extern "C" int nhp_cont_loglik_grad_read(nhp_ctx *ctx, nhp_events *ev, double *ll, double *dlambda0, double *dW, double *dp1, double *dp2) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "nhp_cont_loglik_grad_read: events handle is NULL");
    NHP_CHECK(ctx, ctx->grad_valid, NHP_ERR_STATE, "nhp_cont_loglik_grad_read: run nhp_cont_loglik_grad_dev first");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t K = ctx->K;
    const StatsLayout sl{K};
    cudaStream_t s = ctx->stream;
    double h[2] = {0.0, 0.0};
    NHP_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_stats0, sizeof(h), cudaMemcpyDeviceToHost, s));
    if (dlambda0) NHP_CUDA(ctx, cudaMemcpyAsync(dlambda0, ctx->d_stats0 + sl.off_M0(), (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (dW) NHP_CUDA(ctx, cudaMemcpyAsync(dW, ctx->d_stats0 + sl.off_Mnm(), (size_t)(K * K) * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (dp1) NHP_CUDA(ctx, cudaMemcpyAsync(dp1, ctx->d_stats0 + sl.off_S1(), (size_t)(K * K) * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (dp2) NHP_CUDA(ctx, cudaMemcpyAsync(dp2, ctx->d_stats1, (size_t)(K * K) * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    const double base = nhp_cont_baseline_term(ctx, ev);
    if (ll) *ll = h[0] - h[1] - base;
    return NHP_OK;
}

extern "C" int nhp_cont_loglik_grad(nhp_ctx *ctx, nhp_events *ev, int recursive, double *ll, double *dlambda0, double *dW, double *dp1, double *dp2) {
    NHP_TRY(nhp_cont_loglik_grad_dev(ctx, ev, recursive));
    return nhp_cont_loglik_grad_read(ctx, ev, ll, dlambda0, dW, dp1, dp2);
}
