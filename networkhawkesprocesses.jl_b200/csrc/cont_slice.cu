// cont_slice.cu -- the elliptical-slice update of LogGaussianCoxProcess curves on the device (baselines.jl:214-326).
//
// resample!(process::LogGaussianCoxProcess, data, parents) moves every node's log-curve y_k = log(lambda_k) - m on the ellipse
// through y_k and a prior draw nu_k = L z_k [Murray, Adams & MacKay 2010].  The slice likelihood of node k is
//   ll_k(f) = -trapezoid(f) + sum over the events of node k whose parent is the baseline of log f(t_i),
// so it depends on that node's baseline-attributed events only.  The update runs in lockstep rounds:
//   * once per update, the baseline events of every node are collected from the by-node order of the handle (d_order,
//     d_node_ptr) and the parent offsets (d_poff) into compact records (grid interval, time) at the node's own offset, and
//     split into work items of at most SL_ITEM events;
//   * round 0 evaluates the current curves, every later round one candidate per node that is still active: one warp per
//     work item writes a partial log-sum, then one warp per node sums its partials in a fixed order (same inputs, same bits),
//     adds -trapezoid once, accepts or shrinks the bracket and writes the next candidate;
//   * a multi-GPU job all-reduces the K per-node sums between the two kernels: every rank draws the same random numbers and
//     reaches the same decisions, so the curves agree without a broadcast;
//   * the host reads the active count (4 bytes) per round; the curves replace the context's only when every node accepted.
// The random numbers are consumed in the layout of the host mirror (LogGaussianCoxProcess.resample_): z[g + G k] standard
// normals, u[j + 101 k] with j = 0 the slice height and j = 1 + a the angle uniform of attempt a.
#include "nhp_internal.cuh"
#include <algorithm>
#include <chrono>
#include <cmath>
#include <vector>

constexpr int SL_MAX_ATTEMPTS = 100;             // baselines.jl:316
constexpr int SL_NU = 1 + SL_MAX_ATTEMPTS;       // uniforms per node
constexpr int SL_ITEM = 512;                     // baseline events per work item (one warp)
constexpr int SL_MAX_GRID = 4096;                // largest grid of nhp_cont_baseline_prior
constexpr double SL_TWO_PI = 6.283185307179586;  // 2.0 * pi in double, as numpy forms it

struct SliceState { double theta, lo, hi, lly; };

struct SliceArgs {
    int K, G;
    double m;
    const double *x;             // [G] grid
    const double *z, *u;         // [K][G] normals, [K][SL_NU] uniforms
    double *y, *nu, *cand;       // [K][G] current log-curve - m, prior draw, candidate curve
    double *integ, *cmin;        // [K] trapezoid and minimum of the candidate
    SliceState *st;              // [K]
    int *active, *att, *cnt;     // [K] still searching, candidates evaluated, baseline events
    int *item_ptr, *item_node;   // [K+1] first work item of every node, [items] node of every work item
    const int *node_ptr;         // [K+1] by-node offsets of the handle
    const int *rg;               // [own] grid interval of every baseline record (G - 1: the last grid point)
    const double *rt;            // [own] time of every baseline record
    double *part;                // [items] partial log-sums
    int *ctl;                    // [4] active count, error flags
};

// Philox4x32-10 keyed by seed ^ "ELLIPSLC", counter words (node, draw index, sweep counter)
__device__ __forceinline__ void slice_philox(uint64_t seed, uint32_t node, uint32_t draw, uint64_t counter, uint32_t r[4]) {
    const uint64_t key = seed ^ 0x454C4C4950534C43ull;
    philox4x32_10(node, draw, (uint32_t)counter, (uint32_t)(counter >> 32), (uint32_t)key, (uint32_t)(key >> 32), r);
}
__device__ __forceinline__ double slice_u53(uint32_t hi, uint32_t lo) {  // (0, 1): 53 bits, never exactly 0
    const uint64_t v = (((uint64_t)hi << 32) | (uint64_t)lo) >> 11;
    return ((double)v + 0.5) * 1.1102230246251565e-16;
}
// z[g + G k] = Box-Muller normal of draw g of node k; u[j + SL_NU k] = uniform of draw 2^31 + j
__global__ void k_slice_draw(uint64_t seed, uint64_t counter, int K, int G, double *__restrict__ z, double *__restrict__ u) {
    const int64_t nz = (int64_t)K * G, n = nz + (int64_t)K * SL_NU;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < n; e += (int64_t)gridDim.x * blockDim.x) {
        uint32_t r[4];
        if (e < nz) {
            const int k = (int)(e / G), g = (int)(e % G);
            slice_philox(seed, (uint32_t)k, (uint32_t)g, counter, r);
            z[e] = sqrt(-2.0 * log(slice_u53(r[0], r[1]))) * cospi(2.0 * slice_u53(r[2], r[3]));
        } else {
            const int64_t f = e - nz;
            const int k = (int)(f / SL_NU), j = (int)(f % SL_NU);
            slice_philox(seed, (uint32_t)k, 0x80000000u | (uint32_t)j, counter, r);
            u[f] = slice_u53(r[0], r[1]);
        }
    }
}

// one CTA per node: nu = L z (lower triangle of the column-major L), y = log(v) - m, candidate = current curve, its trapezoid
__global__ void k_slice_setup(SliceArgs a, const double *__restrict__ L, const double *__restrict__ v) {
    extern __shared__ double s_z[];
    __shared__ double s_red[32];
    const int G = a.G;
    for (int k = blockIdx.x; k < a.K; k += gridDim.x) {
        for (int g = threadIdx.x; g < G; g += blockDim.x) s_z[g] = a.z[(int64_t)k * G + g];
        __syncthreads();
        const double *vk = v + (int64_t)k * G;
        double tr = 0.0;
        for (int g = threadIdx.x; g < G; g += blockDim.x) {
            double s = 0.0;
            for (int h = 0; h <= g; h++) s = fma(L[g + (int64_t)G * h], s_z[h], s);
            a.nu[(int64_t)k * G + g] = s;
            a.y[(int64_t)k * G + g] = log(vk[g]) - a.m;
            a.cand[(int64_t)k * G + g] = vk[g];
            if (g + 1 < G) tr += 0.5 * (vk[g] + vk[g + 1]) * (a.x[g + 1] - a.x[g]);
        }
        for (int d = 16; d > 0; d >>= 1) tr += __shfl_xor_sync(0xffffffffu, tr, d);
        if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = tr;
        __syncthreads();
        if (threadIdx.x == 0) {
            for (int w = 1; w < (int)(blockDim.x >> 5); w++) tr += s_red[w];
            a.integ[k] = tr;
            a.active[k] = 1;
            a.att[k] = 0;
        }
        __syncthreads();
    }
}

// one warp per node: the node's baseline events (parent offset 0) in by-node order -> records (grid interval, time) at
// node_ptr[k]; cnt[k] = their number.  ctl[1] bit 256: a time outside the grid, bit 512: no parent assignment
__global__ void k_slice_collect(SliceArgs a, const double *__restrict__ t, const int *__restrict__ poff, const int *__restrict__ order,
                                int *__restrict__ rg, double *__restrict__ rt) {
    const int lane = threadIdx.x & 31, G = a.G;
    const double *x = a.x;
    for (int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); k < a.K; k += gridDim.x * (blockDim.x >> 5)) {
        const int e0 = a.node_ptr[k], e1 = a.node_ptr[k + 1];
        int n = 0, bad = 0;
        for (int eb = e0; eb < e1; eb += 32) {
            const int e = eb + lane;
            int po = 1, g = 0;
            double ti = 0.0;
            if (e < e1) {
                const int i = order[e];
                po = poff[i];
                if (po < 0) bad |= 512;
                if (po == 0) {
                    ti = t[i];
                    if (!(ti >= x[0]) || !(ti <= x[G - 1])) { bad |= 256; g = 0; }
                    else if (ti >= x[G - 1]) g = G - 1;
                    else {
                        int lo = 0, hi = G - 1;  // last g with x[g] <= t (grid_interp)
                        while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (x[mid] <= ti) lo = mid; else hi = mid; }
                        g = lo;
                    }
                }
            }
            const unsigned m = __ballot_sync(0xffffffffu, po == 0);
            if (po == 0) {
                const int p = e0 + n + __popc(m & ((1u << lane) - 1u));
                rg[p] = g; rt[p] = ti;
            }
            n += __popc(m);
        }
        for (int d = 16; d > 0; d >>= 1) bad |= __shfl_xor_sync(0xffffffffu, bad, d);
        if (lane == 0) {
            a.cnt[k] = n;
            if (bad) atomicOr(a.ctl + 1, bad);
        }
    }
}

// one CTA: item_ptr = exclusive scan of ceil(cnt / SL_ITEM) over the nodes, item_node of every work item
__global__ void k_slice_items(SliceArgs a) {
    __shared__ int s_sum[1024];
    const int K = a.K, per = (K + blockDim.x - 1) / blockDim.x;
    const int k0 = min(K, (int)threadIdx.x * per), k1 = min(K, k0 + per);
    int loc = 0;
    for (int k = k0; k < k1; k++) loc += (a.cnt[k] + SL_ITEM - 1) / SL_ITEM;
    s_sum[threadIdx.x] = loc;
    __syncthreads();
    for (int d = 1; d < (int)blockDim.x; d <<= 1) {  // inclusive Hillis-Steele scan
        const int v = threadIdx.x >= (unsigned)d ? s_sum[threadIdx.x - d] : 0;
        __syncthreads();
        s_sum[threadIdx.x] += v;
        __syncthreads();
    }
    int run = s_sum[threadIdx.x] - loc;
    for (int k = k0; k < k1; k++) {
        const int ni = (a.cnt[k] + SL_ITEM - 1) / SL_ITEM;
        a.item_ptr[k] = run;
        for (int j = 0; j < ni; j++) a.item_node[run + j] = k;
        run += ni;
    }
    if (threadIdx.x == blockDim.x - 1) a.item_ptr[K] = s_sum[threadIdx.x];
}

// one warp per work item of an active node: partial sum of log f(t_i) over its records, f the node's candidate curve
__global__ void __launch_bounds__(256) k_slice_round(SliceArgs a) {
    __shared__ FastTables ft;
    fast_tables_load(&ft);
    __syncthreads();
    const int lane = threadIdx.x & 31, G = a.G, n_items = a.item_ptr[a.K];
    for (int w = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); w < n_items; w += gridDim.x * (blockDim.x >> 5)) {
        const int k = a.item_node[w];
        if (!a.active[k]) continue;
        const int j = w - a.item_ptr[k], p0 = a.node_ptr[k] + j * SL_ITEM, len = min(SL_ITEM, a.cnt[k] - j * SL_ITEM);
        const double *v = a.cand + (int64_t)k * G;
        double s = 0.0;
        for (int e = lane; e < len; e += 32) {
            const int g = a.rg[p0 + e];
            const double ti = a.rt[p0 + e];
            double f;
            if (g == G - 1) f = v[g];
            else {
                const double x0 = a.x[g], x1 = a.x[g + 1];
                f = (v[g + 1] * (ti - x0) + v[g] * (x1 - ti)) / (x1 - x0);  // interpolation.jl:31
            }
            s += fast_log(f, &ft);
        }
        for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
        if (lane == 0) a.part[w] = s;
    }
}

// the node's partials in a fixed order (lane-strided, then a butterfly): every lane returns the same value
__device__ __forceinline__ double slice_node_sum(const SliceArgs &a, int k, int lane) {
    double s = 0.0;
    for (int w = a.item_ptr[k] + lane; w < a.item_ptr[k + 1]; w += 32) s += a.part[w];
    for (int d = 16; d > 0; d >>= 1) s += __shfl_xor_sync(0xffffffffu, s, d);
    return s;
}

// multi-GPU: the per-node sums of this rank's shard, all-reduced before k_slice_decide
__global__ void k_slice_node_sums(SliceArgs a, double *__restrict__ nsum) {
    const int lane = threadIdx.x & 31;
    for (int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); k < a.K; k += gridDim.x * (blockDim.x >> 5)) {
        const double s = a.active[k] ? slice_node_sum(a, k, lane) : 0.0;
        if (lane == 0) nsum[k] = s;
    }
}

// one warp per active node: the slice decision of round `round` (round 0: the current curve), then the next candidate
//   exp(m + y cos(theta) + nu sin(theta)),  its trapezoid and minimum.  Products and sums are rounded one by one, as numpy
// evaluates them.  ctl[0] counts the nodes still active; a node whose 100th candidate is rejected stays active without a new
// candidate (the caller reports the attempt limit).
__global__ void k_slice_decide(SliceArgs a, int round, const double *__restrict__ nsum) {
    const int lane = threadIdx.x & 31, G = a.G;
    for (int k = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5); k < a.K; k += gridDim.x * (blockDim.x >> 5)) {
        if (!a.active[k]) continue;
        const double ll = (nsum ? nsum[k] : slice_node_sum(a, k, lane)) - a.integ[k];
        const double *u = a.u + (int64_t)k * SL_NU;
        SliceState st = a.st[k];
        bool next = true, keep = true;  // write a new candidate; still active after this round
        if (round == 0) {
            st.lly = ll + log(u[0]);
            st.theta = __dmul_rn(SL_TWO_PI, u[1]);            // rng.uniform(0, 2 pi)
            st.lo = __dsub_rn(st.theta, SL_TWO_PI); st.hi = st.theta;
        } else if (ll >= st.lly) {
            next = keep = false;                              // accepted: the candidate stays in cand
            if (lane == 0) { a.active[k] = 0; a.att[k] = round; }
        } else {
            const int at = round - 1;                         // the attempt just rejected
            if (st.theta < 0.0) st.lo = st.theta; else st.hi = st.theta;
            if (at + 1 >= SL_MAX_ATTEMPTS) {
                next = false;
                if (lane == 0) a.att[k] = round;
            } else {
                st.theta = __dadd_rn(st.lo, __dmul_rn(__dsub_rn(st.hi, st.lo), u[2 + at]));  // rng.uniform(lo, hi)
            }
        }
        if (lane == 0) a.st[k] = st;
        if (next) {
            double sn, cs;
            sincos(st.theta, &sn, &cs);
            double *c = a.cand + (int64_t)k * G;
            const double *y = a.y + (int64_t)k * G, *nu = a.nu + (int64_t)k * G;
            for (int g = lane; g < G; g += 32) c[g] = exp(__dadd_rn(a.m, __dadd_rn(__dmul_rn(y[g], cs), __dmul_rn(nu[g], sn))));
            __syncwarp();
            double tr = 0.0, mn = INFINITY;
            for (int g = lane; g < G; g += 32) {
                mn = fmin(mn, c[g]);
                if (g + 1 < G) tr += 0.5 * (c[g] + c[g + 1]) * (a.x[g + 1] - a.x[g]);
            }
            for (int d = 16; d > 0; d >>= 1) {
                tr += __shfl_xor_sync(0xffffffffu, tr, d);
                mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, d));
            }
            if (lane == 0) { a.integ[k] = tr; a.cmin[k] = mn; }
        }
        if (lane == 0 && keep) atomicAdd(a.ctl, 1);
    }
}

// one CTA: sum of the accepted curves' integrals and their minimum
__global__ void k_slice_commit(SliceArgs a, double *__restrict__ out2) {
    __shared__ double s_t[32], s_m[32];
    double tr = 0.0, mn = INFINITY;
    for (int k = threadIdx.x; k < a.K; k += blockDim.x) { tr += a.integ[k]; mn = fmin(mn, a.cmin[k]); }
    for (int d = 16; d > 0; d >>= 1) { tr += __shfl_xor_sync(0xffffffffu, tr, d); mn = fmin(mn, __shfl_xor_sync(0xffffffffu, mn, d)); }
    if ((threadIdx.x & 31) == 0) { s_t[threadIdx.x >> 5] = tr; s_m[threadIdx.x >> 5] = mn; }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (int w = 1; w < (int)(blockDim.x >> 5); w++) { tr += s_t[w]; mn = fmin(mn, s_m[w]); }
        out2[0] = tr; out2[1] = mn;
    }
}

int nhp_comm_allreduce_dev(nhp_ctx *ctx, double *buf, int64_t n);  // comm.cu

extern "C" int nhp_cont_baseline_prior(nhp_ctx *ctx, int64_t n_grid, const double *L, double m) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set && ctx->bgrid_n > 0, NHP_ERR_STATE, "nhp_cont_baseline_prior: set the curves first (nhp_cont_baseline_grid)");
    NHP_CHECK(ctx, n_grid == ctx->bgrid_n && n_grid <= SL_MAX_GRID && L != nullptr, NHP_ERR_INVALID,
              "nhp_cont_baseline_prior: the prior needs the curves' grid (%lld points, at most %d) and its Cholesky factor", (long long)ctx->bgrid_n, SL_MAX_GRID);
    NHP_CHECK(ctx, std::isfinite(m), NHP_ERR_INVALID, "nhp_cont_baseline_prior: the mean m must be finite");
    const int64_t G = n_grid;
    std::vector<double> low((size_t)(G * G), 0.0);
    for (int64_t h = 0; h < G; h++)
        for (int64_t g = h; g < G; g++) {
            const double v = L[g + G * h];
            NHP_CHECK(ctx, std::isfinite(v) && (g != h || v > 0.0), NHP_ERR_INVALID,
                      "nhp_cont_baseline_prior: L must be a finite lower-triangular factor with a positive diagonal (entry %lld, %lld)", (long long)g, (long long)h);
            low[(size_t)(g + G * h)] = v;  // the strictly upper triangle is ignored
        }
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ctx->bprior_cap < G) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_bprior_L); ctx->d_bprior_L = nullptr; ctx->bprior_cap = 0;
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_bprior_L, (size_t)(G * G) * sizeof(double)));
        ctx->bprior_cap = G;
    }
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bprior_L, low.data(), (size_t)(G * G) * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    ctx->bprior_n = G; ctx->bprior_m = m;
    return NHP_OK;
}

extern "C" int nhp_cont_baseline_get(nhp_ctx *ctx, double *values) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, values != nullptr, NHP_ERR_INVALID, "nhp_cont_baseline_get: NULL argument");
    NHP_CHECK(ctx, ctx->cont_set && ctx->bgrid_n > 0, NHP_ERR_STATE, "nhp_cont_baseline_get: the context holds no curves");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CUDA(ctx, cudaMemcpyAsync(values, ctx->d_bgrid_v, (size_t)(ctx->K * ctx->bgrid_n) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

static int slice_buffers(nhp_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->slice_cap) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(ctx->d_slice); ctx->d_slice = nullptr; ctx->slice_cap = 0;
        NHP_CUDA(ctx, cudaMalloc(&ctx->d_slice, bytes));
        ctx->slice_cap = bytes;
    }
    *out = ctx->d_slice;
    return NHP_OK;
}

// the events handle's record and work-item arrays (sized by its own events, kept for later updates)
static int slice_event_buffers(nhp_ctx *ctx, nhp_events *ev) {
    const int64_t own = ev->n - ev->n_halo, items = own / SL_ITEM + ev->K + 1;
    if (ev->d_sl_g) return NHP_OK;
    cudaStream_t s = ctx->stream;
    auto fail = [&](cudaError_t e) {
        cudaFreeAsync(ev->d_sl_g, s); cudaFreeAsync(ev->d_sl_t, s); cudaFreeAsync(ev->d_sl_item, s); cudaFreeAsync(ev->d_sl_part, s);
        ev->d_sl_g = ev->d_sl_item = nullptr; ev->d_sl_t = ev->d_sl_part = nullptr;
        return nhp_fail(ctx, NHP_ERR_CUDA, "slice update: cudaMallocAsync failed: %s", cudaGetErrorString(e));
    };
    cudaError_t e;
    if ((e = cudaMallocAsync(&ev->d_sl_g, (size_t)std::max<int64_t>(own, 1) * sizeof(int), s)) != cudaSuccess) return fail(e);
    if ((e = cudaMallocAsync(&ev->d_sl_t, (size_t)std::max<int64_t>(own, 1) * sizeof(double), s)) != cudaSuccess) return fail(e);
    if ((e = cudaMallocAsync(&ev->d_sl_item, (size_t)items * sizeof(int), s)) != cudaSuccess) return fail(e);
    if ((e = cudaMallocAsync(&ev->d_sl_part, (size_t)items * sizeof(double), s)) != cudaSuccess) return fail(e);
    return NHP_OK;
}

extern "C" int nhp_cont_resample_baseline(nhp_ctx *ctx, nhp_events *ev, uint64_t seed, uint64_t counter, const double *z, const double *u, int64_t *attempts) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "nhp_cont_resample_baseline: events handle is NULL");
    NHP_CHECK(ctx, (z == nullptr) == (u == nullptr), NHP_ERR_INVALID, "nhp_cont_resample_baseline: pass both z and u, or neither (Philox)");
    NHP_CHECK(ctx, ctx->cont_set && ev->K == ctx->K, NHP_ERR_STATE, "nhp_cont_resample_baseline: parameters not set for this data");
    NHP_CHECK(ctx, ctx->bgrid_n > 0, NHP_ERR_STATE, "nhp_cont_resample_baseline: the context holds no curves (nhp_cont_baseline_grid)");
    NHP_CHECK(ctx, ctx->bprior_n == ctx->bgrid_n, NHP_ERR_STATE, "nhp_cont_resample_baseline: no prior for the curves (nhp_cont_baseline_prior)");
    NHP_CHECK(ctx, ctx->parents_valid, NHP_ERR_STATE, "nhp_cont_resample_baseline: no parent assignment on the device (run nhp_cont_resample_parents first)");
    NHP_CHECK(ctx, ctx->bgrid_min > 0.0, NHP_ERR_NUMERIC, "nhp_cont_resample_baseline: a curve value is zero (its logarithm is the slice sampler's state)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const auto t0 = std::chrono::steady_clock::now();
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    cudaStream_t s = ctx->stream;
    const int64_t K = ctx->K, G = ctx->bgrid_n, KG = K * G;
    const bool multi = ctx->comm && ctx->nranks > 1;
    NHP_TRY(nhp_events_build_node_index(ctx, ev));
    NHP_TRY(slice_event_buffers(ctx, ev));
    // context buffers: doubles z, y, nu, cand [K G], u [K SL_NU], integ, cmin, nsum [K], state [K]; ints active, att, cnt [K],
    // item_ptr [K + 1], ctl [4]
    const size_t nd = (size_t)(4 * KG + K * SL_NU + 3 * K + 4 * K + 2), ni = (size_t)(4 * K + 1 + 4);
    void *buf = nullptr;
    NHP_TRY(slice_buffers(ctx, nd * sizeof(double) + ni * sizeof(int), &buf));
    double *dz = (double *)buf, *dy = dz + KG, *dnu = dy + KG, *dcand = dnu + KG, *du = dcand + KG, *dinteg = du + K * SL_NU;
    double *dcmin = dinteg + K, *dnsum = dcmin + K, *dout = dnsum + K;
    SliceState *dst = (SliceState *)(dout + 2);
    int *iact = (int *)(dst + K), *iatt = iact + K, *icnt = iatt + K, *iptr = icnt + K, *ictl = iptr + K + 1;
    SliceArgs a;
    a.K = (int)K; a.G = (int)G; a.m = ctx->bprior_m; a.x = ctx->d_bgrid_x; a.z = dz; a.u = du; a.y = dy; a.nu = dnu; a.cand = dcand;
    a.integ = dinteg; a.cmin = dcmin; a.st = dst; a.active = iact; a.att = iatt; a.cnt = icnt; a.item_ptr = iptr; a.item_node = ev->d_sl_item;
    a.node_ptr = ev->d_node_ptr; a.rg = ev->d_sl_g; a.rt = ev->d_sl_t; a.part = ev->d_sl_part; a.ctl = ictl;
    if (z) {
        NHP_CUDA(ctx, cudaMemcpyAsync(dz, z, (size_t)KG * sizeof(double), cudaMemcpyHostToDevice, s));
        NHP_CUDA(ctx, cudaMemcpyAsync(du, u, (size_t)(K * SL_NU) * sizeof(double), cudaMemcpyHostToDevice, s));
    } else {
        const int64_t n = KG + K * SL_NU;
        k_slice_draw<<<(unsigned)std::min<int64_t>((n + 255) / 256, (int64_t)ctx->sm_count * 16), 256, 0, s>>>(seed, counter, (int)K, (int)G, dz, du);
        NHP_LAUNCHED(ctx);
    }
    NHP_CUDA(ctx, cudaMemsetAsync(ictl, 0, 4 * sizeof(int), s));
    k_slice_setup<<<(unsigned)std::min<int64_t>(K, (int64_t)ctx->sm_count * 8), 256, (size_t)G * sizeof(double), s>>>(a, ctx->d_bprior_L, ctx->d_bgrid_v);
    NHP_LAUNCHED(ctx);
    const unsigned node_blocks = (unsigned)((K + 7) / 8);
    k_slice_collect<<<node_blocks, 256, 0, s>>>(a, ev->d_t, ev->d_poff, ev->d_order, ev->d_sl_g, ev->d_sl_t);
    NHP_LAUNCHED(ctx);
    k_slice_items<<<1, 1024, 0, s>>>(a);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    int hctl[3] = {0, 0, 0};  // work items (iptr[K]), ctl[0], ctl[1]: adjacent in the buffer
    NHP_CUDA(ctx, cudaMemcpyAsync(hctl, iptr + K, 3 * sizeof(int), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->slice_info[3] = (double)hctl[0];
    NHP_CHECK(ctx, !(hctl[2] & 256), NHP_ERR_INVALID, "baseline: an event time is outside the interpolation support of the grid (interpolation.jl:29)");
    NHP_CHECK(ctx, !(hctl[2] & 512), NHP_ERR_STATE, "nhp_cont_resample_baseline: events without a parent assignment");
    const auto t1 = std::chrono::steady_clock::now();
    const int64_t own = ev->n - ev->n_halo, max_items = own / SL_ITEM + K + 1;
    const unsigned round_blocks = (unsigned)std::max<int64_t>(1, std::min<int64_t>((max_items + 7) / 8, (int64_t)ctx->sm_count * 8));
    int round = 0;
    for (;; round++) {
        k_slice_round<<<round_blocks, 256, 0, s>>>(a);
        NHP_LAUNCHED(ctx);
        if (multi) {
            k_slice_node_sums<<<node_blocks, 256, 0, s>>>(a, dnsum);
            NHP_LAUNCHED(ctx);
            NHP_TRY(nhp_comm_allreduce_dev(ctx, dnsum, K));
        }
        NHP_CUDA(ctx, cudaMemsetAsync(ictl, 0, sizeof(int), s));
        k_slice_decide<<<node_blocks, 256, 0, s>>>(a, round, multi ? dnsum : nullptr);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
        int active = 0;
        NHP_CUDA(ctx, cudaMemcpyAsync(&active, ictl, sizeof(int), cudaMemcpyDeviceToHost, s));
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
        if (active == 0) break;
        NHP_CHECK(ctx, round < SL_MAX_ATTEMPTS, NHP_ERR_NUMERIC, "Elliptical slice sampling reached maximum attempts (baselines.jl:316): %d node(s)", active);
    }
    if (attempts) {
        std::vector<int> h((size_t)K);
        NHP_CUDA(ctx, cudaMemcpyAsync(h.data(), iatt, (size_t)K * sizeof(int), cudaMemcpyDeviceToHost, s));
        NHP_CUDA(ctx, cudaStreamSynchronize(s));
        for (int64_t k = 0; k < K; k++) attempts[k] = h[(size_t)k];
    }
    // commit: the accepted curves replace the context's; the per-event rates rebuild lazily for the new curve version
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_bgrid_v, dcand, (size_t)KG * sizeof(double), cudaMemcpyDeviceToDevice, s));
    k_slice_commit<<<1, 1024, 0, s>>>(a, dout);
    NHP_LAUNCHED(ctx);
    double hout[2];
    NHP_CUDA(ctx, cudaMemcpyAsync(hout, dout, 2 * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    ctx->bgrid_version++;
    ctx->baseline_integral = hout[0];
    ctx->bgrid_min = hout[1];
    ctx->lambda0_min = hout[1];
    ctx->sweep_ll_valid = false; ctx->parents_valid = false;
    const auto t2 = std::chrono::steady_clock::now();
    ctx->slice_info[0] = std::chrono::duration<double, std::milli>(t1 - t0).count();
    ctx->slice_info[1] = std::chrono::duration<double, std::milli>(t2 - t1).count();
    ctx->slice_info[2] = (double)(round + 1);
    ctx->last_ms = ctx->slice_info[0] + ctx->slice_info[1];
    return NHP_OK;
}

// last nhp_cont_resample_baseline: [list build ms, rounds + commit ms, rounds, work items]
extern "C" int nhp_cont_slice_info(const nhp_ctx *ctx, double *out4) {
    if (!ctx || !out4) return NHP_ERR_INVALID;
    for (int i = 0; i < 4; i++) out4[i] = ctx->slice_info[i];
    return NHP_OK;
}
