// cont_sweep.cu -- dense predecessor-window sweeps over the time-sorted event stream:
//   * log-likelihood / per-event total intensity   (continuous.jl:210-239, 286-300, 360-405)
//   * Gibbs parent resampling fused with the counters and impulse statistics
//     (parents.jl:1-46, 61-79; baselines.jl:87-96; impulses.jl:84-96, 230-252)
// One CTA owns a tile of consecutive child events; the union of their dtmax windows is staged
// into shared memory with one cp.async.bulk (TMA) transaction; a group of G lanes walks one
// event's window most-recent-first, exactly the order of the reference loops.
#include "cont_sweep.cuh"
#include <algorithm>
#include <cstdlib>

enum { MODE_LOGLIK = 0, MODE_INTENSITY = 1 };

// ---------------------------------------------------------------------------------------
// window-start prepass: lo(i0) = first j with t[j] > t[i0] - horizon, for i0 = first + 64 b
// ---------------------------------------------------------------------------------------
__global__ void k_tile_lo(const double *__restrict__ t, int64_t first, int64_t n, double horizon, int *__restrict__ tile_lo, int64_t nb,
                          unsigned long long *__restrict__ winstat) {
    int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= nb) return;
    int64_t i0 = first + b * NHP_TQ;
    double thr = t[i0] - horizon;
    int64_t good = i0, bad = -1, step = 64;
    while (true) {  // gallop backwards: windows are short compared with the stream
        int64_t cand = i0 - step;
        if (cand <= 0) {
            if (t[0] > thr) good = 0; else bad = 0;
            break;
        }
        if (t[cand] > thr) { good = cand; step <<= 1; }
        else { bad = cand; break; }
    }
    while (good - bad > 1) {
        int64_t mid = (good + bad) >> 1;
        if (t[mid] > thr) good = mid; else bad = mid;
    }
    if (good > i0) good = i0;
    tile_lo[b] = (int)good;
    unsigned long long w = (unsigned long long)(i0 - good);
    atomicMax(&winstat[0], w);
    atomicAdd(&winstat[1], w);
}

// window length of every own event: i - (first j with t[j] > t[i] - horizon), saturated at 65535.  The windows of
// consecutive events overlap almost completely, so a short backward gallop from the event finds the start.
__global__ void k_win_len(const double *__restrict__ t, int64_t first, int64_t n, double horizon, unsigned short *__restrict__ wlen) {
    int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double thr = t[i] - horizon;
    int64_t good = i, bad = -1, step = 16;
    while (true) {
        int64_t cand = i - step;
        if (cand <= 0) { if (t[0] > thr) good = 0; else bad = 0; break; }
        if (t[cand] > thr) { good = cand; step <<= 1; if (step > 131072) { bad = -2; break; } }
        else { bad = cand; break; }
    }
    if (bad == -2) { wlen[i - first] = 65535; return; }
    while (good - bad > 1) { int64_t mid = (good + bad) >> 1; if (t[mid] > thr) good = mid; else bad = mid; }
    int64_t w = i - good;
    wlen[i - first] = (unsigned short)(w > 65535 ? 65535 : w);
}

int nhp_cont_prepare_windows(nhp_ctx *ctx, nhp_events *ev, double horizon) {
    if (ev->cache_horizon == horizon && ev->d_tile_lo) return NHP_OK;
    int64_t own = ev->n - ev->n_halo;
    int64_t nb = (own + NHP_TQ - 1) / NHP_TQ;
    if (!ev->d_tile_lo) {
        NHP_CUDA(ctx, cudaMallocAsync(&ev->d_tile_lo, (size_t)std::max<int64_t>(nb, 1) * sizeof(int), ctx->stream));
        NHP_CUDA(ctx, cudaMallocAsync(&ev->d_wlen, (size_t)std::max<int64_t>(own, 1) * sizeof(unsigned short), ctx->stream));
        ev->n_bound = nb;
    }
    ev->max_win = 0; ev->mean_win = 0.0;
    if (nb > 0) {
        NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_winstat, 0, 2 * sizeof(int64_t), ctx->stream));
        k_tile_lo<<<(unsigned)((nb + 127) / 128), 128, 0, ctx->stream>>>(ev->d_t, ev->n_halo, ev->n, horizon, ev->d_tile_lo, nb,
                                                                          (unsigned long long *)ctx->d_winstat);
        NHP_LAUNCHED(ctx);
        k_win_len<<<(unsigned)((own + 255) / 256), 256, 0, ctx->stream>>>(ev->d_t, ev->n_halo, ev->n, horizon, ev->d_wlen);
        NHP_LAUNCHED(ctx);
        int64_t ws[2];
        NHP_CUDA(ctx, cudaMemcpyAsync(ws, ctx->d_winstat, sizeof(ws), cudaMemcpyDeviceToHost, ctx->stream));
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        ev->max_win = ws[0];
        ev->mean_win = (double)ws[1] / (double)nb;
    }
    ev->cache_horizon = horizon;
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// log-likelihood / intensity sweep (persistent CTAs looping over tiles of a.te child events)
// ---------------------------------------------------------------------------------------
template <int KIND, int G, int MODE, bool ST>
__device__ __forceinline__ void sweep_body(const SweepArgs &a, const Tile &tl, const FastTables *ft, double &sum_log, double &sum_row) {
    typedef typename EntryOf<KIND>::type E;
    constexpr int NG = NHP_BLOCK / G;
    const int gid = threadIdx.x / G, gl = threadIdx.x % G;
    const unsigned gmask = group_mask<G>();
    const WinView<ST> W(a, tl);
    const int jl_lo = (int)(max(tl.lo, a.jmin) - tl.base);
    const int ib0 = (int)(tl.i0 - tl.base), nev = (int)(tl.i1 - tl.i0);
    for (int ev = gid; ev < nev; ev += NG) {
        const int ib = ib0 + ev;
        const double ti = W.T(ib);
        const int ci = W.C(ib);
        const double thr = ti - a.horizon;
        const E *col = reinterpret_cast<const E *>(a.table) + (size_t)ci * a.K;
        double acc = 0.0;
        for (int jl = ib - 1 - gl; jl >= jl_lo; jl -= G) {
            const double tj = W.T(jl);
            if (!(tj > thr)) break;  // events[parentindex] > time - dtmax   (continuous.jl:291)
            acc += pair_value(load_entry(col + W.C(jl)), ti - tj, a.D, ft);
        }
        acc = group_sum<G>(acc, gmask);
        if (gl == 0) {
            const double lam = base_rate(a, tl.i0 + ev, ci) + acc;
            if (MODE == MODE_INTENSITY) a.lam_out[tl.i0 + ev - a.first] = lam;
            else { sum_log += log(lam); sum_row += __ldg(a.rowsum + ci); }
        }
    }
}

template <int KIND, int G, int MODE>
__global__ void __launch_bounds__(NHP_BLOCK) k_sweep(const SweepArgs a, const int64_t ntiles) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ double red[16];
    __shared__ FastTables s_ft;
    fast_tables_load(&s_ft);
    Stager sg = stager_init(a, smem);
    __syncthreads();
    double sum_log = 0.0, sum_row = 0.0;
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        Tile tl = stage_tile_at(a, sg, tile);
        if (tl.staged) sweep_body<KIND, G, MODE, true>(a, tl, &s_ft, sum_log, sum_row);
        else sweep_body<KIND, G, MODE, false>(a, tl, &s_ft, sum_log, sum_row);
        __syncthreads();  // the staging buffers are refilled by the next tile
    }
    if (MODE == MODE_LOGLIK) {
        block_sum2(sum_log, sum_row, red);
        if (threadIdx.x == 0) { a.partials[2 * (size_t)blockIdx.x] = sum_log; a.partials[2 * (size_t)blockIdx.x + 1] = sum_row; }
    }
}

// fixed-order second-stage reduction of the per-CTA partials -> out[0], out[1].  When Mn is given the sweep did not
// accumulate the compensator term per event and out[1] = sum_c Mn[c] * rowsum[c] (= sum_i rowsum[c_i] over the own events).
__global__ void k_reduce_partials(const double *__restrict__ partials, int64_t nblocks, double *__restrict__ out,
                                  const double *__restrict__ Mn, const double *__restrict__ rowsum, int K) {
    __shared__ double sx[1024], sy[1024];
    double x = 0.0, y = 0.0;
    for (int64_t b = threadIdx.x; b < nblocks; b += blockDim.x) { x += partials[2 * b]; y += partials[2 * b + 1]; }
    if (Mn) {
        y = 0.0;
        for (int c = threadIdx.x; c < K; c += blockDim.x) y += Mn[c] * rowsum[c];
    }
    sx[threadIdx.x] = x; sy[threadIdx.x] = y;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) { sx[threadIdx.x] += sx[threadIdx.x + s]; sy[threadIdx.x] += sy[threadIdx.x + s]; }
        __syncthreads();
    }
    if (threadIdx.x == 0) { out[0] = sx[0]; out[1] = sy[0]; }
}

// ---------------------------------------------------------------------------------------
// Gibbs parent sweep (parents.jl:25-46): weights most-recent-first then the baseline,
// one uniform per event, inverse-cdf walk in that order; fused statistics.
// ---------------------------------------------------------------------------------------
template <int KIND, int G, int R, bool ST>
__device__ __forceinline__ void parents_body(const SweepArgs &a, const Tile &tl, const FastTables *ft, int *m0_hist, double *s_v, double &sum_log, double &sum_row) {
    typedef typename EntryOf<KIND>::type E;
    constexpr int NG = NHP_BLOCK / G;
    const int gid = threadIdx.x / G, gl = threadIdx.x % G;
    const unsigned gmask = group_mask<G>();
    const int gshift = (threadIdx.x & 31) / G * G;
    const unsigned gbits = G == 32 ? 0xffffffffu : ((1u << G) - 1u);
    const WinView<ST> W(a, tl);
    const int jl_lo = (int)(max(tl.lo, a.jmin) - tl.base);
    const int ib0 = (int)(tl.i0 - tl.base), nev = (int)(tl.i1 - tl.i0);
    const StatsLayout sl{a.K};
    double *my_v = s_v + threadIdx.x;  // this lane's cached weights: row r at my_v[r * NHP_BLOCK] (conflict-free)
    for (int ev = gid; ev < nev; ev += NG) {
        const int ib = ib0 + ev;
        const int64_t i = tl.i0 + ev;
        const double ti = W.T(ib);
        const int ci = W.C(ib);
        const double thr = ti - a.horizon;
        const E *col = reinterpret_cast<const E *>(a.table) + (size_t)ci * a.K;
        // pass 1: window weights, most recent first; the first R rows (G entries each) are kept in shared memory
        double acc = 0.0;
        int nr = 0;  // rows in which this lane has an in-window entry
        for (int jl = ib - 1 - gl; jl >= jl_lo; jl -= G, nr++) {
            const double tj = W.T(jl);
            if (!(tj > thr)) break;  // events[parentindex] > time - dtmax   (parents.jl:32)
            const double v = pair_value(load_entry(col + W.C(jl)), ti - tj, a.D, ft);
            acc += v;
            if (nr < R) my_v[nr * NHP_BLOCK] = v;
        }
        const double lam0 = base_rate(a, i, ci);
        const double S = group_sum<G>(acc, gmask) + lam0;  // sum([weights...; baseline])
        const int64_t gi = a.index_base + i;
        const double u = a.u ? __ldg(a.u + (i - a.first)) : philox_uniform(a.seed, (uint64_t)gi, a.counter);
        const double target = u * S;
        // pass 2: first k with cumulative weight > u * S   (cp <= draw keeps walking); lane 0 owns the most
        // recent entry of every row, so its row count bounds the walk
        const int nrows = (gi == 0) ? 0 : __shfl_sync(gmask, nr, 0, G);  // index == 1 && return 0, 0   (parents.jl:26-28)
        int chosen = 0;  // i - j of the chosen parent, 0 = baseline
        double carry = 0.0;
        for (int r = 0; r < nrows; r++) {
            double v = 0.0;
            if (r < nr) {
                if (r < R) v = my_v[r * NHP_BLOCK];
                else {
                    const int jj = ib - 1 - gl - r * G;
                    v = pair_value(load_entry(col + W.C(jj)), ti - W.T(jj), a.D, ft);
                }
            }
            const double x = group_incl_scan<G>(v, gmask, gl);
            const unsigned b = (__ballot_sync(gmask, carry + x > target) >> gshift) & gbits;
            if (b) { chosen = r * G + (__ffs(b) - 1) + 1; break; }
            carry += __shfl_sync(gmask, x, G - 1, G);
        }
        if (gl == 0) {
            if (!(S > 0.0) || S > 1.7976931348623157e308) atomicOr(a.flag, 8);  // Categorical would reject the vector
            // S is the event's total intensity: the log-likelihood terms come for free with the sweep
            if (a.want_ll) { sum_log += log(S); sum_row += __ldg(a.rowsum + ci); }
            a.poff[i] = chosen;
            if (chosen == 0) {
                if (m0_hist) atomicAdd(m0_hist + ci, 1);
                else red_add_f64(a.stats + sl.off_M0() + ci, 1.0);
            } else {
                const int jp = ib - chosen;
                const int cj = W.C(jp);
                const double dt = ti - W.T(jp);
                const int64_t k = cj + (int64_t)a.K * ci;
                red_add_f64(a.stats + sl.off_Mnm() + k, 1.0);
                red_add_f64(a.stats + sl.off_S1() + k, KIND == NHP_LOGITNORMAL ? log_duration_dev(dt, a.D) : dt);
            }
        }
    }
}

template <int KIND, int G, int R>
__global__ void __launch_bounds__(NHP_BLOCK) k_parents(const SweepArgs a, const int64_t ntiles, const int m0_smem) {
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ FastTables s_ft;
    __shared__ double s_v[R * NHP_BLOCK];  // cached window weights of pass 1
    __shared__ double red[16];
    double sum_log = 0.0, sum_row = 0.0;
    fast_tables_load(&s_ft);
    Stager sg = stager_init(a, smem);
    // baseline-attribution histogram in shared memory behind the staging area (most events are baseline events)
    int *m0_hist = m0_smem ? reinterpret_cast<int *>(smem + ((16 + (size_t)a.cap * 12 + 15) & ~(size_t)15)) : nullptr;
    if (m0_hist) for (int k = threadIdx.x; k < a.K; k += NHP_BLOCK) m0_hist[k] = 0;
    __syncthreads();
    for (int64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x) {
        Tile tl = stage_tile_at(a, sg, tile);
        if (tl.staged) parents_body<KIND, G, R, true>(a, tl, &s_ft, m0_hist, s_v, sum_log, sum_row);
        else parents_body<KIND, G, R, false>(a, tl, &s_ft, m0_hist, s_v, sum_log, sum_row);
        __syncthreads();
    }
    block_sum2(sum_log, sum_row, red);
    if (threadIdx.x == 0) { a.partials[2 * (size_t)blockIdx.x] = sum_log; a.partials[2 * (size_t)blockIdx.x + 1] = sum_row; }
    if (m0_hist) {
        const StatsLayout sl{a.K};
        for (int k = threadIdx.x; k < a.K; k += NHP_BLOCK)
            if (m0_hist[k]) red_add_f64(a.stats + sl.off_M0() + k, (double)m0_hist[k]);
    }
}

// ---------------------------------------------------------------------------------------
// statistics helpers
// ---------------------------------------------------------------------------------------
__global__ void k_xbar(const double *__restrict__ Mnm, const double *__restrict__ S1, double *__restrict__ xbar, int64_t KK) {
    int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < KK) xbar[k] = S1[k] / Mnm[k];  // NaN where no pair was observed (impulses.jl:222-223)
}

// log_duration_variation (impulses.jl:242-252): second pass around the per-pair mean
__global__ void k_second_pass(const double *__restrict__ t, const int *__restrict__ c, const int *__restrict__ poff, int64_t first, int64_t n,
                              int K, double D, const double *__restrict__ xbar, double *__restrict__ S2) {
    int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int off = poff[i];
    if (off <= 0) return;
    int64_t j = i - off;
    int64_t k = c[j] + (int64_t)K * c[i];
    double d = log_duration_dev(t[i] - t[j], D) - xbar[k];
    red_add_f64(S2 + k, d * d);
}

// counters + first-pass statistics from a stored parent assignment
template <int KIND>
__global__ void k_stats_from_parents(const double *__restrict__ t, const int *__restrict__ c, const int *__restrict__ poff, int64_t first,
                                     int64_t n, int K, double D, double *__restrict__ stats) {
    int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    StatsLayout sl{K};
    int off = poff[i];
    if (off == 0) red_add_f64(stats + sl.off_M0() + c[i], 1.0);
    else if (off > 0) {
        int64_t j = i - off;
        int64_t k = c[j] + (int64_t)K * c[i];
        double dt = t[i] - t[j];
        red_add_f64(stats + sl.off_Mnm() + k, 1.0);
        red_add_f64(stats + sl.off_S1() + k, KIND == NHP_LOGITNORMAL ? log_duration_dev(dt, D) : dt);
    }
}

__global__ void k_export_parents(const int *__restrict__ c, const int *__restrict__ poff, int64_t first, int64_t n, int64_t index_base,
                                 int64_t *__restrict__ parents, int64_t *__restrict__ parentnodes) {
    int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int off = poff[i];
    int64_t j = i - off;
    if (parents) parents[i - first] = off > 0 ? index_base + j + 1 : 0;
    if (parentnodes) parentnodes[i - first] = off > 0 ? (int64_t)c[j] + 1 : 0;
}

__global__ void k_import_parents(const int64_t *__restrict__ parents, int64_t first, int64_t n, int64_t index_base, int *__restrict__ poff,
                                 int *__restrict__ flag) {
    int64_t i = first + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    int64_t p = parents[i - first];
    if (p == 0) { poff[i] = 0; return; }
    int64_t j = p - 1 - index_base;  // local index of the parent
    if (j < 0 || j >= i) { atomicOr(flag, 16); poff[i] = 0; return; }
    poff[i] = (int)(i - j);
}

// ---------------------------------------------------------------------------------------
// host-side dispatch
// ---------------------------------------------------------------------------------------
static int pick_group(const nhp_events *ev) {
    const char *env = getenv("NHP_G");
    if (env) {
        int g = atoi(env);
        if (g == 1 || g == 2 || g == 4 || g == 8 || g == 16 || g == 32) return g;
    }
    double w = ev->mean_win;
    int64_t own = ev->n - ev->n_halo;
    if (own < 200000) return w < 8 ? 8 : 32;  // small streams: spread each event over more lanes to fill the chip
    if (w < 3) return 1;
    if (w < 6) return 2;
    if (w < 12) return 4;
    if (w < 160) return 8;
    if (w < 640) return 16;
    return 32;
}

struct LaunchPlan { int G, te, cap, grid; size_t smem; int64_t tiles; };

static LaunchPlan make_plan(nhp_ctx *ctx, const nhp_events *ev) {
    LaunchPlan p;
    p.G = pick_group(ev);
    int64_t own = ev->n - ev->n_halo;
    p.te = 256;
    if (p.G == 32 && own < 200000) p.te = 64;
    p.tiles = (own + p.te - 1) / p.te;
    int64_t need = ((ev->max_win + p.te + 8) + 3) & ~(int64_t)3;
    int64_t limit = ((int64_t)ctx->smem_optin - 1024 - 16) / 12;
    limit &= ~(int64_t)3;
    int64_t soft = 8192;  // keep several CTAs per SM resident; larger ranges fall back to L1/L2 reads
    p.cap = (int)std::min(need, std::min(limit, soft));
    p.smem = 16 + (size_t)p.cap * 12;
    return p;
}

// persistent launch: one resident wave of CTAs looping over the tiles
template <typename KernelT, typename... Extra>
static int launch_persistent(nhp_ctx *ctx, KernelT kernel, LaunchPlan &p, size_t smem, const SweepArgs &a, Extra... extra) {
    NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));  // always: static + dynamic may exceed the 48 KB default even when the dynamic part is small
    NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    int per_sm = 1;
    NHP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, NHP_BLOCK, smem));
    p.grid = (int)std::min<int64_t>(p.tiles, (int64_t)ctx->sm_count * std::max(per_sm, 1));
    kernel<<<p.grid, NHP_BLOCK, smem, ctx->stream>>>(a, p.tiles, extra...);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

template <int KIND, int MODE> static int dispatch_sweep(nhp_ctx *ctx, LaunchPlan &p, const SweepArgs &a) {
    switch (p.G) {
        case 1: return launch_persistent(ctx, k_sweep<KIND, 1, MODE>, p, p.smem, a);
        case 2: return launch_persistent(ctx, k_sweep<KIND, 2, MODE>, p, p.smem, a);
        case 4: return launch_persistent(ctx, k_sweep<KIND, 4, MODE>, p, p.smem, a);
        case 8: return launch_persistent(ctx, k_sweep<KIND, 8, MODE>, p, p.smem, a);
        case 16: return launch_persistent(ctx, k_sweep<KIND, 16, MODE>, p, p.smem, a);
        default: return launch_persistent(ctx, k_sweep<KIND, 32, MODE>, p, p.smem, a);
    }
}

template <int KIND> static int dispatch_parents(nhp_ctx *ctx, LaunchPlan &p, const SweepArgs &a) {
    const int m0 = a.K <= 8192 ? 1 : 0;
    const size_t smem = m0 ? ((p.smem + 15) & ~(size_t)15) + (size_t)a.K * sizeof(int) : p.smem;
    switch (p.G) {
        case 1: return launch_persistent(ctx, k_parents<KIND, 1, 16>, p, smem, a, m0);
        case 2: return launch_persistent(ctx, k_parents<KIND, 2, 16>, p, smem, a, m0);
        case 4: return launch_persistent(ctx, k_parents<KIND, 4, 16>, p, smem, a, m0);
        case 8: return launch_persistent(ctx, k_parents<KIND, 8, 16>, p, smem, a, m0);
        case 16: return launch_persistent(ctx, k_parents<KIND, 16, 8>, p, smem, a, m0);
        default: return launch_persistent(ctx, k_parents<KIND, 32, 8>, p, smem, a, m0);
    }
}

// Look-back horizon.  LogitNormal: dtmax.  Exponential: dtmax, shortened to the cut-off beyond
// which the omitted tail is < 1e-14 of the smallest baseline rate: every omitted term is at most
// wt_max exp(-theta_min H) and an event has fewer than n_total predecessors.
double nhp_cont_horizon_value(const nhp_ctx *ctx, int64_t n_total, int recursive) {
    double h = ctx->dtmax;
    if (ctx->kind != NHP_EXPONENTIAL) return h;
    if (recursive) h = INFINITY;  // recursive_loglikelihood ignores dtmax (quirk Q7)
    if (ctx->wt_max <= 0.0) return std::min(h, 0.0 + 1e-300);  // no active pair: any horizon gives zero impulse mass
    if (ctx->theta_min > 0.0 && std::isfinite(ctx->theta_min) && ctx->lambda0_min > 0.0 && n_total > 0) {
        double cut = log((double)n_total * ctx->wt_max / (1e-14 * ctx->lambda0_min)) / ctx->theta_min;
        if (cut > 0.0 && cut < h) h = cut;
    }
    return h;
}

extern "C" int nhp_cont_horizon(nhp_ctx *ctx, int64_t n_total, int recursive, double *horizon) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CHECK(ctx, horizon != nullptr, NHP_ERR_INVALID, "nhp_cont_horizon: horizon is NULL");
    *horizon = nhp_cont_horizon_value(ctx, n_total, recursive && ctx->kind == NHP_EXPONENTIAL);
    return NHP_OK;
}

static int fill_args(nhp_ctx *ctx, nhp_events *ev, int recursive, SweepArgs &a, LaunchPlan &p) {
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set (call nhp_cont_params_set)");
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "events handle is NULL");
    NHP_CHECK(ctx, ev->K == ctx->K, NHP_ERR_INVALID, "events were uploaded with K=%lld but parameters have K=%lld", (long long)ev->K, (long long)ctx->K);
    bool rec = recursive && ctx->kind == NHP_EXPONENTIAL;
    double horizon = nhp_cont_horizon_value(ctx, ev->index_base + ev->n, rec);
    NHP_TRY(nhp_cont_prepare_windows(ctx, ev, horizon));
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    p = make_plan(ctx, ev);
    a.t = ev->d_t; a.c = ev->d_c; a.n = ev->n; a.first = ev->n_halo; a.index_base = ev->index_base;
    a.jmin = rec ? ev->n_t0 : 0;
    a.tile_lo = ev->d_tile_lo; a.te = p.te; a.cap = p.cap; a.K = (int)ctx->K;
    a.table = ctx->d_table; a.lambda0 = ctx->d_lambda0;
    NHP_TRY(nhp_cont_event_baseline(ctx, ev, &a.lam0ev));
    a.rowsum = (rec && ctx->has_A) ? ctx->d_rowsum_w : ctx->d_rowsum;  // quirk Q3
    a.D = ctx->dtmax; a.horizon = horizon;
    a.partials = nullptr; a.lam_out = nullptr; a.poff = ev->d_poff; a.u = nullptr; a.seed = 0; a.counter = 0;
    a.stats = ctx->d_stats0; a.flag = ctx->d_flag; a.want_ll = ctx->opt_sweep_ll ? 1 : 0;
    return NHP_OK;
}

int nhp_cont_try_sparse(nhp_ctx *ctx, const nhp_events *ev, SweepArgs &a, int mode, int *grid_out);  // cont_sparse.cu
int nhp_cont_try_child(nhp_ctx *ctx, nhp_events *ev, SweepArgs &a, int mode, int *grid_out);          // cont_child.cu
int nhp_cont_try_exp_scan(nhp_ctx *ctx, nhp_events *ev, SweepArgs &a, int *grid_out);                  // cont_exp_scan.cu

// sparse-adjacency sweep if it applies, else the child-major sweep for large tables; 1 = neither (time-tiled dense sweep)
static int try_special(nhp_ctx *ctx, nhp_events *ev, SweepArgs &a, int mode, int *grid_out) {
    int sp = nhp_cont_try_sparse(ctx, ev, a, mode, grid_out);
    if (sp != 1) return sp;
    return nhp_cont_try_child(ctx, ev, a, mode, grid_out);
}

// leaves (log-sum, row-sum) in stats0[0..1]; no host synchronisation
int nhp_cont_run_loglik(nhp_ctx *ctx, nhp_events *ev, int recursive) {
    SweepArgs a; LaunchPlan p;
    NHP_TRY(fill_args(ctx, ev, recursive, a, p));
    if (p.tiles == 0) { NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats0, 0, 2 * sizeof(double), ctx->stream)); return NHP_OK; }
    NHP_TRY(nhp_partials(ctx, 2 * (int64_t)ctx->sm_count * 32, &a.partials));  // one partial per persistent CTA
    int sgrid = 0;
    // recursive Exponential on unsharded data: the chunked scan when it beats the cut-off window (cont_exp_scan.cu)
    int sp = (recursive && ctx->kind == NHP_EXPONENTIAL) ? nhp_cont_try_exp_scan(ctx, ev, a, &sgrid) : 1;
    if (sp == 1 && !recursive) sp = nhp_cont_try_adj_loglik(ctx, ev, a, &sgrid);  // sparse network with a cached pair structure: active buckets only
    if (sp == 1) sp = try_special(ctx, ev, a, 0, &sgrid);
    if (sp < 0) return sp;
    if (sp == NHP_OK) p.grid = sgrid;
    else if (ctx->kind == NHP_LOGITNORMAL) NHP_TRY((dispatch_sweep<NHP_LOGITNORMAL, MODE_LOGLIK>(ctx, p, a)));
    else NHP_TRY((dispatch_sweep<NHP_EXPONENTIAL, MODE_LOGLIK>(ctx, p, a)));
    k_reduce_partials<<<1, 1024, 0, ctx->stream>>>(a.partials, p.grid, ctx->d_stats0, ev->d_Mn, a.rowsum, (int)ctx->K);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

// Log-likelihood share of this rank in a multi-GPU job (sum over ranks = ll).  When the replicated stream `ev_full` carries this
// rank's part of the adjacency structure (the columns c = rank mod nranks, built by the first adjacency sweep) the share is taken from
// it -- sum log lambda over the events on the rank's columns, active buckets only; rank 0 adds the baseline and compensator terms.
// Otherwise (no structure yet, dense network, recursive semantics) it is the time shard's share as in nhp_cont_loglik(ev_shard).
extern "C" int nhp_cont_loglik_dist(nhp_ctx *ctx, nhp_events *ev_shard, nhp_events *ev_full, int recursive, double *share) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev_shard != nullptr && share != nullptr, NHP_ERR_INVALID, "nhp_cont_loglik_dist: NULL argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (ev_full && !recursive && ctx->nranks > 1 && ev_full->d_adj_i && ev_full->adj_cb == ctx->rank && ev_full->adj_cs == ctx->nranks) {
        SweepArgs a; LaunchPlan p;
        NHP_TRY(fill_args(ctx, ev_full, 0, a, p));
        if (p.tiles > 0) {
            NHP_TRY(nhp_partials(ctx, 2 * (int64_t)ctx->sm_count * 32, &a.partials));
            NHP_TRY(nhp_timer_begin(ctx));
            int sgrid = 0;
            const int sp = nhp_cont_try_adj_loglik(ctx, ev_full, a, &sgrid, ctx->rank, ctx->nranks);
            if (sp < 0) return sp;
            if (sp == NHP_OK) {
                k_reduce_partials<<<1, 1024, 0, ctx->stream>>>(a.partials, sgrid, ctx->d_stats0, ev_full->d_Mn, a.rowsum, (int)ctx->K);
                NHP_LAUNCHED(ctx);
                double h[2];
                NHP_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_stats0, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
                NHP_TRY(nhp_timer_end(ctx));
                *share = h[0] - (ctx->rank == 0 ? nhp_cont_baseline_term(ctx, ev_full) + h[1] : 0.0);
                return NHP_OK;
            }
            NHP_TRY(nhp_timer_end(ctx));
        }
    }
    return nhp_cont_loglik(ctx, ev_shard, recursive, share);
}

extern "C" int nhp_cont_loglik_dev(nhp_ctx *ctx, nhp_events *ev, int recursive) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    return nhp_cont_run_loglik(ctx, ev, recursive);
}

extern "C" int nhp_cont_loglik(nhp_ctx *ctx, nhp_events *ev, int recursive, double *ll) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ll != nullptr, NHP_ERR_INVALID, "nhp_cont_loglik: ll is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_TRY(nhp_timer_begin(ctx));
    NHP_TRY(nhp_cont_run_loglik(ctx, ev, recursive));
    double h[2];
    NHP_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_stats0, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_TRY(nhp_timer_end(ctx));
    double base = nhp_cont_baseline_term(ctx, ev);  // sum(integrated_intensity(baseline, duration))
    // ll = -sum_k lambda0_k T - sum_i rowsum(c_i) + sum_i log lambda_i   (continuous.jl:217-238)
    *ll = (0.0 - base) - h[1] + h[0];
    return NHP_OK;
}

// total intensity at every own event into a device buffer (no host synchronisation); shared with the gradient sweep
int nhp_cont_run_event_intensity(nhp_ctx *ctx, nhp_events *ev, int recursive, double *d_out) {
    SweepArgs a; LaunchPlan p;
    NHP_TRY(fill_args(ctx, ev, recursive, a, p));
    if (ev->n - ev->n_halo == 0) return NHP_OK;
    a.lam_out = d_out;
    int sgrid = 0;
    int sp = try_special(ctx, ev, a, 1, &sgrid);
    if (sp < 0) return sp;
    if (sp == NHP_OK) {}
    else if (ctx->kind == NHP_LOGITNORMAL) NHP_TRY((dispatch_sweep<NHP_LOGITNORMAL, MODE_INTENSITY>(ctx, p, a)));
    else NHP_TRY((dispatch_sweep<NHP_EXPONENTIAL, MODE_INTENSITY>(ctx, p, a)));
    return NHP_OK;
}

int nhp_cont_fill_args(nhp_ctx *ctx, nhp_events *ev, int recursive, SweepArgs &a) {
    LaunchPlan p;
    return fill_args(ctx, ev, recursive, a, p);
}

// (sum log lambda, compensator) -> stats0[0..1] from the per-CTA partials of any sweep
int nhp_cont_reduce_partials(nhp_ctx *ctx, nhp_events *ev, const double *partials, int grid, const double *rowsum) {
    k_reduce_partials<<<1, 1024, 0, ctx->stream>>>(partials, grid, ctx->d_stats0, ev->d_Mn, rowsum, (int)ctx->K);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

extern "C" int nhp_cont_event_intensity(nhp_ctx *ctx, nhp_events *ev, double *out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, out != nullptr, NHP_ERR_INVALID, "nhp_cont_event_intensity: out is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "events handle is NULL");
    int64_t own = ev->n - ev->n_halo;
    void *scratch = nullptr;
    if (own > 0) NHP_TRY(nhp_scratch(ctx, (size_t)own * sizeof(double), &scratch));
    NHP_TRY(nhp_timer_begin(ctx));
    NHP_TRY(nhp_cont_run_event_intensity(ctx, ev, 0, (double *)scratch));
    NHP_TRY(nhp_timer_end(ctx));
    if (own == 0) return NHP_OK;
    NHP_CUDA(ctx, cudaMemcpyAsync(out, scratch, (size_t)own * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

// ---- parents + statistics -----------------------------------------------------------------
static int zero_stats(nhp_ctx *ctx, nhp_events *ev) {
    StatsLayout sl{ctx->K};
    ctx->grad_valid = false;  // the gradient planes share these buffers
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats0 + sl.off_M0(), 0, (size_t)(sl.total() - sl.off_M0()) * sizeof(double), ctx->stream));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_stats0 + sl.off_Mn(), ev->d_Mn, (size_t)ctx->K * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats1, 0, (size_t)(ctx->K * ctx->K) * sizeof(double), ctx->stream));
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), ctx->stream));
    return NHP_OK;
}

static int export_parents(nhp_ctx *ctx, nhp_events *ev, int64_t *parents, int64_t *parentnodes) {
    int64_t own = ev->n - ev->n_halo;
    if (own == 0 || (!parents && !parentnodes)) return NHP_OK;
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)own * 2 * sizeof(int64_t), &scratch));
    int64_t *dp = (int64_t *)scratch, *dn = dp + own;
    k_export_parents<<<(unsigned)((own + 255) / 256), 256, 0, ctx->stream>>>(ev->d_c, ev->d_poff, ev->n_halo, ev->n, ev->index_base, dp, dn);
    NHP_LAUNCHED(ctx);
    if (parents) NHP_CUDA(ctx, cudaMemcpyAsync(parents, dp, (size_t)own * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    if (parentnodes) NHP_CUDA(ctx, cudaMemcpyAsync(parentnodes, dn, (size_t)own * sizeof(int64_t), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

extern "C" int nhp_cont_resample_parents(nhp_ctx *ctx, nhp_events *ev, uint64_t seed, uint64_t counter, const double *u, int64_t *parents,
                                         int64_t *parentnodes) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    SweepArgs a; LaunchPlan p;
    NHP_TRY(fill_args(ctx, ev, 0, a, p));
    int64_t own = ev->n - ev->n_halo;
    ctx->parents_valid = false;
    ctx->sweep_ll_valid = false;
    NHP_TRY(zero_stats(ctx, ev));
    double *du = nullptr;
    if (u && own > 0) {
        // uniforms live behind the export scratch area
        void *scratch;
        NHP_TRY(nhp_scratch(ctx, (size_t)own * 3 * sizeof(int64_t), &scratch));
        du = (double *)scratch + 2 * own;
        NHP_CUDA(ctx, cudaMemcpyAsync(du, u, (size_t)own * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    a.u = du; a.seed = seed; a.counter = counter;
    NHP_TRY(nhp_partials(ctx, 2 * (int64_t)ctx->sm_count * 32, &a.partials));  // one partial per persistent CTA
    NHP_TRY(nhp_timer_begin(ctx));
    if (p.tiles > 0) {
        int sgrid = 0;
        int sp = try_special(ctx, ev, a, 2, &sgrid);
        if (sp < 0) return sp;
        if (sp == NHP_OK) p.grid = sgrid;
        else if (ctx->kind == NHP_LOGITNORMAL) NHP_TRY(dispatch_parents<NHP_LOGITNORMAL>(ctx, p, a));
        else NHP_TRY(dispatch_parents<NHP_EXPONENTIAL>(ctx, p, a));
        // the sweep also produced the log-likelihood terms (sum log lambda_i, sum rowsum): stats0[0..1]
        k_reduce_partials<<<1, 1024, 0, ctx->stream>>>(a.partials, p.grid, ctx->d_stats0, ev->d_Mn, a.rowsum, (int)ctx->K);
        NHP_LAUNCHED(ctx);
    } else NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats0, 0, 2 * sizeof(double), ctx->stream));
    int flag = 0;
    NHP_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_TRY(nhp_timer_end(ctx));
    NHP_CHECK(ctx, !(flag & 8), NHP_ERR_NUMERIC, "resample_parents: non-positive or non-finite total intensity (Categorical would throw, parents.jl:42)");
    ctx->parents_valid = true;
    ctx->sweep_ll_valid = ctx->opt_sweep_ll;
    return export_parents(ctx, ev, parents, parentnodes);
}

// (parents, parentnodes) of the assignment the device currently holds (the last sweep, or nhp_cont_parents_set), in the reference's format
extern "C" int nhp_cont_parents_get(nhp_ctx *ctx, nhp_events *ev, int64_t *parents, int64_t *parentnodes) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev != nullptr, NHP_ERR_INVALID, "nhp_cont_parents_get: events handle is NULL");
    NHP_CHECK(ctx, ctx->parents_valid, NHP_ERR_STATE, "nhp_cont_parents_get: no parent assignment (call nhp_cont_resample_parents or nhp_cont_parents_set)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    return export_parents(ctx, ev, parents, parentnodes);
}

// log-likelihood of the parameters used by the most recent parent sweep, from the terms that sweep accumulated
extern "C" int nhp_cont_sweep_loglik(nhp_ctx *ctx, nhp_events *ev, double *ll) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ev && ll, NHP_ERR_INVALID, "nhp_cont_sweep_loglik: NULL argument");
    NHP_CHECK(ctx, ctx->parents_valid && ctx->sweep_ll_valid, NHP_ERR_STATE,
              "nhp_cont_sweep_loglik: enable NHP_OPT_SWEEP_LOGLIK (nhp_set_option) and run nhp_cont_resample_parents with the current parameters first");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    double h[2];
    NHP_CUDA(ctx, cudaMemcpyAsync(h, ctx->d_stats0, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    double base = nhp_cont_baseline_term(ctx, ev);
    *ll = (0.0 - base) - h[1] + h[0];
    return NHP_OK;
}

extern "C" int nhp_cont_parents_set(nhp_ctx *ctx, nhp_events *ev, const int64_t *parents) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CHECK(ctx, ev && parents, NHP_ERR_INVALID, "nhp_cont_parents_set: NULL argument");
    NHP_CHECK(ctx, ev->K == ctx->K, NHP_ERR_INVALID, "events/parameter K mismatch");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t own = ev->n - ev->n_halo;
    ctx->parents_valid = false;
    ctx->sweep_ll_valid = false;
    NHP_TRY(zero_stats(ctx, ev));
    if (own > 0) {
        void *scratch;
        NHP_TRY(nhp_scratch(ctx, (size_t)own * sizeof(int64_t), &scratch));
        NHP_CUDA(ctx, cudaMemcpyAsync(scratch, parents, (size_t)own * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
        unsigned blocks = (unsigned)((own + 255) / 256);
        k_import_parents<<<blocks, 256, 0, ctx->stream>>>((const int64_t *)scratch, ev->n_halo, ev->n, ev->index_base, ev->d_poff, ctx->d_flag);
        NHP_LAUNCHED(ctx);
        if (ctx->kind == NHP_LOGITNORMAL)
            k_stats_from_parents<NHP_LOGITNORMAL><<<blocks, 256, 0, ctx->stream>>>(ev->d_t, ev->d_c, ev->d_poff, ev->n_halo, ev->n, (int)ctx->K, ctx->dtmax, ctx->d_stats0);
        else
            k_stats_from_parents<NHP_EXPONENTIAL><<<blocks, 256, 0, ctx->stream>>>(ev->d_t, ev->d_c, ev->d_poff, ev->n_halo, ev->n, (int)ctx->K, ctx->dtmax, ctx->d_stats0);
        NHP_LAUNCHED(ctx);
    }
    int flag = 0;
    NHP_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    NHP_CHECK(ctx, !(flag & 16), NHP_ERR_INVALID, "nhp_cont_parents_set: a parent index is not an earlier event of this handle");
    ctx->parents_valid = true;
    return NHP_OK;
}

extern "C" int nhp_cont_suffstats_second_pass(nhp_ctx *ctx, nhp_events *ev) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->parents_valid, NHP_ERR_STATE, "no parent assignment (call nhp_cont_resample_parents or nhp_cont_parents_set)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    int64_t KK = ctx->K * ctx->K;
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_stats1, 0, (size_t)KK * sizeof(double), ctx->stream));
    if (ctx->kind != NHP_LOGITNORMAL) return NHP_OK;
    StatsLayout sl{ctx->K};
    k_xbar<<<(unsigned)((KK + 255) / 256), 256, 0, ctx->stream>>>(ctx->d_stats0 + sl.off_Mnm(), ctx->d_stats0 + sl.off_S1(), ctx->d_xbar, KK);
    NHP_LAUNCHED(ctx);
    int64_t own = ev->n - ev->n_halo;
    if (own > 0) {
        k_second_pass<<<(unsigned)((own + 255) / 256), 256, 0, ctx->stream>>>(ev->d_t, ev->d_c, ev->d_poff, ev->n_halo, ev->n, (int)ctx->K, ctx->dtmax, ctx->d_xbar, ctx->d_stats1);
        NHP_LAUNCHED(ctx);
    }
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

extern "C" int nhp_cont_suffstats_read(nhp_ctx *ctx, double *M0, double *Mn, double *Mnm, double *S1, double *S2) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    StatsLayout sl{ctx->K};
    int64_t K = ctx->K, KK = K * K;
    cudaStream_t s = ctx->stream;
    if (M0) NHP_CUDA(ctx, cudaMemcpyAsync(M0, ctx->d_stats0 + sl.off_M0(), (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (Mn) NHP_CUDA(ctx, cudaMemcpyAsync(Mn, ctx->d_stats0 + sl.off_Mn(), (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (Mnm) NHP_CUDA(ctx, cudaMemcpyAsync(Mnm, ctx->d_stats0 + sl.off_Mnm(), (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (S1) NHP_CUDA(ctx, cudaMemcpyAsync(S1, ctx->d_stats0 + sl.off_S1(), (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (S2) NHP_CUDA(ctx, cudaMemcpyAsync(S2, ctx->d_stats1, (size_t)KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

extern "C" int nhp_cont_suffstats(nhp_ctx *ctx, nhp_events *ev, double *M0, double *Mn, double *Mnm, double *S1, double *S2) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    if (S2) NHP_TRY(nhp_cont_suffstats_second_pass(ctx, ev));
    else NHP_CHECK(ctx, ctx->parents_valid, NHP_ERR_STATE, "no parent assignment");
    return nhp_cont_suffstats_read(ctx, M0, Mn, Mnm, S1, S2);
}

extern "C" int nhp_cont_stats_dev(nhp_ctx *ctx, int phase, void **ptr_dev, int64_t *count) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set");
    NHP_CHECK(ctx, ptr_dev && count, NHP_ERR_INVALID, "nhp_cont_stats_dev: NULL output");
    StatsLayout sl{ctx->K};
    if (phase == 0) { *ptr_dev = ctx->d_stats0; *count = sl.total(); }
    else { *ptr_dev = ctx->d_stats1; *count = ctx->K * ctx->K; }
    return NHP_OK;
}
