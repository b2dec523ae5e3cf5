// cont_adjacency.cu -- resample_adjacency_matrix!(process, data)  (continuous.jl:444-519).
//
// The reference evaluates, for every (p, c), two full passes over all N events (2 K^2 N work).  The
// conditional it samples from only depends on the child events on c whose window holds an event of
// node p:  with G_i[p] = W[p,c] sum_{j in win(i), c_j = p} h_pc(t_i - t_j)  and
// lambda_i = lambda0_c(t_i) + sum_p A[p,c] G_i[p]  (lambda0_c(t_i) = lambda0_c for a homogeneous baseline),
//     ll1 - ll0 = -W[p,c] n_p + sum_{i on c, G_i[p] > 0} [ log(lambda_i^{-p} + G_i[p]) - log(lambda_i^{-p}) ]
//                 + log rho - log(1 - rho),          A[p,c] ~ Bernoulli(exp(ll1 - logsumexp(ll0, ll1))),
// p = 1..K sequentially inside a column, columns independent (the reference's Threads.@threads axis).
// Same conditional distribution, O(N w) work per sweep instead of O(K^2 N).  The baseline integral cancels in ll1 - ll0: a grid
// baseline (LogGaussianCoxProcess) only changes the intensities a column starts from (the per-event rates in by-node order) and the
// lower bound lambda0min_c = min over the column's events of lambda0_c(t_i) that the certification and the ON-bucket floor use.
//
// Cached form (default; k_adj_build + k_adj_sweep).  WHICH (child event, window predecessor) pairs exist, and their
// lags, depends on the data and the look-back horizon only, so the pairs are bucketed once per events handle:
//   virtual column = (child column c, time chunk g of the column's events), buckets by parent node p inside it, entries
//   stably ordered by (child event, window position); per pair a u16 event index inside the chunk and either the f64 lag
//   (10 B) or -- LogitNormal, memory permitting -- the parameter-free part of the impulse, logit(dt/D) and 1/(dt (D-dt))
//   (18 B), so that a sweep pays one exp per pair; entries of one (event, parent) that repeat sit next to each other, flagged.
// A Gibbs sweep streams that structure.  The intensities lambda_i of a column stay in SHARED MEMORY for the whole column: a
// thread-block CLUSTER of 1, 2, 4 or 8 CTAs (1024 threads each, one per SM) owns a column, CTA r holding chunk r (up to
// 26 624 events = 208 KB each), so the per-entry gather that bound the first version (one DRAM sector per entry) is an LDS
// and a flip never leaves the chip.  The K sequential Bernoulli steps run speculatively in batches of S <= 32 buckets: a
// step only changes lambda when its link flips, so the S sums are evaluated in parallel (32/S warps per bucket) from the
// current lambda, every CTA's partial sums travel through distributed shared memory to all CTAs of the cluster (one cluster
// barrier per batch), each CTA then takes the same decisions in order and accepts them as far as they can be CERTIFIED: a
// flip moves every intensity by at most its bucket's largest contribution, which bounds a later sum S from both sides,
// S / (1 + on / lambda0min_c) <= S' <= S (1 + off / lambda0min_c); a decision whose margin exceeds its side's bound is the decision of
// the sequential sweep (see the decision block of k_adj_sweep).  The batch is cut at the first bucket that cannot be
// certified and restarts there; the accepted flips are applied (S follows the observed restart rate, down to 1, the plain
// sequential sweep).  The result is exactly that of the sequential sweep.  The log terms are
// accumulated as a quotient of running products (one log per lane and batch instead of one per entry).
// Columns too large for a cluster's shared memory keep lambda in global memory between batches and stream their chunks
// per batch through one CTA.  Everything is order-deterministic: no atomics, fixed reduction trees.
//
// Uncached form (k_adjacency): the structure is re-bucketed inside every sweep; used when it does not fit in memory.
#include "cont_sweep.cuh"
int nhp_cont_params_refresh(nhp_ctx *ctx);  // cont_conjugate.cu
#include <cub/cub.cuh>
#include <algorithm>
#include <utility>

struct AdjArgs {
    const double *t; const int *c; int64_t n;
    const int *order;        // child events sorted by (node, time): event indices
    const int *node_ptr;     // [K+1] offsets into order
    const double *Mn;        // [K] events per node
    int K; const void *table_w;  // table without the adjacency factor
    const double *lambda0; const double *W; double *A;  // A: [K*K] parent-major as passed, updated in place
    const double *lam0bn, *lam0min;  // grid baseline: per-event rates in by-node order, per-node minima (NULL: lambda0)
    const double *rho; const double *u; uint64_t seed, counter;
    double D, horizon, duration;
    int64_t cap;             // scratch entries per CTA
    int *ent_i; double *ent_v; double *lam; double *gacc;  // per-CTA scratch regions
    int64_t max_col;         // max child events per column
    int *flag;
    int col_begin, col_stride;  // this call owns the columns c with c % col_stride == col_begin
};

__device__ __forceinline__ int lo_of_event(const double *t, int64_t i, double horizon) {
    // first j with t[j] > t[i] - horizon (galloping backwards, as k_tile_lo)
    double thr = t[i] - horizon;
    int64_t good = i, bad = -1, step = 32;
    while (true) {
        int64_t cand = i - step;
        if (cand <= 0) { if (t[0] > thr) good = 0; else bad = 0; break; }
        if (t[cand] > thr) { good = cand; step <<= 1; } else { bad = cand; break; }
    }
    while (good - bad > 1) { int64_t mid = (good + bad) >> 1; if (t[mid] > thr) good = mid; else bad = mid; }
    return (int)good;
}

template <int KIND> __global__ void __launch_bounds__(256) k_adjacency(const AdjArgs a) {
    typedef typename EntryOf<KIND>::type E;
    extern __shared__ int s_dyn[];  // [K+1] bucket offsets, [K] cursors
    __shared__ FastTables s_ft;
    __shared__ double s_red[8];
    __shared__ double s_anew;
    int *s_off = s_dyn, *s_cur = s_dyn + a.K + 1;
    fast_tables_load(&s_ft);
    int *ent_i = a.ent_i + (size_t)blockIdx.x * a.cap;
    double *ent_v = a.ent_v + (size_t)blockIdx.x * a.cap;
    double *lam = a.lam + (size_t)blockIdx.x * a.max_col;
    double *gacc = a.gacc + (size_t)blockIdx.x * a.max_col;
    for (int c = a.col_begin + blockIdx.x * a.col_stride; c < a.K; c += gridDim.x * a.col_stride) {
        const int e0 = a.node_ptr[c], e1 = a.node_ptr[c + 1];
        const E *col = reinterpret_cast<const E *>(a.table_w) + (size_t)c * a.K;
        const double lam0 = a.lam0min ? a.lam0min[c] : a.lambda0[c];  // lower bound of every event's baseline rate
        // ---- A1: bucket sizes
        for (int k = threadIdx.x; k <= a.K; k += blockDim.x) s_off[k] = 0;
        __syncthreads();
        // one warp per child event, lanes striding its window (coalesced reads of the time-sorted stream)
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = blockDim.x >> 5;
        for (int e = e0 + wid; e < e1; e += nw) {
            int i = a.order[e];
            double thr = a.t[i] - a.horizon;
            for (int j = i - 1 - lane; j >= 0; j -= 32) {
                if (!(__ldg(a.t + j) > thr)) break;
                atomicAdd(&s_off[__ldg(a.c + j) + 1], 1);
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) {  // exclusive scan (K is small next to the event work)
            int run = 0;
            for (int k = 0; k < a.K; k++) { int v = s_off[k + 1]; s_off[k] = run; s_cur[k] = run; run += v; }
            s_off[a.K] = run;
            if (run > a.cap) atomicOr(a.flag, 32);
        }
        __syncthreads();
        if (s_off[a.K] > a.cap) continue;  // cannot happen: cap is sized from the exact per-column totals
        // ---- A2: emit (event, G) entries and the current intensities
        for (int e = e0 + wid; e < e1; e += nw) {
            int i = a.order[e];
            double ti = a.t[i], thr = ti - a.horizon, s = 0.0;
            for (int j = i - 1 - lane; j >= 0; j -= 32) {
                double tj = __ldg(a.t + j);
                if (!(tj > thr)) break;
                int p = __ldg(a.c + j);
                double v = pair_value(load_entry(col + p), ti - tj, a.D, &s_ft);
                int pos = atomicAdd(&s_cur[p], 1);
                ent_i[pos] = e - e0;
                ent_v[pos] = v;
                s += a.A[p + (int64_t)a.K * c] * v;
            }
            s = warp_sum(s);
            if (lane == 0) { lam[e - e0] = (a.lam0bn ? a.lam0bn[e] : lam0) + s; gacc[e - e0] = 0.0; }
        }
        __syncthreads();
        // ---- B: K sequential Bernoulli steps
        for (int p = 0; p < a.K; p++) {
            const int b0 = s_off[p], b1 = s_off[p + 1];
            const int64_t kk = p + (int64_t)a.K * c;
            const double a_old = a.A[kk];
            double part = 0.0;
            if (b1 > b0) {
                // aggregate G_i[p] over the (rare) events that hold node p more than once in their window:
                // fire-and-forget reductions, no ownership protocol
                for (int e = b0 + threadIdx.x; e < b1; e += blockDim.x) {
                    const double v = ent_v[e];
                    if (v > 0.0) red_add_f64(&gacc[ent_i[e]], v);
                }
                __syncthreads();
                // every entry carries its share v/g of the event's term log((base + g)/base)
                for (int e = b0 + threadIdx.x; e < b1; e += blockDim.x) {
                    const double v = ent_v[e];
                    if (v > 0.0) {
                        const int ii = ent_i[e];
                        const double g = gacc[ii], l = lam[ii];
                        const double base = a_old != 0.0 ? fmax(l - g, lam0) : l;  // the intensity without this parent is at least lambda0min_c
                        const double term = log((base + g) / base);
                        part += (v == g) ? term : term * (v / g);
                    }
                }
                part = warp_sum(part);
                if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = part;
                __syncthreads();
            }
            if (threadIdx.x == 0) {
                double sum = 0.0;
                if (b1 > b0) for (int w = 0; w < 8; w++) sum += s_red[w];
                double rho = a.rho[kk];
                // ll1 - ll0 (continuous.jl:477-483): integrated-intensity difference, log-intensity difference, prior
                double delta = -a.W[kk] * a.Mn[p] + sum + (log(rho) - log(1.0 - rho));
                double p1 = delta >= 0.0 ? 1.0 / (1.0 + exp(-delta)) : exp(delta) / (1.0 + exp(delta));
                if (delta != delta) { atomicOr(a.flag, 64); p1 = 0.0; }
                double uu = a.u ? a.u[kk] : philox_uniform(a.seed, (uint64_t)kk, a.counter);
                double an = uu <= p1 ? 1.0 : 0.0;  // rand(Bernoulli(p)) = rand() <= p
                a.A[kk] = an;
                s_anew = an;
            }
            __syncthreads();
            if (b1 > b0) {
                const double an = s_anew;
                const double sgn = an - a_old;  // +1 link switched on, -1 switched off, 0 unchanged
                for (int e = b0 + threadIdx.x; e < b1; e += blockDim.x) {
                    const double v = ent_v[e];
                    if (v > 0.0) {
                        const int ii = ent_i[e];
                        if (sgn != 0.0) red_add_f64(&lam[ii], sgn * v);
                        gacc[ii] = 0.0;
                    }
                }
                __syncthreads();
            }
        }
        __syncthreads();
    }
}


// ---------------------------------------------------------------------------------------
// cached structure: build once, sweep many times
// ---------------------------------------------------------------------------------------
constexpr int ADJ_CHUNK_MAX = 26624;   // child events per chunk: 208 KB of shared-memory intensities
constexpr int ADJ_THREADS = 1024;      // sweep CTA: one per SM (512 threads with 128 registers each measured 8 % slower: 45.3 vs 41.9 ms)
constexpr int ADJ_VW = 32;             // bucket slots of a batch: one per warp (a CTA with fewer warps takes several slots per warp, one after the other)
constexpr int ADJ_SMAX_LOG2 = 5;
constexpr int ADJ_SMAX = 1 << ADJ_SMAX_LOG2;  // largest speculative batch (buckets per batch); the size follows the observed flip rate, down to 1
constexpr int ADJ_INIT_PF = 8;       // links ahead whose buckets are prefetched to L2 while a column's intensities are built up
constexpr int ADJ_CLUSTER_MAX = 8;     // portable cluster size limit

// a column's ne child events are split into G chunks of this many events (the last one may be shorter)
__host__ __device__ inline int adj_chunk_size(int ne, int G) { return G > 0 ? (ne + G - 1) / G : 0; }

// entries per virtual column: every child event adds its window length; the window start of every owned event is kept for the build
__global__ void k_adj_count(const double *__restrict__ t, const int *__restrict__ c, const int *__restrict__ order, const int *__restrict__ node_ptr,
                            const int *__restrict__ vstart, int64_t n_own, double horizon, int cb, int cs, unsigned long long *__restrict__ vcount,
                            int *__restrict__ lo_out, int *__restrict__ max_win, const unsigned short *__restrict__ wlen) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;  // blockDim.x is a multiple of 32: whole warps reach the votes below
    int v = -1;
    unsigned w = 0u;
    if (e < n_own) {
        const int i = order[e], col = c[i];
        if (col % cs == cb) {
            const int le = (int)(e - node_ptr[col]), ne = node_ptr[col + 1] - node_ptr[col], G = vstart[col + 1] - vstart[col];
            v = vstart[col] + le / adj_chunk_size(ne, G);
            // the sweeps' cached window length when it was taken with this horizon (saturated values are searched)
            const unsigned wl = wlen ? (unsigned)wlen[i] : 65535u;
            const int lo = wl < 65535u ? i - (int)wl : lo_of_event(t, i, horizon);
            if (lo_out) lo_out[i] = lo;
            w = (unsigned)(i - lo);
        }
    }
    // consecutive events of the by-node order share their virtual column: one atomic per warp instead of 32 on the same address
    const int v0 = __shfl_sync(0xffffffffu, v, 0);
    if (__all_sync(0xffffffffu, v == v0 && w < (1u << 26))) {
        const unsigned tot = __reduce_add_sync(0xffffffffu, w), mx = __reduce_max_sync(0xffffffffu, w);
        if ((threadIdx.x & 31) == 0 && v0 >= 0 && tot > 0u) {
            atomicAdd(&vcount[v0], (unsigned long long)tot);
            if (max_win) atomicMax(max_win, (int)mx);
        }
    } else if (v >= 0 && w > 0u) {
        atomicAdd(&vcount[v], (unsigned long long)w);
        if (max_win) atomicMax(max_win, (int)min(w, 0x7fffffffu));
    }
}

// Per event: node | distance to the previous event of the same node | distance to the next one (22 bits each, saturated).  With it
// the build knows, from the predecessor alone, whether a window holds the predecessor's node more than once.
constexpr int ADJ_LINK_BITS = 22, ADJ_NODE_BITS = 20;
constexpr unsigned ADJ_LINK_SAT = (1u << ADJ_LINK_BITS) - 1u;
__global__ void k_adj_links(const int *__restrict__ order, const int *__restrict__ node_ptr, const int *__restrict__ c, int64_t n,
                            unsigned long long *__restrict__ pk) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n) return;
    const int i = order[e], col = c[i];
    unsigned dp = ADJ_LINK_SAT, dn = ADJ_LINK_SAT;
    if (e > node_ptr[col]) dp = min(ADJ_LINK_SAT, (unsigned)(i - order[e - 1]));
    if (e + 1 < node_ptr[col + 1]) dn = min(ADJ_LINK_SAT, (unsigned)(order[e + 1] - i));
    pk[i] = (unsigned long long)(unsigned)col | ((unsigned long long)dp << ADJ_NODE_BITS) | ((unsigned long long)dn << (ADJ_NODE_BITS + ADJ_LINK_BITS));
}

struct AdjBuildArgs {
    const double *t; const unsigned long long *pk; const int *lo; const int *order, *node_ptr;
    int K; double D;
    const int *vstart, *vnode, *vorder; const int64_t *vbase;   // vorder: the order in which the virtual columns are taken
    int *boff; unsigned short *ent_i; double *ent_x; int pre;   // pre: LogitNormal payload (logit, Jacobian), one 16-byte record per entry, instead of the lag
    int nv, nw;      // virtual columns; warps per CTA
    int *next, *flag;
};

// Counting sort of one virtual column's (child event, window predecessor) pairs by parent node.  A parent's bucket has two
// sections: first the SINGLES -- pairs whose (event, parent) occurs once in the event's window (94 % at config 4), which a sweep
// streams with no bookkeeping at all -- then the RUNS: the entries of one (event, parent) next to each other in window order, all but
// the first carrying the continuation bit.
// Singles take their slot from ONE cursor per (parent) shared by the CTA's warps (shared-memory atomics): a section then fills
// front to back, the partially written sectors of a column's 2 K sections stay few enough to sit in L2 until they are complete, and
// DRAM sees whole sectors (per-warp cursors multiplied the open sectors by the warp count: 570 GB written for 116 GB of payload);
// their order inside a section follows the scheduling, which only moves the rounding of a bucket's sum.  Run entries keep private
// per-warp cursors (warp w owns a contiguous range of the chunk's events), so a run is contiguous and in window order.
// Payload per entry: the lag t_i - t_j, or -- LogitNormal, when memory allows -- what the impulse needs of it and what does not
// depend on the parameters: z = logit(dt / D) and q = 1 / (dt (D - dt)), so that a sweep evaluates one exp per pair instead of
// a log, a reciprocal and an exp (pairs outside the support get q = 0).
// cache policy of the build: the event stream is read once per pass (evict first), the half-written output sectors should stay in
// L2 until their neighbours arrive (evict last)
__device__ __forceinline__ unsigned long long l2_policy_evict_first() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_normal() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_normal.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long l2_policy_evict_last() {
    unsigned long long pol;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
    return pol;
}
__device__ __forceinline__ unsigned long long ldg_stream_u64(const unsigned long long *p, unsigned long long pol) {
    unsigned long long v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.u64 %0, [%1], %2;" : "=l"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ double ldg_stream_f64(const double *p, unsigned long long pol) {
    double v;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(v) : "l"(p), "l"(pol));
    return v;
}
__device__ __forceinline__ void st_keep_f64(double *p, double v, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep_f64x2(double *p, double v0, double v1, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.v2.f64 [%0], {%1, %2}, %3;" ::"l"(p), "d"(v0), "d"(v1), "l"(pol) : "memory");
}
__device__ __forceinline__ void st_keep_u16(unsigned short *p, unsigned short v, unsigned long long pol) {
    asm volatile("st.global.L2::cache_hint.u16 [%0], %1, %2;" ::"l"(p), "h"(v), "l"(pol) : "memory");
}

__device__ __forceinline__ int adj_pk_dprev(unsigned long long pk) { return (int)((unsigned)(pk >> ADJ_NODE_BITS) & ADJ_LINK_SAT); }
__device__ __forceinline__ void adj_pk_decode(unsigned long long pk, int j, int i, int lo, int &p, bool &multi, bool &cont) {
    p = (int)((unsigned)pk & ((1u << ADJ_NODE_BITS) - 1u));
    const int dp = adj_pk_dprev(pk), dn = (int)(pk >> (ADJ_NODE_BITS + ADJ_LINK_BITS));
    cont = (int64_t)j + dn < (int64_t)i;  // a more recent event of the same node sits in the window: this entry continues its run
    multi = cont || (j - dp >= lo);
}
// one entry: index word + payload (the lag, or the parameter-free part of the LogitNormal impulse)
static __device__ __noinline__ double2 adj_payload_slow(double dt, double D) {  // lags at the edge of the support (or outside it)
    const double b = D - dt;
    double z = 0.0, q = 0.0;
    if (dt > 0.0 && b > 0.0) {  // Distributions.pdf(LogitNormal, x) is zero outside 0 < x < 1 (impulses.jl:174-178)
        q = 1.0 / (dt * b);
        z = log(dt / b);
        if (!(q <= 1.7976931348623157e308) || !(fabs(z) <= 1.7976931348623157e308)) { z = 0.0; q = 0.0; }  // lag so small that the pdf underflows
    }
    return make_double2(z, q);
}
__device__ __forceinline__ void adj_store_entry(unsigned short *ei, double *ex, int pre, unsigned pos, unsigned tag, double dt, double D, unsigned long long pol,
                                                const FastTables *ft) {
    st_keep_u16(ei + pos, (unsigned short)tag, pol);
    if (pre) {
        const double b = D - dt;
        double2 zq;
        if (in_mid_range(dt) && in_mid_range(b)) {  // the arithmetic of pair_value: one reciprocal serves the Jacobian and the logit argument
            zq.y = fast_rcp_mid(dt * b);
            zq.x = fast_log_n(dt * dt * zq.y, ft);
        } else zq = adj_payload_slow(dt, D);
        st_keep_f64x2(ex + 2 * (size_t)pos, zq.x, zq.y, pol);
    } else st_keep_f64(ex + pos, dt, pol);
}

constexpr int ADJ_BUILD_PF = 4;  // events of look-ahead of the L2 prefetch (windows longer than 32 / 16 lines are covered in part)
__global__ void __launch_bounds__(1024) k_adj_build(const AdjBuildArgs a) {
    extern __shared__ int s_dyn[];
    __shared__ int s_v;
    __shared__ FastTables s_ft;
    fast_tables_load(&s_ft);
    const FastTables *ft = &s_ft;
    const int K = a.K;
    int *s_off = s_dyn;                                                  // [2K+1] section offsets: singles of p, runs of p, ...
    unsigned *s_curS = reinterpret_cast<unsigned *>(s_dyn + 2 * K + 1);  // [K] singles: count, then the CTA-wide cursor
    unsigned *s_curM = s_curS + K;                                       // [K] run entries: count, then the CTA-wide cursor (a run is reserved whole)
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5, nw = blockDim.x >> 5;
    const unsigned long long pol_rd = l2_policy_evict_normal(), pol_wr = l2_policy_evict_last();  // reads: shared through L2 by the CTAs of a time slice
    for (;;) {
        __syncthreads();
        if (tid == 0) s_v = atomicAdd(a.next, 1);
        __syncthreads();
        if (s_v >= a.nv) break;
        const int v = a.vorder[s_v];
        const int col = a.vnode[v], g = v - a.vstart[col], G = a.vstart[col + 1] - a.vstart[col];
        const int ne = a.node_ptr[col + 1] - a.node_ptr[col], csz = adj_chunk_size(ne, G);
        const int eb = a.node_ptr[col] + g * csz, ee = min(a.node_ptr[col] + ne, eb + csz);  // positions in the by-node order
        for (int k = tid; k < 2 * K; k += blockDim.x) s_curS[k] = 0u;
        __syncthreads();
        // ---- A: counts.  Warps take blocks of 32 events round robin.
        for (int e0 = eb + wid * 32; e0 < ee; e0 += nw * 32) {
            int my_i = 0, my_lo = 0;
            if (e0 + lane < ee) { my_i = a.order[e0 + lane]; my_lo = a.lo[my_i]; }  // 32 events' headers in one round trip
            const int cnt = min(32, ee - e0);
            for (int s = 0; s < cnt; s++) {
                const int i = __shfl_sync(0xffffffffu, my_i, s), lo = __shfl_sync(0xffffffffu, my_lo, s);
                {   // the window of the event ADJ_BUILD_PF places ahead starts towards L2 (one 128-byte line per lane)
                    const int sp = min(s + ADJ_BUILD_PF, cnt - 1);
                    const int ip = __shfl_sync(0xffffffffu, my_i, sp), lp = __shfl_sync(0xffffffffu, my_lo, sp);
                    const int j = (lp & ~15) + lane * 16;
                    if (s + ADJ_BUILD_PF < cnt && j < ip) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.pk + j));
                }
                for (int j = i - 1 - lane; j >= lo; j -= 64) {  // two rounds in flight
                    const int j2 = j - 32;
                    const unsigned long long pk = ldg_stream_u64(a.pk + j, pol_rd), pk2 = j2 >= lo ? ldg_stream_u64(a.pk + j2, pol_rd) : 0ull;
                    int p; bool multi, cont;
                    adj_pk_decode(pk, j, i, lo, p, multi, cont);
                    atomicAdd(multi ? &s_curM[p] : &s_curS[p], 1u);
                    if (j2 >= lo) {
                        adj_pk_decode(pk2, j2, i, lo, p, multi, cont);
                        atomicAdd(multi ? &s_curM[p] : &s_curS[p], 1u);
                    }
                }
            }
        }
        __syncthreads();
        // ---- section sizes (singles padded to whole blocks of 64 entries, runs to whole groups of 32)
        for (int p = tid; p < K; p += blockDim.x) {
            s_off[2 * p + 1] = (int)((s_curS[p] + 63u) & ~63u);   // singles: whole blocks of 64 entries (the sweep reads them unconditionally)
            s_off[2 * p + 2] = (int)((s_curM[p] + 31u) & ~31u);
        }
        if (tid == 0) s_off[0] = 0;
        __syncthreads();
        if (tid < 32) {  // exclusive scan of the 2 K section sizes by one warp
            int carry = 0;
            for (int k0 = 0; k0 < 2 * K; k0 += 32) {
                const int k = k0 + lane;
                int x = k < 2 * K ? s_off[k + 1] : 0;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
                if (k < 2 * K) s_off[k + 1] = carry + x;
                carry += __shfl_sync(0xffffffffu, x, 31);
            }
            if (lane == 0 && (int64_t)carry > a.vbase[v + 1] - a.vbase[v]) atomicOr(a.flag, 128);
        }
        __syncthreads();
        for (int k = tid; k <= 2 * K; k += blockDim.x) a.boff[(int64_t)v * (2 * K + 1) + k] = s_off[k];
        for (int p = tid; p < K; p += blockDim.x) { s_curS[p] = (unsigned)s_off[2 * p]; s_curM[p] = (unsigned)s_off[2 * p + 1]; }
        __syncthreads();
        // ---- B: scatter, one pass over every window.  A single takes the next slot of its section.  The most recent entry of a run (its
        //      head) follows the same-node links back through the window, reserves the run's slots at once and writes the run in window order.
        unsigned short *ei = a.ent_i + a.vbase[v];
        double *ex = a.ent_x + (a.pre ? 2 : 1) * a.vbase[v];
        for (int e0 = eb + wid * 32; e0 < ee; e0 += nw * 32) {
            int my_i = 0, my_lo = 0;
            double my_t = 0.0;
            if (e0 + lane < ee) { my_i = a.order[e0 + lane]; my_lo = a.lo[my_i]; my_t = a.t[my_i]; }
            const int cnt = min(32, ee - e0);
            for (int s = 0; s < cnt; s++) {
                const int i = __shfl_sync(0xffffffffu, my_i, s), lo = __shfl_sync(0xffffffffu, my_lo, s);
                {   // lanes 0-15: the packed records, lanes 16-31: the times of the window ADJ_BUILD_PF events ahead
                    const int sp = min(s + ADJ_BUILD_PF, cnt - 1);
                    const int ip = __shfl_sync(0xffffffffu, my_i, sp), lp = __shfl_sync(0xffffffffu, my_lo, sp);
                    const int j = (lp & ~15) + (lane & 15) * 16;
                    if (s + ADJ_BUILD_PF < cnt && j < ip) {
                        if (lane < 16) asm volatile("prefetch.global.L2 [%0];" ::"l"(a.pk + j));
                        else asm volatile("prefetch.global.L2 [%0];" ::"l"(a.t + j));
                    }
                }
                const double ti = __shfl_sync(0xffffffffu, my_t, s);
                const unsigned le = (unsigned)(e0 + s - eb);
                for (int j = i - 1 - lane; j >= lo; j -= 64) {  // two rounds in flight
                    const int j2 = j - 32;
                    const bool has2 = j2 >= lo;
                    const unsigned long long pk = ldg_stream_u64(a.pk + j, pol_rd), pk2 = has2 ? ldg_stream_u64(a.pk + j2, pol_rd) : 0ull;
                    const double tj = ldg_stream_f64(a.t + j, pol_rd), tj2 = has2 ? ldg_stream_f64(a.t + j2, pol_rd) : 0.0;
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        if (r == 1 && !has2) break;
                        const int jc = r ? j2 : j;
                        const unsigned long long pkc = r ? pk2 : pk;
                        const double dt = ti - (r ? tj2 : tj);
                        int p; bool multi, cont;
                        adj_pk_decode(pkc, jc, i, lo, p, multi, cont);
                        if (!multi) adj_store_entry(ei, ex, a.pre, atomicAdd(&s_curS[p], 1u), le, dt, a.D, pol_wr, ft);
                        else if (!cont) {
                            int len = 1;
                            for (int jj = jc - adj_pk_dprev(pkc); jj >= lo; len++) jj -= adj_pk_dprev(__ldg(a.pk + jj));
                            unsigned pos = atomicAdd(&s_curM[p], (unsigned)len);
                            adj_store_entry(ei, ex, a.pre, pos, le, dt, a.D, pol_wr, ft);
                            for (int jj = jc - adj_pk_dprev(pkc); jj >= lo;) {
                                adj_store_entry(ei, ex, a.pre, ++pos, le | 0x8000u, ti - __ldg(a.t + jj), a.D, pol_wr, ft);
                                jj -= adj_pk_dprev(__ldg(a.pk + jj));
                            }
                        }
                    }
                }
            }
        }
        __syncthreads();
        // ---- padding: entries that evaluate to exactly zero (event 0, q = 0 | lag -1), so the sweeps read whole groups unconditionally
        for (int k = tid; k < 2 * K; k += blockDim.x) {
            const int p = k >> 1;
            for (int e = (k & 1) ? (int)s_curM[p] : (int)s_curS[p]; e < s_off[k + 1]; e++) {  // from the section's true end (its cursor)
                ei[e] = 0;
                if (a.pre) { ex[2 * (size_t)e] = 0.0; ex[2 * (size_t)e + 1] = 0.0; } else ex[e] = -1.0;
            }
        }
    }
}

// Inputs of the K^2 Bernoulli decisions, computed ahead of the sweep so that the deciding lanes only load them:
// ll1 - ll0 = -W[p,c] Mn[p] + (log-intensity difference) + logit(rho)  (continuous.jl:477-483), the uniform and its logit
__global__ void k_adj_prep(int K, const double *__restrict__ W, const double *__restrict__ Mn, const double *__restrict__ rho, double rho_scalar,
                           const double *__restrict__ u, uint64_t seed, uint64_t counter, double4 *__restrict__ dec) {
    const int64_t kk = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (kk >= (int64_t)K * K) return;
    const double r = rho ? rho[kk] : rho_scalar;
    const double uu = u ? u[kk] : philox_uniform(seed, (uint64_t)kk, counter);
    dec[kk] = make_double4(W[kk] * Mn[kk % K], log(r) - log(1.0 - r), uu, log(uu) - log(1.0 - uu));
}

struct AdjSweepArgs {
    const int *node_ptr;
    int K; const void *table_w;
    const double *lambda0; double *A;   // A: [K*K] parent-major, device, updated in place
    const double *lam0bn, *lam0min;     // grid baseline: per-event rates in by-node order, per-node minima (NULL: lambda0)
    const double4 *dec;    // [K*K] per link: W Mn[p], logit(rho), u, logit(u)  (k_adj_prep)
    double D;
    const int *vstart; const int64_t *vbase; const int *boff; const unsigned short *ent_i; const double *ent_x;   // PRE: ent_x holds (logit, Jacobian) pairs
    double *lam;           // [n] by-node order (only used when a column's chunks do not all sit in shared memory)
    int chunk_max;         // doubles of shared memory in front of the adjacency bit row
    int *flag, *next; unsigned long long *stat;
    int col_begin, col_stride, ncols;
    const int *corder;     // [ncols] owned columns, most child events first (NULL: col_begin + i col_stride)
    int s0;         // first batch size
    int bo_smem;    // 1: the bucket offsets of the resident chunk are kept in shared memory behind the adjacency bits ((2 K + 1) ints)
};

// thread-block cluster primitives (distributed shared memory of the CTAs that share a column)
__device__ __forceinline__ unsigned cluster_ctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ unsigned cluster_nctarank() { unsigned r; asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_cluster_u32(int *local_smem, unsigned rank, int v) {
    unsigned ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(local_smem)), "r"(rank));
    asm volatile("st.shared::cluster.u32 [%0], %1;" ::"r"(ra), "r"(v) : "memory");
}
__device__ __forceinline__ void st_cluster_f64(double *local_smem, unsigned rank, double v) {
    unsigned ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(smem_u32(local_smem)), "r"(rank));
    asm volatile("st.shared::cluster.f64 [%0], %1;" ::"r"(ra), "d"(v) : "memory");
}

// impulse value of one cached pair.  PRE = 0: x is the lag.  PRE = 1 (LogitNormal): x = logit(dt / D), y = 1 / (dt (D - dt)) from the
// structure, so the pair costs one exp: cf y exp(-h (x - mu)^2)   (cf carries W sqrt(tau / 2 pi) D^2; y = 0 outside the support)
template <int KIND, int PRE>
__device__ __forceinline__ double adj_value(const typename EntryOf<KIND>::type &en, double x, double y, double D, const FastTables *ft);
template <> __device__ __forceinline__ double adj_value<NHP_EXPONENTIAL, 0>(const EntryEX &en, double x, double, double D, const FastTables *ft) { return pair_value(en, x, D, ft); }
template <> __device__ __forceinline__ double adj_value<NHP_LOGITNORMAL, 0>(const EntryLN &en, double x, double, double D, const FastTables *ft) { return pair_value(en, x, D, ft); }
template <> __device__ __forceinline__ double adj_value<NHP_LOGITNORMAL, 1>(const EntryLN &en, double x, double y, double, const FastTables *ft) {
    const double dz = x - en.mu;
    return (en.cf * y) * fast_exp_c(-(en.h * dz) * dz, ft);  // exponent <= 0: no overflow branch; flushes to 0 below -707
}

// payload of entry k.  PRE: the 16-byte record (x, y) at ex[2k], one 128-bit load; else the lag at ex[k]
template <int PRE> __device__ __forceinline__ void adj_ld(const double *__restrict__ ex, int k, double &x, double &y) {
    if (PRE) { const double2 v = __ldg(reinterpret_cast<const double2 *>(ex) + k); x = v.x; y = v.y; }
    else { x = __ldg(ex + k); y = 0.0; }
}
// payloads of the entries k (even) and k + 1: one 256-bit (PRE) or 128-bit load
template <int PRE> __device__ __forceinline__ void adj_ld2(const double *__restrict__ ex, int k, double2 &x, double2 &y) {
    if (PRE) asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(x.x), "=d"(y.x), "=d"(x.y), "=d"(y.y) : "l"(ex + 2 * (size_t)k));
    else x = __ldg(reinterpret_cast<const double2 *>(ex + k));
}
// L2 prefetch of the entries [f0, f1) of one virtual column by the whole CTA (one 128-byte line per thread and step)
template <int PRE> __device__ __forceinline__ void adj_pf_range(const unsigned short *ei, const double *ex, int f0, int f1, int tid) {
    constexpr int per = PRE ? 8 : 16;  // entries per line of the payload
    for (int e = f0 + tid * per; e < f1; e += ADJ_THREADS * per) {
        asm volatile("prefetch.global.L2 [%0];" ::"l"(ex + (PRE ? 2 : 1) * (size_t)e));
        if (((e - f0) & 63) == 0) asm volatile("prefetch.global.L2 [%0];" ::"l"(ei + e));
    }
}

// One group of 32 consecutive entries [eb, eb + 32) of a run section that ends at b1, one entry per lane: the impulse value of
// every entry and, for the first entry of each (event, parent) run (the "head"), the run's total.  Returns head.
template <int KIND, int PRE>
__device__ __forceinline__ bool adj_group(const typename EntryOf<KIND>::type &en, const unsigned short *__restrict__ ei, const double *__restrict__ ex,
                                          int eb, int b1, int lane, unsigned ii, double x, double y, double D,
                                          const FastTables *ft, double &gsum, int next_first = -1) {  // next_first: index word of entry eb + 32 when the caller already holds it
    const bool valid = eb + lane < b1;
    double v = adj_value<KIND, PRE>(en, x, y, D, ft);
    v = valid ? v : 0.0;
    const unsigned contmask = __ballot_sync(0xffffffffu, valid && (ii & 0x8000u));
    const bool head = valid && !((contmask >> lane) & 1u);
    int runlen = 0;
    gsum = v;
    if (contmask) {  // warp-uniform: some run has more than one entry in this group
        const unsigned fol = (contmask >> lane) >> 1;
        runlen = __ffs(~fol) - 1;  // entries behind this one that continue its run (inside the group)
        const int mr = __reduce_max_sync(0xffffffffu, head ? runlen : 0);
        for (int d = 1; d <= mr; d++) {
            const double vv = __shfl_down_sync(0xffffffffu, v, d);
            if (d <= runlen) gsum += vv;
        }
    }
    if (eb + 32 < b1) {  // warp-uniform: does the run that reaches lane 31 go on in the section's next group?  (one broadcast load)
        if ((next_first >= 0 ? (unsigned)next_first : (unsigned)__ldg(ei + eb + 32)) & 0x8000u) {
            if (head && lane + runlen == 31)
                for (int e2 = eb + 32; e2 < b1 && (__ldg(ei + e2) & 0x8000u); e2++) { double x2, y2; adj_ld<PRE>(ex, e2, x2, y2); gsum += adj_value<KIND, PRE>(en, x2, y2, D, ft); }
        }
    }
    return head;
}

// The log terms log((base + g) / base) of a bucket are accumulated as a quotient of running products -- one pair of logs per lane and
// bucket instead of one log per entry.  The exponents are taken out of the products every ADJ_RENORM factors (integer work); the
// smallest base and the largest base + g are tracked through their high words, and a bucket whose factors leave [2^-100, 2^100]
// (which the products could not hold) is redone with direct logs (adj_direct).
constexpr int ADJ_RENORM = 8;
struct AdjAcc {
    double num, den;  // running products of (base + g) and of base, both in [2^-801, 2^801)
    int bal;          // binary exponents taken out so far: log ratio = log(num) - log(den) + bal ln 2
    int mn, mx, gm;   // high words of the smallest base, the largest base + g, the largest g
};
__device__ __forceinline__ void acc_init(AdjAcc &A) { A.num = 1.0; A.den = 1.0; A.bal = 0; A.mn = 0x7fffffff; A.mx = 0; A.gm = 0; }
__device__ __forceinline__ void acc_renorm(AdjAcc &A) {
    const int hn = __double2hiint(A.num), hd = __double2hiint(A.den);
    const int en = (hn >> 20) - 1023, ed = (hd >> 20) - 1023;
    A.num = __hiloint2double(hn - (en << 20), __double2loint(A.num));
    A.den = __hiloint2double(hd - (ed << 20), __double2loint(A.den));
    A.bal += en - ed;
}
__device__ __forceinline__ bool acc_in_range(const AdjAcc &A) { return A.mn >= 0x39B00000 && A.mx < 0x46300000; }  // 2^-100 <= base, base + g < 2^100
// ON: the bucket's link is on, the intensity without this parent is l - g, kept at or above lambda0 (floor_); a link that is off -- 95 % of
// the buckets of a sparse network -- takes the intensity as it is (no subtraction, no clamp: 8 of the loop's 140 instructions)
template <bool ON> __device__ __forceinline__ void acc_factor(AdjAcc &A, double v, double l, double floor_) {
    double base = l;
    if (ON) { const double t = l - v; base = t > floor_ ? t : floor_; }
    const double hi = base + v;
    A.num *= hi; A.den *= base;
    A.mn = min(A.mn, __double2hiint(base)); A.mx = max(A.mx, __double2hiint(hi)); A.gm = max(A.gm, __double2hiint(v));
}

template <bool ON> __device__ __forceinline__ void acc_factor2(AdjAcc &A, double v0, double l0, double v1, double l1, double floor_) {
    double b0 = l0, b1 = l1;
    if (ON) {
        const double t0 = l0 - v0, t1 = l1 - v1;
        b0 = t0 > floor_ ? t0 : floor_; b1 = t1 > floor_ ? t1 : floor_;
    }
    const double h0 = b0 + v0, h1 = b1 + v1;
    A.num *= h0 * h1; A.den *= b0 * b1;
    A.mn = min(A.mn, min(__double2hiint(b0), __double2hiint(b1)));
    A.mx = max(A.mx, max(__double2hiint(h0), __double2hiint(h1)));
    A.gm = max(A.gm, max(__double2hiint(v0), __double2hiint(v1)));
}

// L2 prefetch of the 64-entry block that starts at entry kb: lanes 0-1 take the two 64-byte halves of the indices, lanes 2-9 (2-17 with
// the 16-byte payload) the 64-byte pieces of the payload (one instruction per block; the arrays carry slack behind their last entry)
struct AdjPf { const char *base; int scale; };
template <int PRE> __device__ __forceinline__ AdjPf adj_pf_setup(const unsigned short *ei, const double *ex, int lane) {
    AdjPf f;
    f.base = nullptr; f.scale = 0;
    if (lane < 2) { f.base = reinterpret_cast<const char *>(ei) + lane * 64; f.scale = 2; }
    else if (lane < (PRE ? 18 : 10)) { f.base = reinterpret_cast<const char *>(ex) + (lane - 2) * 64; f.scale = PRE ? 16 : 8; }
    return f;
}
__device__ __forceinline__ void adj_pf(const AdjPf &f, int kb) {
    if (f.base) asm volatile("prefetch.global.L2 [%0];" ::"l"(f.base + (int64_t)kb * f.scale));
}

// singles of one bucket: this warp takes the blocks of 64 entries that start at gb, gb + stride, ... below s1 (the section is padded to
// whole blocks and starts on a 32-entry boundary: a lane reads entries 2 lane, 2 lane + 1 of its block with one 32-bit and one 256-bit
// load); one block ahead in registers, the block three ahead on its way to L2.  Padding entries evaluate to zero: factor 1.
// (Measured alternatives: two blocks ahead in registers spills at 64 registers per thread, 66 vs 42 ms; 512-thread CTAs with 128
// registers and that loop, 45 ms; loads made unconditional on the warp-uniform block test, 43.6 ms.)
template <int KIND, int PRE, bool ON>
__device__ __forceinline__ void adj_singles(const typename EntryOf<KIND>::type &en, const unsigned short *__restrict__ ei, const double *__restrict__ ex,
                                            int gb, const int s1, const int stride, const int lane,
                                            const double floor_, const double D, const double *lam_s, const FastTables *ft, const AdjPf &pf, AdjAcc &A) {
    const double xdef = PRE ? 0.0 : -1.0;
    adj_pf(pf, gb + stride); adj_pf(pf, gb + 2 * stride);
    int k = gb + 2 * lane;
    unsigned iw = 0u;
    double2 xw = make_double2(xdef, xdef), yw = make_double2(0.0, 0.0);
    if (k < s1) { iw = __ldg(reinterpret_cast<const unsigned *>(ei + k)); adj_ld2<PRE>(ex, k, xw, yw); }
    while (gb < s1) {
#pragma unroll 1
        for (int u = 0; u < ADJ_RENORM / 2; u++) {
            const unsigned ii = iw;
            const double2 x = xw, y = yw;
            adj_pf(pf, gb + 3 * stride);  // in L2 by the time the register load two blocks later asks for it
            k += stride;
            iw = 0u; xw = make_double2(xdef, xdef); yw = make_double2(0.0, 0.0);
            if (k < s1) { iw = __ldg(reinterpret_cast<const unsigned *>(ei + k)); adj_ld2<PRE>(ex, k, xw, yw); }
            const double v0 = adj_value<KIND, PRE>(en, x.x, y.x, D, ft), v1 = adj_value<KIND, PRE>(en, x.y, y.y, D, ft);
            acc_factor2<ON>(A, v0, lam_s[ii & 0xffffu], v1, lam_s[ii >> 16], floor_);
            gb += stride;
            if (gb >= s1) break;
        }
        acc_renorm(A);
    }
}

// run section of one bucket (general form: several entries of one (event, parent))
template <int KIND, int PRE, bool ON>
__device__ __forceinline__ void adj_runs(const typename EntryOf<KIND>::type &en, const unsigned short *__restrict__ ei, const double *__restrict__ ex,
                                         int eb, const int b1, const int stride, const int lane,
                                         const double floor_, const double D, const double *lam_s, const FastTables *ft, AdjAcc &A) {
    // one group ahead in registers: the lane's entry of the next group and the index word behind it (the look-ahead of adj_group)
    const double xdef = PRE ? 0.0 : -1.0;
    unsigned iw = 0u;
    double xw = xdef, yw = 0.0;
    int nfw = -1;
    if (eb < b1) {
        if (eb + lane < b1) { iw = (unsigned)__ldg(ei + eb + lane); adj_ld<PRE>(ex, eb + lane, xw, yw); }
        if (eb + 32 < b1) nfw = (int)__ldg(ei + eb + 32);
    }
    while (eb < b1) {
#pragma unroll 1
        for (int u = 0; u < ADJ_RENORM; u++) {
            const unsigned ii = iw;
            const double x = xw, y = yw;
            const int nf = nfw;
            const int en_ = eb + stride;
            iw = 0u; xw = xdef; yw = 0.0; nfw = -1;
            if (en_ < b1) {  // warp-uniform
                if (en_ + lane < b1) { iw = (unsigned)__ldg(ei + en_ + lane); adj_ld<PRE>(ex, en_ + lane, xw, yw); }
                if (en_ + 32 < b1) nfw = (int)__ldg(ei + en_ + 32);
            }
            double gs;
            const bool head = adj_group<KIND, PRE>(en, ei, ex, eb, b1, lane, ii, x, y, D, ft, gs, nf);
            acc_factor<ON>(A, head ? gs : 0.0, lam_s[ii & 0x7fffu], floor_);
            eb = en_;
            if (eb >= b1) break;
        }
        acc_renorm(A);
    }
}

// direct route (rare): the same share of a bucket -- groups eb, eb + stride, ... of [.., b1), singles and runs alike, a single is a
// run of one -- with one log per event; extreme or non-positive intensities end up here and a NaN surfaces as NHP_ERR_NUMERIC
template <int KIND, int PRE>
__device__ __noinline__ double2 adj_direct(const typename EntryOf<KIND>::type en, const unsigned short *__restrict__ ei, const double *__restrict__ ex,
                                           int eb, const int b1, const int stride, const int lane, const double onf,
                                           const double floor_, const double D, const double *lam_s, const FastTables *ft) {  // (sum of log terms, largest contribution)
    const double xdef = PRE ? 0.0 : -1.0;
    double acc = 0.0, gmx = 0.0;
    for (; eb < b1; eb += stride) {
        const bool valid = eb + lane < b1;
        const unsigned ii = valid ? (unsigned)__ldg(ei + eb + lane) : 0u;
        double x = xdef, y = 0.0;
        if (valid) adj_ld<PRE>(ex, eb + lane, x, y);
        double gs;
        if (adj_group<KIND, PRE>(en, ei, ex, eb, b1, lane, ii, x, y, D, ft, gs) && gs > 0.0) {
            const double l = lam_s[ii & 0x7fffu], t = fma(-onf, gs, l), base = t > floor_ ? t : floor_;
            acc += log((base + gs) / base);
            gmx = fmax(gmx, gs);
        }
    }
    return make_double2(acc, gmx);
}

// add sgn * (this parent's contribution) to the intensities of a bucket's events: all warps of the CTA.  A bucket holds about one entry
// per thread, so the call is a chain of latencies rather than a stream: the loads of the thread's first single and of the warp's first
// run group (and the look-ahead word of that group) are all issued before the first of them is used, and the run groups go to the warps
// from the last one down (the first warps are the ones that get a second single).
template <int KIND, int PRE>
__device__ __forceinline__ void adj_apply(const typename EntryOf<KIND>::type &en, const unsigned short *__restrict__ ei, const double *__restrict__ ex,
                                          const int s0, const int sm, const int rs, const int s1, const int warp, const int lane,
                                          const double sgn, double *lam, const double D, const FastTables *ft) {  // singles [s0, sm), run groups from rs (a group boundary) to s1
    const double xdef = PRE ? 0.0 : -1.0;
    int k = s0 + warp * 32 + lane;
    const bool hs = k < sm;
    unsigned iis = 0u;
    double xs = xdef, ys = 0.0;
    if (hs) { iis = __ldg(ei + k); adj_ld<PRE>(ex, k, xs, ys); }
    int eb = rs + (ADJ_THREADS / 32 - 1 - warp) * 32;
    const bool hr = eb < s1;  // warp-uniform
    unsigned iir = 0u;
    double xr = xdef, yr = 0.0;
    int nf = -1;
    if (hr) {
        if (eb + lane < s1) { iir = __ldg(ei + eb + lane); adj_ld<PRE>(ex, eb + lane, xr, yr); }
        if (eb + 32 < s1) nf = (int)__ldg(ei + eb + 32);
    }
    if (hs) {  // singles: distinct events, no bookkeeping
        const double v = adj_value<KIND, PRE>(en, xs, ys, D, ft);
        if (v > 0.0) lam[iis] += sgn * v;
    }
    for (k += ADJ_THREADS; k < sm; k += ADJ_THREADS) {
        const unsigned ii = __ldg(ei + k);
        double x, y;
        adj_ld<PRE>(ex, k, x, y);
        const double v = adj_value<KIND, PRE>(en, x, y, D, ft);
        if (v > 0.0) lam[ii] += sgn * v;
    }
    if (hr) {  // runs: the head carries the run's total
        double gs;
        if (adj_group<KIND, PRE>(en, ei, ex, eb, s1, lane, iir, xr, yr, D, ft, gs, nf) && gs > 0.0) lam[iir & 0x7fffu] += sgn * gs;
        for (eb += ADJ_THREADS; eb < s1; eb += ADJ_THREADS) {
            const bool valid = eb + lane < s1;
            const unsigned ii = valid ? (unsigned)__ldg(ei + eb + lane) : 0u;
            double x = xdef, y = 0.0;
            if (valid) adj_ld<PRE>(ex, eb + lane, x, y);
            if (adj_group<KIND, PRE>(en, ei, ex, eb, s1, lane, ii, x, y, D, ft, gs) && gs > 0.0) lam[ii & 0x7fffu] += sgn * gs;
        }
    }
}

// CL: the CTAs of a thread-block cluster share a column -- CTA r keeps chunk r's intensities in its shared memory for the whole column,
// partial sums are exchanged through distributed shared memory, one cluster barrier per batch.  Without CL a single CTA owns the
// column and, when it has several chunks, streams them through shared memory once per batch (intensities in global memory in between).
template <int KIND, int PRE, bool CL> __global__ void __launch_bounds__(ADJ_THREADS, 1) k_adj_sweep(const AdjSweepArgs a) {
    typedef typename EntryOf<KIND>::type E;
    extern __shared__ __align__(16) double lam_s[];  // [chunk_max] intensities of the resident chunk | adjacency bits of the column
    __shared__ FastTables s_ft;
    __shared__ double s_part[2][ADJ_VW], s_pmax[2][ADJ_VW];                                // [batch parity][warp]: this CTA's partial sums, largest contributions
    __shared__ double s_cl[2][ADJ_CLUSTER_MAX][32], s_cm[2][ADJ_CLUSTER_MAX][32];  // [batch parity][source CTA][bucket of the batch]: the same, cluster-wide
    __shared__ double s_dec[2][4][32];                                             // [batch parity][W Mn, logit rho, u, logit u][bucket of the batch]
    __shared__ int s_col;
    fast_tables_load(&s_ft);
    const FastTables *ft = &s_ft;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.K, brow = 2 * K + 1;
    unsigned *s_ab = reinterpret_cast<unsigned *>(lam_s + a.chunk_max);  // [(K + 31) / 32]
    const int abw = (K + 31) >> 5;
    const unsigned crank = CL ? cluster_ctarank() : 0u, csize = CL ? cluster_nctarank() : 1u;
    const int ncl = CL ? (int)(gridDim.x / csize) : (int)gridDim.x, cid = CL ? (int)(blockIdx.x / csize) : (int)blockIdx.x;
    unsigned n_steps = 0, n_batches = 0, n_flips = 0, n_redo = 0, parity = 0;
    // Batch size policy: with a flip probability f per step a batch of S buckets costs c0 + S c1 and gets (1 - (1-f)^S) / f steps accepted,
    // which is cheapest near S ~ 2 / sqrt(f) for the measured c0 / c1 ~ 2; f is an exponentially weighted estimate carried across columns
    // (the same arithmetic in every CTA of a cluster, so they agree on S).
    float fw_steps = 64.f, fw_flips = 64.f * fmaxf(4.f / (float)(a.s0 * a.s0) - 1e-3f, 0.f);
    int S = a.s0;
    (void)ncl; (void)cid;
    for (;;) {
        // dynamic scheduling, longest columns first (a.corder): a CTA, or the first CTA of a cluster for all of its cluster, takes the
        // next column
        __syncthreads();
        if (CL) {
            if (crank == 0 && tid == 0) {
                const int nx = atomicAdd(a.next, 1);
                for (unsigned r = 0; r < csize; r++) st_cluster_u32(&s_col, r, nx);
            }
            cluster_sync_all();
        } else {
            if (tid == 0) s_col = atomicAdd(a.next, 1);
            __syncthreads();
        }
        const int ci = s_col;
        if (ci >= a.ncols) break;
        const int c = a.corder ? a.corder[ci] : a.col_begin + ci * a.col_stride;
        const int e0 = a.node_ptr[c], ne = a.node_ptr[c + 1] - e0;
        const int v0 = a.vstart[c], G = a.vstart[c + 1] - v0;  // CL: G == cluster size
        const int csz = adj_chunk_size(ne, G);
        const int g_lo = CL ? (int)crank : 0, g_hi = CL ? (int)crank + 1 : G;
        const bool resident = CL || G == 1;
        const E *col = reinterpret_cast<const E *>(a.table_w) + (size_t)c * K;
        // lower bound of every intensity of the column without a parent's share: one value per column, so that the CTAs of a
        // cluster certify alike
        const double lam0 = a.lam0min ? a.lam0min[c] : a.lambda0[c];
        double *lamg = a.lam + e0;
        double *Acol = a.A + (size_t)K * c;
        __syncthreads();
        // adjacency bits of the column
        for (int w = warp; w < abw; w += ADJ_THREADS / 32) {
            const int p = w * 32 + lane;
            const unsigned m = __ballot_sync(0xffffffffu, p < K && Acol[p] != 0.0);
            if (lane == 0) s_ab[w] = m;
        }
        // bucket offsets of the resident chunk: every phase starts from them (a slot's section bounds, a flip's bucket, the prefetch
        // targets), and the stream of pair records leaves nothing of this array in L2 -- from shared memory when there is room
        const int *bo_res = a.boff + (int64_t)(v0 + g_lo) * brow;
        if (a.bo_smem && resident) {
            int *s_bo = reinterpret_cast<int *>(s_ab + ((abw + 3) & ~3));
            for (int e = tid; e < brow; e += ADJ_THREADS) s_bo[e] = __ldg(bo_res + e);
            bo_res = s_bo;  // visible behind the barrier that follows the intensities' initialisation
        }
        // ---- current intensities: the baseline rates + the links that are on
        for (int g = g_lo; g < g_hi; g++) {
            const int len = max(0, min(csz, ne - g * csz));
            if (a.lam0bn) for (int e = tid; e < len; e += ADJ_THREADS) lam_s[e] = __ldg(a.lam0bn + e0 + (size_t)g * csz + e);
            else for (int e = tid; e < len; e += ADJ_THREADS) lam_s[e] = lam0;
            __syncthreads();
            const int *bo = resident ? bo_res : a.boff + (int64_t)(v0 + g) * brow;
            const int64_t vb = a.vbase[v0 + g];
            const unsigned short *ei = a.ent_i + vb;
            const double *ex = a.ent_x + (PRE ? 2 : 1) * vb;
            // the links that are on, listed (the exchange buffers are idle here) so that the buckets of the links ahead can be pulled into L2
            // (the half the peers do not write before the next cluster barrier: they fill [parity] at the end of their first batch)
            int *s_on = reinterpret_cast<int *>(&s_cl[parity ^ 1u][0][0]);
            constexpr int ON_CAP = (int)(sizeof(s_cl) / 2 / sizeof(int));
            for (int w0 = 0; w0 < abw;) {
                int non = 0, w1 = w0;
                for (; w1 < abw && non + __popc(s_ab[w1]) <= ON_CAP; w1++) non += __popc(s_ab[w1]);  // block-uniform
                if (tid < w1 - w0) {
                    int o = 0;
                    for (int w = w0; w < w0 + tid; w++) o += __popc(s_ab[w]);
                    for (unsigned bits = s_ab[w0 + tid]; bits; bits &= bits - 1) s_on[o++] = (w0 + tid) * 32 + __ffs(bits) - 1;
                }
                __syncthreads();
                // A link's step is short (a bucket holds about one entry per thread), so the buckets ADJ_INIT_PF links ahead are on their way
                // to L2 -- two ahead would arrive behind their turn -- and the table entries of all listed links start at once
                for (int j = tid; j < non; j += ADJ_THREADS) asm volatile("prefetch.global.L2 [%0];" ::"l"(col + s_on[j]));
                for (int r = 1; r < min(ADJ_INIT_PF, non); r++) adj_pf_range<PRE>(ei, ex, bo[2 * s_on[r]], bo[2 * s_on[r] + 2], tid);
                for (int j = 0; j < non; j++) {
                    if (j + ADJ_INIT_PF < non) { const int pp = s_on[j + ADJ_INIT_PF]; adj_pf_range<PRE>(ei, ex, bo[2 * pp], bo[2 * pp + 2], tid); }
                    const int p = s_on[j];
                    const int b0 = bo[2 * p], bm = bo[2 * p + 1], b1 = bo[2 * p + 2];
                    if (b1 != b0) {
                        const E en = load_entry(col + p);
                        adj_apply<KIND, PRE>(en, ei, ex, b0, bm, bm, b1, warp, lane, 1.0, lam_s, a.D, ft);  // one head per event and bucket
                    }
                    __syncthreads();  // the next parent may touch the same events
                }
                w0 = w1;
            }
            if (!resident) {
                for (int e = tid; e < len; e += ADJ_THREADS) lamg[(size_t)g * csz + e] = lam_s[e];
                __syncthreads();
            }
        }
        // ---- K Bernoulli steps in speculative batches
        int p = 0;
        while (p < K) {
            const int Sc = min(S, K - p);
            const int lg = 31 - __clz(S);
            const int nsub = ADJ_VW >> lg;  // slots per bucket: slot vw works on bucket vw & (S - 1), share vw >> lg
            // the deciding lanes fetch their inputs before the batch so that the latency hides behind it
            // (into shared memory: every warp takes the decisions for itself behind the batch's one barrier)
            if (warp == 0 && lane < Sc) {
                double d0, d1, d2, d3;
                const double *dp = reinterpret_cast<const double *>(a.dec + ((p + lane) + (int64_t)K * c));
                asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(d0), "=d"(d1), "=d"(d2), "=d"(d3) : "l"(dp));
                s_dec[parity][0][lane] = d0; s_dec[parity][1][lane] = d1; s_dec[parity][2][lane] = d2; s_dec[parity][3][lane] = d3;
            }
            // lane = bucket: the state of its link now (warp 0 changes the bits while slower warps still take their decisions)
            const bool old_on = lane < Sc && ((s_ab[(p + lane) >> 5] >> ((p + lane) & 31)) & 1u);
            if (S <= 4 && resident) {
                // short batches are latency bound: pull the entries of the buckets that can come next (they follow in memory) into L2 now
                const int g = g_lo;
                const int *bo = bo_res;
                const int q0 = min(p + Sc, K), q1 = min(p + Sc + 2 * S + 2, K);
                const int64_t vb = a.vbase[v0 + g];
                const int f0 = bo[2 * q0], f1 = bo[2 * q1];
                adj_pf_range<PRE>(a.ent_i + vb, a.ent_x + (PRE ? 2 : 1) * vb, f0, f1, tid);
            }
            constexpr int NR = ADJ_VW / (ADJ_THREADS / 32);  // slots per warp, taken one after the other
            double acc[NR], gmx[NR];
#pragma unroll
            for (int r = 0; r < NR; r++) { acc[r] = 0.0; gmx[r] = 0.0; }
            for (int g = g_lo; g < g_hi; g++) {
                if (!resident) {
                    const int len = max(0, min(csz, ne - g * csz));
                    __syncthreads();
                    for (int e = tid; e < len; e += ADJ_THREADS) lam_s[e] = __ldcg(lamg + (size_t)g * csz + e);  // written by this CTA: read through L2
                    __syncthreads();
                }
                const int *bo = resident ? bo_res : a.boff + (int64_t)(v0 + g) * brow;
                const int64_t vb = a.vbase[v0 + g];
                const unsigned short *ei = a.ent_i + vb;
                const double *ex = a.ent_x + (PRE ? 2 : 1) * vb;
                const AdjPf pf = adj_pf_setup<PRE>(ei, ex, lane);
#pragma unroll
                for (int r = 0; r < NR; r++) {
                    const int vw = warp + r * (ADJ_THREADS / 32);
                    const int qi = vw & (S - 1), sub = vw >> lg, q = p + qi;
                    if (qi < Sc) {
                        const E en = load_entry(col + q);
                        const bool on = (s_ab[q >> 5] >> (q & 31)) & 1u;
                        const double onf = on ? 1.0 : 0.0, floor_ = on ? lam0 : -__longlong_as_double(0x7ff0000000000000LL);
                        const int b0 = bo[2 * q], bm = bo[2 * q + 1], b1 = bo[2 * q + 2];
                        if (q + Sc < K) {  // the bucket this slot takes if the whole batch is accepted: its first blocks go to L2 now
                            const int nb = bo[2 * (q + Sc)] + sub * 64;
                            adj_pf(pf, nb); adj_pf(pf, nb + nsub * 64);
                            if (lane == 31) asm volatile("prefetch.global.L2 [%0];" ::"l"(col + q + Sc));  // and its table entry
                        }
                        AdjAcc A;
                        acc_init(A);
                        if (on) {  // warp-uniform
                            adj_singles<KIND, PRE, true>(en, ei, ex, b0 + sub * 64, bm, nsub * 64, lane, floor_, a.D, lam_s, ft, pf, A);
                            adj_runs<KIND, PRE, true>(en, ei, ex, bm + sub * 32, b1, nsub * 32, lane, floor_, a.D, lam_s, ft, A);
                        } else {
                            adj_singles<KIND, PRE, false>(en, ei, ex, b0 + sub * 64, bm, nsub * 64, lane, floor_, a.D, lam_s, ft, pf, A);
                            adj_runs<KIND, PRE, false>(en, ei, ex, bm + sub * 32, b1, nsub * 32, lane, floor_, a.D, lam_s, ft, A);
                        }
                        if (__all_sync(0xffffffffu, acc_in_range(A))) {
                            acc[r] += (fast_log_n(A.num, ft) - fast_log_n(A.den, ft)) + (double)A.bal * 0.6931471805599453;
                            if (A.gm > 0) gmx[r] = fmax(gmx[r], __hiloint2double(A.gm + 1, 0));  // upper bound of the largest contribution
                        } else {  // warp-uniform, rare
                            const double2 d0 = adj_direct<KIND, PRE>(en, ei, ex, b0 + sub * 64, bm, nsub * 64, lane, onf, floor_, a.D, lam_s, ft);  // the same blocks, half by half
                            const double2 d1 = adj_direct<KIND, PRE>(en, ei, ex, b0 + sub * 64 + 32, bm, nsub * 64, lane, onf, floor_, a.D, lam_s, ft);
                            const double2 d2 = adj_direct<KIND, PRE>(en, ei, ex, bm + sub * 32, b1, nsub * 32, lane, onf, floor_, a.D, lam_s, ft);
                            acc[r] += d0.x + d1.x + d2.x;
                            gmx[r] = fmax(gmx[r], fmax(d0.y, fmax(d1.y, d2.y)));
                        }
                    }
                }
            }
#pragma unroll
            for (int r = 0; r < NR; r++) {
                acc[r] = warp_sum(acc[r]);
                {   // largest contribution of the warp: the values are >= 0 and only serve as upper bounds, so the maximum is taken over the
                    // high words (rounded up): one integer warp reduction instead of a butterfly of FP64 maxima
                    const int hw = __double2hiint(gmx[r]) + (__double2loint(gmx[r]) != 0 ? 1 : 0);
                    gmx[r] = __hiloint2double(__reduce_max_sync(0xffffffffu, hw), 0);
                }
            }
            // One barrier per batch.  With one slot per bucket (S = 32) the warp sends its sums straight to every CTA of the cluster; the
            // buffers alternate with the batch parity (a CTA or warp that runs ahead writes the other half).
            if (CL && nsub == 1) {
                if (lane == 0) {
#pragma unroll
                    for (int r = 0; r < NR; r++) {
                        const int qi = warp + r * (ADJ_THREADS / 32);
                        if (qi < Sc)
                            for (unsigned rk = 0; rk < csize; rk++) { st_cluster_f64(&s_cl[parity][crank][qi], rk, acc[r]); st_cluster_f64(&s_cm[parity][crank][qi], rk, gmx[r]); }
                    }
                }
                cluster_sync_all();
            } else {
                if (lane == 0) {
#pragma unroll
                    for (int r = 0; r < NR; r++) { s_part[parity][warp + r * (ADJ_THREADS / 32)] = acc[r]; s_pmax[parity][warp + r * (ADJ_THREADS / 32)] = gmx[r]; }
                }
                __syncthreads();
                if (CL) {  // this CTA's share of every bucket of the batch goes to all CTAs of the cluster
                    if (warp == 0 && lane < Sc) {
                        double mine = 0.0, mmax = 0.0;
                        for (int s = 0; s < nsub; s++) { mine += s_part[parity][lane + (s << lg)]; mmax = fmax(mmax, s_pmax[parity][lane + (s << lg)]); }
                        for (unsigned r = 0; r < csize; r++) { st_cluster_f64(&s_cl[parity][crank][lane], r, mine); st_cluster_f64(&s_cm[parity][crank][lane], r, mmax); }
                    }
                    cluster_sync_all();
                }
            }
            int stop;
            unsigned fm, onm;
            {   // the decisions of the batch, taken by every warp alike (lane = bucket)
                const bool have = lane < Sc;
                double sum = 0.0, gmax = 0.0;  // log-intensity difference of the bucket; largest change a flip of its link makes to any intensity
                if (have) {
                    if (CL) for (unsigned r = 0; r < csize; r++) { sum += s_cl[parity][r][lane]; gmax = fmax(gmax, s_cm[parity][r][lane]); }  // fixed order: every CTA decides alike
                    else for (int s = 0; s < nsub; s++) { sum += s_part[parity][lane + (s << lg)]; gmax = fmax(gmax, s_pmax[parity][lane + (s << lg)]); }
                }
                const double d_wmn = s_dec[parity][0][lane], d_lrho = s_dec[parity][1][lane], d_u = s_dec[parity][2][lane];
                const double d_lu = s_dec[parity][3][lane];  // logit(u): delta - logit(u) is the margin by which the decision u <= sigmoid(delta) holds
                const int qq = p + lane;
                // ll1 - ll0 (continuous.jl:477-483): integrated-intensity difference, log-intensity difference, prior
                const double delta = -d_wmn + sum + d_lrho;
                // rand(Bernoulli(p1)) = rand() <= p1 with p1 = sigmoid(delta).  u <= sigmoid(delta) <=> logit(u) <= delta, and the two sides
                // are known to ~1e-14, so a clear margin decides without the exp and the division; a close call takes the reference's form
                const double margin = fabs(delta - d_lu);
                bool new_on = d_lu <= delta;
                if (__any_sync(0xffffffffu, have && !(margin > 1e-6 * (1.0 + fabs(delta))))) {  // warp-uniform, rare
                    double p1 = delta >= 0.0 ? 1.0 / (1.0 + exp(-delta)) : exp(delta) / (1.0 + exp(delta));
                    if (delta != delta) p1 = 0.0;
                    new_on = d_u <= p1;
                }
                if (have && delta != delta) atomicOr(a.flag, 64);
                const unsigned flipmask = __ballot_sync(0xffffffffu, have && new_on != old_on);
                // Certified speculation.  The sums of this batch were taken with the intensities as they stood at its start.  A flip of
                // bucket j moves the intensity of every event by at most gmax_j: up when the link goes on, down when it goes off.  A term
                // of a later bucket is f(b) = log(1 + g / b) with b >= lambda0 its intensity without that bucket's parent (lambda0: the
                // column's smallest baseline rate lambda0min_c for a grid baseline, the same in every CTA of a cluster), and for r >= 1
                // log(1 + r x) <= r log(1 + x) (Bernoulli), so with b' the intensity after the flips
                //   b' <  b:  f(b') <= (b / b') f(b) <= (1 + off / lambda0) f(b),      off = sum of gmax over the accepted flips that went off
                //   b' >= b:  f(b') >= (b / b') f(b) >= f(b) / (1 + on / lambda0),     on  = ... that went on
                // for ANY size of the change.  The later sum S (>= 0) therefore ends up in [S / (1 + on / lambda0), S (1 + off / lambda0)]:
                // a decision "off" (delta < logit u) can only be overturned by the upper end, a decision "on" only by the lower end.
                // A decision whose margin |delta - logit(u)| exceeds its side's bound (plus rounding slack) is the decision the sequential
                // sweep takes; the batch is accepted up to the first bucket that cannot be certified, and restarts there.
                // on / off = exclusive prefix sums over the flips (warp scan: the same values in every CTA of the cluster).
                // (The first version used one symmetric bound, 4 S cum / lambda0 from the derivative, valid only while cum <= lambda0 / 2,
                // so every larger flip ended its batch; DESIGN.md §3.3.)
                const bool flip = (flipmask >> lane) & 1u;
                double inc_on = (flip && new_on) ? gmax : 0.0, inc_off = (flip && !new_on) ? gmax : 0.0;
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) {
                    const double t1 = __shfl_up_sync(0xffffffffu, inc_on, d), t0 = __shfl_up_sync(0xffffffffu, inc_off, d);
                    if (lane >= d) { inc_on += t1; inc_off += t0; }
                }
                double cum_on = __shfl_up_sync(0xffffffffu, inc_on, 1), cum_off = __shfl_up_sync(0xffffffffu, inc_off, 1);
                if (lane == 0) { cum_on = 0.0; cum_off = 0.0; }
                const double slack = 1e-7 + 1e-10 * fabs(delta);
                const double S_ = fabs(sum);
                // (1.0000001: the scan's own rounding, so that the bound stays an upper bound)
                const double shift = new_on ? S_ * (cum_on / (lam0 + cum_on)) : S_ * (cum_off / lam0);
                const bool uncertified = have && (cum_on > 0.0 || cum_off > 0.0) && !(margin > 1.0000001 * shift + slack);
                const unsigned um = __ballot_sync(0xffffffffu, uncertified);
                stop = Sc;
                if (um) stop = min(stop, __ffs(um) - 1);
                fm = stop >= 32 ? flipmask : (flipmask & ((1u << stop) - 1u));
                onm = __ballot_sync(0xffffffffu, new_on);
                // warp 0 records the accepted flips; the others see the new bits behind the barrier of the first flip's application
                if (warp == 0 && have && ((fm >> lane) & 1u)) {
                    if (crank == 0) Acol[qq] = new_on ? 1.0 : 0.0;
                    atomicXor(&s_ab[qq >> 5], 1u << (qq & 31));
                }
            }
            parity ^= 1u;
            n_batches++;
            n_steps += stop; n_flips += __popc(fm); n_redo += Sc - stop;
            if (resident && (fm & (fm - 1))) {  // several flips: all their buckets start towards L2 now, the first one's latency covers the others
                const int *bo = bo_res;
                const int64_t vb = a.vbase[v0 + g_lo];
                for (unsigned f2 = fm & (fm - 1); f2; f2 &= f2 - 1) {
                    const int qf = p + __ffs(f2) - 1;
                    const int f0 = bo[2 * qf], f1 = bo[2 * qf + 2];
                    adj_pf_range<PRE>(a.ent_i + vb, a.ent_x + (PRE ? 2 : 1) * vb, f0, f1, tid);
                }
            }
            while (fm) {
                // the link of bucket qf flipped: move its contribution into / out of the intensities
                const int j = __ffs(fm) - 1;
                fm &= fm - 1;
                const int qf = p + j;
                const double sgn = ((onm >> j) & 1u) ? 1.0 : -1.0;
                const E enf = load_entry(col + qf);
                for (int g = g_lo; g < g_hi; g++) {
                    const int *bo = resident ? bo_res : a.boff + (int64_t)(v0 + g) * brow;
                    const int b0 = bo[2 * qf], bm = bo[2 * qf + 1], b1 = bo[2 * qf + 2];
                    const int64_t vb = a.vbase[v0 + g];
                    const unsigned short *ei = a.ent_i + vb;
                    const double *ex = a.ent_x + (PRE ? 2 : 1) * vb;
                    adj_apply<KIND, PRE>(enf, ei, ex, b0, bm, bm, b1, warp, lane, sgn, resident ? lam_s : lamg + (size_t)g * csz, a.D, ft);
                }
                __syncthreads();  // the next flipped bucket may touch the same events
            }
            p += stop;
            fw_steps = 0.9f * fw_steps + (float)stop; fw_flips = 0.9f * fw_flips + (stop < Sc ? 1.f : 0.f);  // "flip" = a batch cut short
            {
                const float target = 2.f * rsqrtf(fw_flips / fw_steps + 1e-3f);
                const int l2 = min(ADJ_SMAX_LOG2, max(0, __float2int_rn(__log2f(target))));
                S = 1 << l2;
            }
        }
    }
    if (tid == 0 && crank == 0 && a.stat) {
        atomicAdd(a.stat + 0, (unsigned long long)n_steps); atomicAdd(a.stat + 1, (unsigned long long)n_batches);
        atomicAdd(a.stat + 2, (unsigned long long)n_flips); atomicAdd(a.stat + 3, (unsigned long long)n_redo);
    }
}

// ---------------------------------------------------------------------------------------
// log-likelihood of a network process from the cached structure
// ---------------------------------------------------------------------------------------
// lambda_i = lambda0 + sum over the links that are ON of the bucket's contributions: with the pairs already bucketed by
// (child column, parent node) a sparse network touches only the buckets of its active links -- 5 % of the structure at config 4
// (5.8 GB instead of 64 probes per event over the whole stream).  One CTA per virtual column (chunks are independent here), the
// chunk's intensities in shared memory, buckets applied one after the other (two ahead prefetched to L2), then sum log lambda in
// a fixed order.  The compensator comes from the per-node counts as in the window sweeps.
struct AdjLoglikArgs {
    const int *node_ptr; int K; const void *table; const double *lambda0; const uint32_t *abits; int words; double D;
    const double *lam0bn;  // grid baseline: per-event rates in by-node order (NULL: lambda0)
    const int *vstart, *vnode; const int64_t *vbase; const int *boff; const unsigned short *ent_i; const double *ent_x;
    int nv, chunk_max; double *partials; int *flag;
    int cap;   // links whose section bounds are staged in shared memory per round (0: read from global memory)
};
template <int KIND, int PRE> __global__ void __launch_bounds__(ADJ_THREADS, 1) k_adj_loglik(const AdjLoglikArgs a) {
    typedef typename EntryOf<KIND>::type E;
    extern __shared__ __align__(16) double lam_s[];  // [chunk_max] intensities | [K] active parents of the column
    __shared__ FastTables s_ft;
    __shared__ double s_red[ADJ_THREADS / 32];
    __shared__ int s_non;
    fast_tables_load(&s_ft);
    const FastTables *ft = &s_ft;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int K = a.K, brow = 2 * K + 1;
    int *s_on = reinterpret_cast<int *>(lam_s + a.chunk_max);
    double total = 0.0;  // thread 0: this CTA's running sum (static round-robin over the virtual columns: a fixed order)
    for (int v = blockIdx.x; v < a.nv; v += gridDim.x) {
        const int c = a.vnode[v], g = v - a.vstart[c], G = a.vstart[c + 1] - a.vstart[c];
        const int ne = a.node_ptr[c + 1] - a.node_ptr[c], csz = adj_chunk_size(ne, G);
        const int len = max(0, min(csz, ne - g * csz));
        const double lam0 = a.lambda0[c];
        const double *rate = a.lam0bn ? a.lam0bn + a.node_ptr[c] + (size_t)g * csz : nullptr;  // the chunk's baseline rates
        __syncthreads();
        for (int e = tid; e < len; e += ADJ_THREADS) lam_s[e] = rate ? __ldg(rate + e) : lam0;
        if (warp == 0) {  // the column's active parents, in order
            int non = 0;
            const uint32_t *row = a.abits + (size_t)c * a.words;
            for (int w0 = 0; w0 < a.words; w0 += 32) {
                const uint32_t bits = w0 + lane < a.words ? row[w0 + lane] : 0u;
                int x = __popc(bits);
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) { const int y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
                int o = non + x - __popc(bits);
                for (uint32_t b = bits; b; b &= b - 1) { const int p = (w0 + lane) * 32 + __ffs(b) - 1; if (p < K) s_on[o++] = p; }
                non += __shfl_sync(0xffffffffu, x, 31);
            }
            if (lane == 0) s_non = non;
        }
        __syncthreads();
        const int non = s_non;
        const int *bo = a.boff + (int64_t)v * brow;
        const int64_t vb = a.vbase[v];
        const unsigned short *ei = a.ent_i + vb;
        const double *ex = a.ent_x + (PRE ? 2 : 1) * vb;
        const E *col = reinterpret_cast<const E *>(a.table) + (size_t)c * K;
        // The active buckets one after the other.  A bucket holds about one entry per thread, so a link's step is a chain of dependent
        // latencies: the section bounds of up to `cap` links are gathered into shared memory at once (the stream of pair records leaves
        // nothing of the offsets array in L2), their table entries start towards L2 together, and the buckets ADJ_INIT_PF links ahead are
        // prefetched (two ahead arrive behind their turn).
        const int cap = a.cap > 0 ? a.cap : non;
        int *s_b3 = s_on + K;  // [3 cap] when a.cap > 0
        for (int j0 = 0; j0 < non; j0 += max(cap, 1)) {
            const int nj = min(cap, non - j0);
            for (int j = tid; j < nj; j += ADJ_THREADS) {
                const int p = s_on[j0 + j];
                if (a.cap > 0) { s_b3[3 * j] = __ldg(bo + 2 * p); s_b3[3 * j + 1] = __ldg(bo + 2 * p + 1); s_b3[3 * j + 2] = __ldg(bo + 2 * p + 2); }
                asm volatile("prefetch.global.L2 [%0];" ::"l"(col + p));
            }
            if (a.cap > 0) __syncthreads();
            for (int r = 0; r < min(ADJ_INIT_PF, nj); r++) {
                const int p = s_on[j0 + r];
                adj_pf_range<PRE>(ei, ex, a.cap > 0 ? s_b3[3 * r] : bo[2 * p], a.cap > 0 ? s_b3[3 * r + 2] : bo[2 * p + 2], tid);
            }
            for (int j = 0; j < nj; j++) {
                if (j + ADJ_INIT_PF < nj) {
                    const int r = j + ADJ_INIT_PF, p = s_on[j0 + r];
                    adj_pf_range<PRE>(ei, ex, a.cap > 0 ? s_b3[3 * r] : bo[2 * p], a.cap > 0 ? s_b3[3 * r + 2] : bo[2 * p + 2], tid);
                }
                const int p = s_on[j0 + j];
                const int b0 = a.cap > 0 ? s_b3[3 * j] : bo[2 * p], bm = a.cap > 0 ? s_b3[3 * j + 1] : bo[2 * p + 1], b1 = a.cap > 0 ? s_b3[3 * j + 2] : bo[2 * p + 2];
                if (b1 != b0) {
                    const E en = load_entry(col + p);
                    adj_apply<KIND, PRE>(en, ei, ex, b0, bm, bm, b1, warp, lane, 1.0, lam_s, a.D, ft);  // one head per event and bucket
                }
                __syncthreads();  // the next parent may touch the same events (and the next round rewrites the staged bounds)
            }
        }
        double acc = 0.0;
        for (int e = tid; e < len; e += ADJ_THREADS) {
            const double l = lam_s[e];
            if (!(l > 0.0) || l > 1.7976931348623157e308) atomicOr(a.flag, 8);
            acc += fast_log(l, ft);
        }
        acc = warp_sum(acc);
        if (lane == 0) s_red[warp] = acc;
        __syncthreads();
        if (tid == 0) {
            double r = 0.0;
            for (int w = 0; w < ADJ_THREADS / 32; w++) r += s_red[w];
            total += r;
        }
    }
    if (tid == 0) { a.partials[2 * (size_t)blockIdx.x] = total; a.partials[2 * (size_t)blockIdx.x + 1] = 0.0; }
}

// The structure of a handle was built for one model: its payload is read as lags by an Exponential kernel and as the LogitNormal
// terms of its build-time dtmax by the 18-byte kernels, so it serves only a model of the same impulse kind (and dtmax, for that payload).
static bool adj_payload_fits(const nhp_ctx *ctx, const nhp_events *ev) {
    return ev->adj_impulse == ctx->kind && (ev->adj_kind != 1 || ev->adj_D == ctx->dtmax);
}

// Log-likelihood through the cached structure when it exists for this handle and model, covers every column and the horizon, and
// the network is sparse enough that streaming its active buckets beats the window sweep.  Returns 1 when it does not apply.
int nhp_cont_try_adj_loglik(nhp_ctx *ctx, nhp_events *ev, SweepArgs &sa, int *grid_out, int cb, int cs) {  // structure of the columns c % cs == cb: their share
    { const char *e = getenv("NHP_ADJ_LOGLIK"); if (e && atoi(e) == 0) return 1; }
    if (!ctx->has_A || !ev->d_adj_i || ev->adj_cb != cb || ev->adj_cs != cs || ev->n_halo != 0 || ev->adj_cluster < 0) return 1;
    if (!adj_payload_fits(ctx, ev)) return 1;
    if (!(ctx->density <= 0.25) || !(ev->adj_horizon >= sa.horizon) || sa.jmin > 0) return 1;
    if (ctx->kind == NHP_EXPONENTIAL && ev->adj_horizon != sa.horizon && !(sa.horizon < ctx->dtmax)) return 1;  // only a cut-off horizon may be exceeded
    const int64_t K = ctx->K;
    AdjLoglikArgs a;
    a.node_ptr = ev->d_node_ptr; a.K = (int)K; a.table = sa.table; a.lambda0 = sa.lambda0; a.abits = ctx->d_abits; a.words = (int)ctx->abits_words; a.D = ctx->dtmax;
    a.vstart = ev->d_adj_vstart; a.vnode = ev->d_adj_vnode; a.vbase = ev->d_adj_vbase; a.boff = ev->d_adj_boff; a.ent_i = ev->d_adj_i; a.ent_x = ev->d_adj_dt;
    a.nv = (int)ev->adj_nv; a.chunk_max = (ev->adj_chunk_max + 1) & ~1; a.partials = sa.partials; a.flag = sa.flag;
    size_t smem = (size_t)a.chunk_max * sizeof(double) + (size_t)K * sizeof(int) + 16;
    if (smem > (size_t)ctx->smem_optin - 4096) return 1;
    a.cap = 256;  // 3 KB of staged section bounds when they fit next to the intensities
    { const char *e = getenv("NHP_ADJ_LL_STAGE"); if (e && atoi(e) == 0) a.cap = 0; }
    if (smem + 3 * (size_t)a.cap * sizeof(int) > (size_t)ctx->smem_optin - 4096) a.cap = 0;
    smem += 3 * (size_t)a.cap * sizeof(int);
    const double *lam0min = nullptr;  // (the sums of logs need the rates only)
    NHP_TRY(nhp_cont_event_baseline_bynode(ctx, ev, &a.lam0bn, &lam0min));
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    const int grid = (int)std::min<int64_t>(ev->adj_nv, ctx->sm_count);
    if (ctx->kind == NHP_EXPONENTIAL) {
        NHP_CUDA(ctx, cudaFuncSetAttribute(k_adj_loglik<NHP_EXPONENTIAL, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_adj_loglik<NHP_EXPONENTIAL, 0><<<grid, ADJ_THREADS, smem, ctx->stream>>>(a);
    } else if (ev->adj_kind == 1) {
        NHP_CUDA(ctx, cudaFuncSetAttribute(k_adj_loglik<NHP_LOGITNORMAL, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_adj_loglik<NHP_LOGITNORMAL, 1><<<grid, ADJ_THREADS, smem, ctx->stream>>>(a);
    } else {
        NHP_CUDA(ctx, cudaFuncSetAttribute(k_adj_loglik<NHP_LOGITNORMAL, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_adj_loglik<NHP_LOGITNORMAL, 0><<<grid, ADJ_THREADS, smem, ctx->stream>>>(a);
    }
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    *grid_out = grid;
    return NHP_OK;
}

// table without the adjacency factor (the sampler needs W h for both values of A[p,c])
__global__ void k_table_noA_ln(int K, const double *__restrict__ W, const double *__restrict__ mu, const double *__restrict__ tau, double D, EntryLN *__restrict__ table) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)K * K) return;
    int cc = (int)(e / K), p = (int)(e % K);
    int64_t src = p + (int64_t)K * cc;
    double tt = tau[src];
    EntryLN en;
    en.cf = W[src] * sqrt(tt) * NHP_INVSQRT2PI * (D * D); en.mu = mu[src]; en.h = 0.5 * tt; en.pad = 0.0;
    table[e] = en;
}
__global__ void k_table_noA_ex(int K, const double *__restrict__ W, const double *__restrict__ theta, EntryEX *__restrict__ table) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)K * K) return;
    int cc = (int)(e / K), p = (int)(e % K);
    int64_t src = p + (int64_t)K * cc;
    EntryEX en;
    en.theta = theta[src]; en.wt = W[src] * en.theta;
    table[e] = en;
}

// Look-back horizon of the sampler.  It evaluates W h for links that are currently off as well, so the Exponential cut-off is
// taken from ALL entries with W != 0 (the sweeps' horizon only looks at the active links).
static double adj_horizon_value(const nhp_ctx *ctx, int64_t n_total) {
    double h = ctx->dtmax;
    if (ctx->kind != NHP_EXPONENTIAL) return h;
    if (ctx->wt_max_all <= 0.0) return std::min(h, 1e-300);
    if (ctx->theta_min_all > 0.0 && std::isfinite(ctx->theta_min_all) && ctx->lambda0_min > 0.0 && n_total > 0) {
        const double cut = log((double)n_total * ctx->wt_max_all / (1e-14 * ctx->lambda0_min)) / ctx->theta_min_all;
        if (cut > 0.0 && cut < h) h = cut;
    }
    return h;
}

// NHP_TIMING=1: wall-clock phases of the structure build on stderr (development aid)
#include <chrono>
struct AdjPhaseTimer {
    bool on; cudaStream_t s; std::chrono::steady_clock::time_point t0;
    AdjPhaseTimer(cudaStream_t st) : on(getenv("NHP_TIMING") && atoi(getenv("NHP_TIMING"))), s(st), t0(std::chrono::steady_clock::now()) {}
    void lap(const char *what) {
        if (!on) return;
        cudaStreamSynchronize(s);
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[nhp timing] %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

#define ADJ_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); } while (0)

static int adj_ensure_ctx(nhp_ctx *ctx) {
    const size_t KK = (size_t)ctx->K * ctx->K;
    if (!ctx->d_adj_tw) ADJ_CUDA(cudaMalloc(&ctx->d_adj_tw, KK * sizeof(EntryLN)));
    if (!ctx->d_adj_rho) ADJ_CUDA(cudaMalloc(&ctx->d_adj_rho, KK * sizeof(double)));
    if (!ctx->d_adj_u) ADJ_CUDA(cudaMalloc(&ctx->d_adj_u, KK * sizeof(double)));
    if (!ctx->d_adj_dec) ADJ_CUDA(cudaMalloc(&ctx->d_adj_dec, KK * sizeof(double4)));
    if (!ctx->d_adj_A) ADJ_CUDA(cudaMalloc(&ctx->d_adj_A, KK * sizeof(double)));
    if (!ctx->d_adj_ctl) ADJ_CUDA(cudaMalloc(&ctx->d_adj_ctl, 8 * sizeof(int)));
    if (!ctx->d_adj_stat) ADJ_CUDA(cudaMalloc(&ctx->d_adj_stat, 8 * sizeof(unsigned long long)));
    return NHP_OK;
}

// (Re)build the cached structure of `ev` for this horizon / column partition.  Returns 1 when it does not fit (uncached sweep).
static int adj_build_structure(nhp_ctx *ctx, nhp_events *ev, double horizon, int cb, int cs, int chunk_cap) {
    const int64_t K = ctx->K, n = ev->n;
    cudaStream_t s = ctx->stream;
    AdjPhaseTimer tm(s);
    nhp_events_free_adjacency(ctx, ev, s);
    tm.lap("free old structure");
    std::vector<double> mn(K);
    ADJ_CUDA(cudaMemcpyAsync(mn.data(), ev->d_Mn, K * sizeof(double), cudaMemcpyDeviceToHost, s));
    ADJ_CUDA(cudaStreamSynchronize(s));
    // Virtual columns.  When the largest owned column fits the shared memory of a thread-block cluster (<= 8 CTAs), EVERY owned
    // column is cut into `cluster` chunks, one per CTA of the cluster that will sweep it; otherwise columns are cut into chunks of at
    // most chunk_cap events and a single CTA streams them.
    int max_col = 0;
    for (int64_t c = cb; c < K; c += cs) max_col = std::max(max_col, (int)mn[c]);
    int cluster = 1;
    while (cluster < ADJ_CLUSTER_MAX && (int64_t)cluster * chunk_cap < max_col) cluster++;
    if ((int64_t)cluster * chunk_cap < max_col) cluster = 0;  // too large for a cluster: single-CTA streaming form
    { const char *e = getenv("NHP_ADJ_CLUSTER"); if (e && atoi(e) == 0) cluster = 0; else if (e && cluster > 0 && atoi(e) > cluster && atoi(e) <= ADJ_CLUSTER_MAX) cluster = atoi(e); }
    std::vector<int> vstart(K + 1), vnode;
    int chunk_max = 1;
    for (int64_t c = 0; c < K; c++) {
        vstart[c] = (int)vnode.size();
        if (c % cs != cb) continue;
        const int ne = (int)mn[c];
        const int G = cluster > 0 ? cluster : std::max(1, (ne + chunk_cap - 1) / chunk_cap);
        chunk_max = std::max(chunk_max, adj_chunk_size(ne, G));
        for (int g = 0; g < G; g++) vnode.push_back((int)c);
    }
    vstart[K] = (int)vnode.size();
    const int64_t nv = (int64_t)vnode.size();
    if (nv == 0) return 1;
    int *d_vstart = nullptr, *d_vnode = nullptr, *d_lo = nullptr;
    unsigned long long *d_vcount = nullptr, *d_pk = nullptr;
    auto drop = [&](int rc) { cudaFreeAsync(d_vstart, s); cudaFreeAsync(d_vnode, s); cudaFreeAsync(d_vcount, s); cudaFreeAsync(d_lo, s); cudaFreeAsync(d_pk, s); return rc; };
#define ADJ_B(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return drop(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__)); } while (0)
    ADJ_B(cudaMallocAsync(&d_vstart, (size_t)(K + 1) * sizeof(int), s));
    ADJ_B(cudaMallocAsync(&d_vnode, (size_t)nv * sizeof(int), s));
    ADJ_B(cudaMallocAsync(&d_vcount, (size_t)nv * sizeof(unsigned long long), s));
    ADJ_B(cudaMallocAsync(&d_lo, std::max<size_t>((size_t)n, 1) * sizeof(int), s));
    ADJ_B(cudaMemsetAsync(ctx->d_adj_ctl, 0, 8 * sizeof(int), s));
    ADJ_B(cudaMemcpyAsync(d_vstart, vstart.data(), (size_t)(K + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
    ADJ_B(cudaMemcpyAsync(d_vnode, vnode.data(), (size_t)nv * sizeof(int), cudaMemcpyHostToDevice, s));
    ADJ_B(cudaMemsetAsync(d_vcount, 0, (size_t)nv * sizeof(unsigned long long), s));
    if (n > 0) {
        k_adj_count<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ev->d_t, ev->d_c, ev->d_order, ev->d_node_ptr, d_vstart, n, horizon, cb, cs, d_vcount, d_lo,
                                                                 ctx->d_adj_ctl + 4, (ev->cache_horizon == horizon && ev->n_halo == 0) ? ev->d_wlen : nullptr);
        NHP_LAUNCHED(ctx);
    }
    tm.lap("virtual columns + count");
    std::vector<unsigned long long> vc(nv);
    int max_win = 0;
    ADJ_B(cudaMemcpyAsync(&max_win, ctx->d_adj_ctl + 4, sizeof(int), cudaMemcpyDeviceToHost, s));
    ADJ_B(cudaMemcpyAsync(vc.data(), d_vcount, (size_t)nv * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    ADJ_B(cudaStreamSynchronize(s));
    // room per virtual column: its pairs plus the padding of its 2 K sections to whole blocks (64 entries: singles) / groups (32: runs) (an upper bound; the regions
    // start on group boundaries so that the sweeps' paired loads are aligned)
    std::vector<int64_t> vbase(nv + 1);
    int64_t tot = 0, pairs = 0;
    for (int64_t v = 0; v < nv; v++) {
        vbase[v] = tot;
        const unsigned long long room = vc[v] + std::min<unsigned long long>(94ull * (unsigned long long)K, 63ull * vc[v]);
        if (room >= 0x7fffffffull) return drop(nhp_fail(ctx, NHP_ERR_UNSUPPORTED, "adjacency sampler: a column chunk has %llu window entries (limit 2^31)", vc[v]));
        pairs += (int64_t)vc[v];
        tot += (int64_t)((room + 31ull) & ~31ull);
    }
    vbase[nv] = tot;
    // room: the structure (10 B per pair, or 18 B with the LogitNormal payload), the bucket offsets, the per-event intensities;
    // a quarter (payload: a third) of the free memory stays free for everything else
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    {   // what the context's block cache and the stream-ordered pool keep for reuse (a freed structure of the previous data set) is available
        cudaMemPool_t pool;
        unsigned long long reserved = 0, used = 0;
        if (cudaDeviceGetDefaultMemPool(&pool, ctx->device) == cudaSuccess &&
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
            free_b += (size_t)(reserved - used);
        free_b += nhp_big_cached_bytes(ctx);
    }
    const size_t fixed = (size_t)nv * (2 * K + 1) * sizeof(int) + (size_t)(nv + 1) * sizeof(int64_t) + (size_t)n * (sizeof(double) + sizeof(unsigned long long));
    bool pre = ctx->kind == NHP_LOGITNORMAL && (double)tot * 18.0 + (double)fixed <= 0.72 * (double)free_b;
    { const char *e = getenv("NHP_ADJ_PRE"); if (e) pre = pre && atoi(e) != 0; }
    const size_t need = (size_t)tot * (pre ? 18 : 10) + fixed;
    // build kernel: [2K+1] section offsets + 2 K CTA-wide cursors (singles, runs); one CTA of 32 warps per SM
    constexpr int nw = 32;
    const bool fits = (size_t)(4 * K + 1) * sizeof(int) + 2048 <= (size_t)ctx->smem_optin;
    // the packed predecessor record holds 20 bits of node and 22 bits of same-node distances: longer windows take the uncached sweep
    if ((double)need > 0.75 * (double)free_b || !fits || K > (1 << ADJ_NODE_BITS) || max_win >= (int)ADJ_LINK_SAT) return drop(1);
    cudaFreeAsync(d_vcount, s); d_vcount = nullptr;
    ADJ_B(cudaMallocAsync(&d_pk, std::max<size_t>((size_t)n, 1) * sizeof(unsigned long long), s));
    if (n > 0) {
        k_adj_links<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ev->d_order, ev->d_node_ptr, ev->d_c, n, d_pk);
        NHP_LAUNCHED(ctx);
    }
    ev->d_adj_vstart = d_vstart; ev->d_adj_vnode = d_vnode; d_vstart = d_vnode = nullptr;  // owned by the handle from here on
    auto fail = [&](int rc) { cudaFreeAsync(d_lo, s); cudaFreeAsync(d_pk, s); nhp_events_free_adjacency(ctx, ev, s); return rc; };
#define ADJ_S(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__)); } while (0)
    ADJ_S(cudaMallocAsync(&ev->d_adj_vbase, (size_t)(nv + 1) * sizeof(int64_t), s));
    ADJ_S(cudaMallocAsync(&ev->d_adj_boff, (size_t)nv * (2 * K + 1) * sizeof(int), s));
    const size_t slack = 64 * 1024;  // entries: the sweeps' L2 prefetches run a few blocks ahead of the block they read
    ev->adj_bytes_i = ((size_t)tot + slack) * sizeof(unsigned short);
    ev->adj_bytes_dt = ((size_t)tot + slack) * (pre ? 2 : 1) * sizeof(double);
    ev->d_adj_i = (unsigned short *)nhp_big_alloc(ctx, ev->adj_bytes_i);
    ev->d_adj_dt = (double *)nhp_big_alloc(ctx, ev->adj_bytes_dt);
    if (!ev->d_adj_i || !ev->d_adj_dt) return fail(nhp_fail(ctx, NHP_ERR_CUDA, "adjacency sampler: cannot allocate %.1f GB for the cached pair structure", 1e-9 * (double)(ev->adj_bytes_i + ev->adj_bytes_dt)));
    ADJ_S(cudaMallocAsync(&ev->d_adj_lam, std::max<size_t>((size_t)n, 1) * sizeof(double), s));
    tm.lap("links + allocation");
    ADJ_S(cudaMemcpyAsync(ev->d_adj_vbase, vbase.data(), (size_t)(nv + 1) * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    // Order of the build: time slice by time slice -- the CTAs that run together then work on the same stretch of the stream for
    // different columns and move through it at the same pace, so a window is fetched from HBM once and served from L2 to the others
    // (column by column they sat in different quarters of the stream: 373 GB read for 156 GB of input).
    std::vector<int> vorder((size_t)nv);
    {
        std::vector<std::pair<double, int>> key((size_t)nv);
        for (int64_t c = 0; c < K; c++) {
            const int G = vstart[c + 1] - vstart[c];
            for (int g = 0; g < G; g++) key[(size_t)vstart[c] + g] = std::make_pair((double)g / (double)G, vstart[c] + g);
        }
        std::stable_sort(key.begin(), key.end(), [](const std::pair<double, int> &a, const std::pair<double, int> &b) { return a.first < b.first; });
        for (int64_t v = 0; v < nv; v++) vorder[(size_t)v] = key[(size_t)v].second;
    }
    {   // sweep order of the owned columns: most child events first (longest-processing-time scheduling of the clusters)
        std::vector<int> co;
        for (int64_t c = cb; c < K; c += cs) co.push_back((int)c);
        std::stable_sort(co.begin(), co.end(), [&](int x, int y) { return mn[x] > mn[y]; });
        ADJ_S(cudaMallocAsync(&ev->d_adj_corder, std::max<size_t>(co.size(), 1) * sizeof(int), s));
        ADJ_S(cudaMemcpyAsync(ev->d_adj_corder, co.data(), co.size() * sizeof(int), cudaMemcpyHostToDevice, s));
        ADJ_S(cudaStreamSynchronize(s));
    }
    int *d_vorder = nullptr;
    ADJ_S(cudaMallocAsync(&d_vorder, (size_t)nv * sizeof(int), s));
    ADJ_S(cudaMemcpyAsync(d_vorder, vorder.data(), (size_t)nv * sizeof(int), cudaMemcpyHostToDevice, s));
    ADJ_S(cudaMemsetAsync(ctx->d_adj_ctl, 0, 8 * sizeof(int), s));
    AdjBuildArgs b;
    b.t = ev->d_t; b.pk = d_pk; b.lo = d_lo; b.order = ev->d_order; b.node_ptr = ev->d_node_ptr; b.K = (int)K; b.D = ctx->dtmax;
    b.vstart = ev->d_adj_vstart; b.vnode = ev->d_adj_vnode; b.vorder = d_vorder; b.vbase = ev->d_adj_vbase; b.boff = ev->d_adj_boff; b.ent_i = ev->d_adj_i; b.ent_x = ev->d_adj_dt;
    b.pre = pre ? 1 : 0;
    b.nv = (int)nv; b.nw = nw; b.next = ctx->d_adj_ctl; b.flag = ctx->d_flag;
    const size_t bsmem = (size_t)(4 * K + 1) * sizeof(int);
    ADJ_S(cudaFuncSetAttribute(k_adj_build, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(bsmem, 1024)));
    int per_sm = 1;
    ADJ_S(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_adj_build, nw * 32, bsmem));
    const int grid = (int)std::min<int64_t>(nv, (int64_t)ctx->sm_count * std::max(per_sm, 1));
    cudaEvent_t b0, b1;
    ADJ_S(cudaEventCreate(&b0)); ADJ_S(cudaEventCreate(&b1));
    cudaEventRecord(b0, s);
    k_adj_build<<<grid, nw * 32, bsmem, s>>>(b);
    NHP_LAUNCHED(ctx);
    cudaEventRecord(b1, s);
    int flag = 0;
    ADJ_S(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    ADJ_S(cudaStreamSynchronize(s));
    ADJ_S(cudaGetLastError());
    float bms = 0.f;
    cudaEventElapsedTime(&bms, b0, b1);
    cudaEventDestroy(b0); cudaEventDestroy(b1);
    tm.lap("build kernel");
    cudaFreeAsync(d_lo, s); cudaFreeAsync(d_pk, s); cudaFreeAsync(d_vorder, s); d_lo = nullptr; d_pk = nullptr;
    tm.lap("free temporaries");
    if (flag & 128) return fail(nhp_fail(ctx, NHP_ERR_CUDA, "adjacency sampler: structure build disagrees with its own count (internal error)"));
    ev->adj_total = tot; ev->adj_pairs = pairs; ev->adj_nv = nv; ev->adj_horizon = horizon; ev->adj_cb = cb; ev->adj_cs = cs;
    ev->adj_chunk_cap = chunk_cap; ev->adj_chunk_max = chunk_max; ev->adj_cluster = cluster; ev->adj_kind = pre ? 1 : 0;
    ev->adj_impulse = ctx->kind; ev->adj_D = ctx->dtmax;
    ctx->adj_info[7] = bms;
    return NHP_OK;
#undef ADJ_B
#undef ADJ_S
}

// the uncached sweep: per-call scratch, re-bucketing inside the kernel
static int adj_run_uncached(nhp_ctx *ctx, nhp_events *ev, double horizon, const double *d_rho, const double *d_u, uint64_t seed, uint64_t counter,
                            double *d_A, int cb, int cs, const double *lam0bn, const double *lam0min) {
    const int64_t K = ctx->K, n = ev->n;
    cudaStream_t s = ctx->stream;
    unsigned long long *d_cc = nullptr;
    int *d_vstart = nullptr;
    int *d_ent_i = nullptr; double *d_ent_v = nullptr, *d_lam = nullptr, *d_gacc = nullptr;
    auto fin = [&](int rc) {
        cudaStreamSynchronize(s);
        cudaFree(d_cc); cudaFree(d_vstart); cudaFree(d_ent_i); cudaFree(d_ent_v); cudaFree(d_lam); cudaFree(d_gacc);
        return rc;
    };
#define ADJ_U(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fin(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__)); } while (0)
    // per-column window totals size the buckets: one "virtual column" per column
    std::vector<int> vstart(K + 1);
    for (int64_t c = 0; c <= K; c++) vstart[c] = (int)c;
    ADJ_U(cudaMalloc(&d_cc, (size_t)K * sizeof(unsigned long long)));
    ADJ_U(cudaMalloc(&d_vstart, (size_t)(K + 1) * sizeof(int)));
    ADJ_U(cudaMemcpyAsync(d_vstart, vstart.data(), (size_t)(K + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
    ADJ_U(cudaMemsetAsync(d_cc, 0, (size_t)K * sizeof(unsigned long long), s));
    if (n > 0) {
        k_adj_count<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(ev->d_t, ev->d_c, ev->d_order, ev->d_node_ptr, d_vstart, n, horizon, 0, 1, d_cc, nullptr, nullptr, nullptr);
        NHP_LAUNCHED(ctx);
    }
    std::vector<unsigned long long> cc(K);
    std::vector<double> mn(K);
    ADJ_U(cudaMemcpyAsync(cc.data(), d_cc, K * sizeof(unsigned long long), cudaMemcpyDeviceToHost, s));
    ADJ_U(cudaMemcpyAsync(mn.data(), ev->d_Mn, K * sizeof(double), cudaMemcpyDeviceToHost, s));
    ADJ_U(cudaStreamSynchronize(s));
    int64_t cap = 1, mc = 1;
    for (int64_t k = 0; k < K; k++) { cap = std::max<int64_t>(cap, (int64_t)cc[k]); mc = std::max<int64_t>(mc, (int64_t)mn[k]); }
    if (cap >= (int64_t)0x3fffffff) return fin(nhp_fail(ctx, NHP_ERR_UNSUPPORTED, "adjacency sampler: a column has %lld window entries (limit 2^30)", (long long)cap));
    int grid = (int)std::min<int64_t>(K, (int64_t)ctx->sm_count * 8);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    while (grid > 1 && (size_t)grid * ((size_t)cap * 12 + (size_t)mc * 16) > free_b / 2) grid = (grid + 1) / 2;
    if ((size_t)grid * ((size_t)cap * 12 + (size_t)mc * 16) > free_b / 2)
        return fin(nhp_fail(ctx, NHP_ERR_UNSUPPORTED, "adjacency sampler: one column needs %lld window entries, more than the free device memory holds", (long long)cap));
    ADJ_U(cudaMalloc(&d_ent_i, (size_t)grid * cap * sizeof(int)));
    ADJ_U(cudaMalloc(&d_ent_v, (size_t)grid * cap * sizeof(double)));
    ADJ_U(cudaMalloc(&d_lam, (size_t)grid * mc * sizeof(double)));
    ADJ_U(cudaMalloc(&d_gacc, (size_t)grid * mc * sizeof(double)));
    AdjArgs a;
    a.t = ev->d_t; a.c = ev->d_c; a.n = n; a.order = ev->d_order; a.node_ptr = ev->d_node_ptr; a.Mn = ev->d_Mn; a.K = (int)K; a.table_w = ctx->d_adj_tw;
    a.lambda0 = ctx->d_lambda0; a.W = ctx->d_W; a.A = d_A; a.rho = d_rho; a.u = d_u; a.seed = seed; a.counter = counter;
    a.lam0bn = lam0bn; a.lam0min = lam0min;
    a.D = ctx->dtmax; a.horizon = horizon; a.duration = ev->duration; a.flag = ctx->d_flag; a.col_begin = cb; a.col_stride = cs;
    a.cap = cap; a.ent_i = d_ent_i; a.ent_v = d_ent_v; a.lam = d_lam; a.gacc = d_gacc; a.max_col = mc;
    const size_t smem = (size_t)(2 * K + 2) * sizeof(int);
    if (ctx->kind == NHP_LOGITNORMAL) {
        ADJ_U(cudaFuncSetAttribute(k_adjacency<NHP_LOGITNORMAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
        k_adjacency<NHP_LOGITNORMAL><<<grid, 256, smem, s>>>(a);
    } else {
        ADJ_U(cudaFuncSetAttribute(k_adjacency<NHP_EXPONENTIAL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
        k_adjacency<NHP_EXPONENTIAL><<<grid, 256, smem, s>>>(a);
    }
    NHP_LAUNCHED(ctx);
    ADJ_U(cudaGetLastError());
    return fin(NHP_OK);
#undef ADJ_U
}

// launch the cached sweep: one CTA per column, or one thread-block cluster per column (cluster dimension as a launch attribute)
template <int KIND, int PRE> static int adj_launch_sweep(nhp_ctx *ctx, const AdjSweepArgs &w, size_t smem, int cluster) {
    cudaStream_t s = ctx->stream;
    if (cluster <= 1) {
        auto kernel = k_adj_sweep<KIND, PRE, false>;
        NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        const int grid = (int)std::min<int64_t>(w.ncols, ctx->sm_count);
        kernel<<<grid, ADJ_THREADS, smem, s>>>(w);
    } else {
        auto kernel = k_adj_sweep<KIND, PRE, true>;
        NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        cudaLaunchConfig_t cfg = {};
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = (unsigned)cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.blockDim = dim3(ADJ_THREADS); cfg.dynamicSmemBytes = smem; cfg.stream = s; cfg.attrs = attr; cfg.numAttrs = 1;
        cfg.gridDim = dim3((unsigned)(ctx->sm_count / cluster * cluster));
        int nclusters = 0;
        NHP_CUDA(ctx, cudaOccupancyMaxActiveClusters(&nclusters, kernel, &cfg));
        NHP_CHECK(ctx, nclusters >= 1, NHP_ERR_UNSUPPORTED, "adjacency sampler: no cluster of %d CTAs with %zu B of shared memory fits on this device", cluster, smem);
        nclusters = (int)std::min<int64_t>(nclusters, w.ncols);
        cfg.gridDim = dim3((unsigned)(nclusters * cluster));
        NHP_CUDA(ctx, cudaLaunchKernelEx(&cfg, kernel, w));
    }
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

// One adjacency Gibbs sweep over the owned columns of the device-resident matrix d_A (in place).  d_rho: per-link
// probabilities on the device, or NULL for the scalar rho_scalar; d_u: uniforms on the device or NULL (Philox).
static int adj_run(nhp_ctx *ctx, nhp_events *ev, const double *d_rho, double rho_scalar, const double *d_u, uint64_t seed, uint64_t counter,
                   double *d_A, int64_t col_begin, int64_t col_stride) {
    NHP_CHECK(ctx, col_stride >= 1 && col_begin >= 0 && col_begin < col_stride, NHP_ERR_INVALID, "adjacency sampler: need 0 <= col_begin < col_stride");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set (call nhp_cont_params_set)");
    NHP_CHECK(ctx, ev != nullptr && ev->K == ctx->K, NHP_ERR_INVALID, "adjacency sampler: bad events handle");
    NHP_CHECK(ctx, ev->n_halo == 0 && ev->index_base == 0, NHP_ERR_UNSUPPORTED,
              "the adjacency sampler works on unsharded data (multi-GPU partitions the columns, not the time axis)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    NHP_TRY(adj_ensure_ctx(ctx));
    const int64_t K = ctx->K, KK = K * K, n = ev->n;
    cudaStream_t s = ctx->stream;
    const unsigned kb = (unsigned)((KK + 255) / 256);
    if (ctx->kind == NHP_LOGITNORMAL) k_table_noA_ln<<<kb, 256, 0, s>>>((int)K, ctx->d_W, ctx->d_p1, ctx->d_p2, ctx->dtmax, (EntryLN *)ctx->d_adj_tw);
    else k_table_noA_ex<<<kb, 256, 0, s>>>((int)K, ctx->d_W, ctx->d_p1, (EntryEX *)ctx->d_adj_tw);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
    for (int i = 0; i < 7; i++) ctx->adj_info[i] = 0.0;
    AdjPhaseTimer tr(s);
    NHP_TRY(nhp_events_build_node_index(ctx, ev));
    tr.lap("node index");
    // grid baseline: the per-event rates of the columns in by-node order and their minima.  A zero rate at an event of a swept column
    // leaves the conditional undefined (the reference's logsumexp(-Inf, -Inf)): refused before anything changes
    const double *lam0bn = nullptr, *lam0min = nullptr;
    NHP_TRY(nhp_cont_event_baseline_bynode(ctx, ev, &lam0bn, &lam0min));
    if (lam0min)
        for (int64_t c = col_begin; c < K; c += col_stride)
            NHP_CHECK(ctx, ev->lam0min[(size_t)c] > 0.0, NHP_ERR_NUMERIC, "adjacency sampler: the baseline of node %lld is zero at one of its events", (long long)(c + 1));
    tr.lap("baseline rates");
    double horizon = adj_horizon_value(ctx, n);
    const char *envc = getenv("NHP_ADJ_CACHE");
    bool cached = !(envc && atoi(envc) == 0);
    int chunk_cap = ADJ_CHUNK_MAX;
    { const char *e = getenv("NHP_ADJ_CHUNK"); if (e && atoi(e) >= 1 && atoi(e) <= ADJ_CHUNK_MAX) chunk_cap = atoi(e); }
    // The cached structure stays valid for any horizon it covers: extra pairs beyond the requested cut-off are genuine
    // predecessors whose (tiny) contributions are simply included.  With a parameter-dependent horizon (Exponential cut-off,
    // which moves with every conjugate draw) it is built with a 25 % margin so that a chain does not rebuild it every sweep.
    const bool moving = ctx->kind == NHP_EXPONENTIAL && horizon < ctx->dtmax;
    const bool have_cache = cached && ev->d_adj_i && adj_payload_fits(ctx, ev) && ev->adj_cb == (int)col_begin && ev->adj_cs == (int)col_stride && ev->adj_chunk_cap == chunk_cap &&
                            (moving ? (ev->adj_horizon >= horizon && ev->adj_horizon <= 2.0 * horizon) : ev->adj_horizon == horizon);
    if (cached && !have_cache) {
        if (moving) horizon = std::min(ctx->dtmax, 1.25 * horizon);
        const int rc = adj_build_structure(ctx, ev, horizon, (int)col_begin, (int)col_stride, chunk_cap);
        if (rc < 0) return rc;
        if (rc == 1) cached = false;
    } else if (have_cache) horizon = ev->adj_horizon;
    NHP_TRY(nhp_timer_begin(ctx));
    if (cached) {
        AdjSweepArgs w;
        w.node_ptr = ev->d_node_ptr; w.K = (int)K; w.table_w = ctx->d_adj_tw; w.lambda0 = ctx->d_lambda0; w.A = d_A;
        w.lam0bn = lam0bn; w.lam0min = lam0min;
        k_adj_prep<<<kb, 256, 0, s>>>((int)K, ctx->d_W, ev->d_Mn, d_rho, rho_scalar, d_u, seed, counter, ctx->d_adj_dec);
        NHP_LAUNCHED(ctx);
        w.dec = ctx->d_adj_dec; w.D = ctx->dtmax;
        w.vstart = ev->d_adj_vstart; w.vbase = ev->d_adj_vbase; w.boff = ev->d_adj_boff; w.ent_i = ev->d_adj_i; w.ent_x = ev->d_adj_dt;
        w.lam = ev->d_adj_lam;
        w.chunk_max = (ev->adj_chunk_max + 1) & ~1;
        w.flag = ctx->d_flag; w.next = ctx->d_adj_ctl; w.stat = ctx->d_adj_stat;
        w.col_begin = (int)col_begin; w.col_stride = (int)col_stride; w.corder = ev->d_adj_corder;
        w.ncols = (int)((K - col_begin + col_stride - 1) / col_stride);
        w.s0 = ADJ_SMAX;
        { const char *e = getenv("NHP_ADJ_S0"); if (e && atoi(e) >= 1 && atoi(e) <= 32 && (atoi(e) & (atoi(e) - 1)) == 0) w.s0 = atoi(e); }
        size_t smem = (size_t)w.chunk_max * sizeof(double) + (size_t)((K + 31) / 32) * sizeof(unsigned) + 16;
        {   // room for the resident chunk's bucket offsets?  (the kernel's static shared memory: 12.1 KB, see -Xptxas -v)
            const size_t bo_bytes = (size_t)(((K + 31) / 32 + 3) & ~3) * sizeof(unsigned) - (size_t)((K + 31) / 32) * sizeof(unsigned) + (size_t)(2 * K + 1) * sizeof(int);
            const char *e = getenv("NHP_ADJ_BO_SMEM");
            w.bo_smem = !(e && atoi(e) == 0) && smem + bo_bytes + 12800 <= (size_t)ctx->smem_optin;
            if (w.bo_smem) smem += bo_bytes;
        }
        NHP_CHECK(ctx, smem <= (size_t)ctx->smem_optin - 4096, NHP_ERR_UNSUPPORTED, "adjacency sampler: K=%lld needs more shared memory than the device has", (long long)K);
        NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_adj_ctl, 0, 8 * sizeof(int), s));
        NHP_CUDA(ctx, cudaMemsetAsync(ctx->d_adj_stat, 0, 8 * sizeof(unsigned long long), s));
        if (w.ncols > 0) {
            const int cl = ev->adj_cluster;
            if (ctx->kind == NHP_EXPONENTIAL) NHP_TRY((adj_launch_sweep<NHP_EXPONENTIAL, 0>(ctx, w, smem, cl)));
            else if (ev->adj_kind == 1) NHP_TRY((adj_launch_sweep<NHP_LOGITNORMAL, 1>(ctx, w, smem, cl)));
            else NHP_TRY((adj_launch_sweep<NHP_LOGITNORMAL, 0>(ctx, w, smem, cl)));
        }
    } else {
        // the uncached kernel wants per-link probabilities and the matrix it updates on the device
        const double *rho_dev = d_rho;
        if (!rho_dev) {
            std::vector<double> r((size_t)KK, rho_scalar);
            NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_adj_rho, r.data(), (size_t)KK * sizeof(double), cudaMemcpyHostToDevice, s));
            NHP_CUDA(ctx, cudaStreamSynchronize(s));
            rho_dev = ctx->d_adj_rho;
        }
        NHP_TRY(adj_run_uncached(ctx, ev, horizon, rho_dev, d_u, seed, counter, d_A, (int)col_begin, (int)col_stride, lam0bn, lam0min));
    }
    int flag = 0;
    unsigned long long st[4] = {0, 0, 0, 0};
    NHP_CUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    if (cached) NHP_CUDA(ctx, cudaMemcpyAsync(st, ctx->d_adj_stat, sizeof(st), cudaMemcpyDeviceToHost, s));
    NHP_TRY(nhp_timer_end(ctx));
    NHP_CHECK(ctx, !(flag & 32), NHP_ERR_CUDA, "adjacency sampler: scratch overflow (internal error)");
    NHP_CHECK(ctx, !(flag & 64), NHP_ERR_NUMERIC, "adjacency sampler: NaN log-likelihood difference");
    ctx->adj_info[0] = (double)st[0]; ctx->adj_info[1] = (double)st[1]; ctx->adj_info[2] = (double)st[2]; ctx->adj_info[3] = (double)st[3];
    ctx->adj_info[4] = cached ? (double)ev->adj_pairs : 0.0;
    ctx->adj_info[5] = cached ? (double)ev->adj_nv + 1e-3 * ev->adj_cluster + 1e-6 * (ev->adj_kind ? 18 : 10) : 0.0;  // virtual columns . cluster size, bytes per pair
    ctx->adj_info[6] = ctx->last_ms;
    return NHP_OK;
}

static int adj_commit(nhp_ctx *ctx) {  // the masked tables, bit rows and row sums follow the new matrix
    if (!ctx->has_A) return NHP_OK;
    const double ms = ctx->last_ms;
    ctx->cont_set = false;
    ctx->sweep_ll_valid = false;
    NHP_TRY(nhp_cont_params_refresh(ctx));
    ctx->cont_set = true;
    ctx->last_ms = ms;
    return NHP_OK;
}

extern "C" int nhp_cont_resample_adjacency(nhp_ctx *ctx, nhp_events *ev, const double *rho, uint64_t seed, uint64_t counter, const double *u,
                                           double *A_inout) {
    return nhp_cont_resample_adjacency_cols(ctx, ev, rho, seed, counter, u, A_inout, 0, 1);
}

extern "C" int nhp_cont_resample_adjacency_cols(nhp_ctx *ctx, nhp_events *ev, const double *rho, uint64_t seed, uint64_t counter, const double *u,
                                                double *A_inout, int64_t col_begin, int64_t col_stride) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set (call nhp_cont_params_set)");
    NHP_CHECK(ctx, rho && A_inout, NHP_ERR_INVALID, "nhp_cont_resample_adjacency: NULL rho/A");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_TRY(adj_ensure_ctx(ctx));
    const size_t KK = (size_t)ctx->K * ctx->K;
    cudaStream_t s = ctx->stream;
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_adj_rho, rho, KK * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_adj_A, A_inout, KK * sizeof(double), cudaMemcpyHostToDevice, s));
    if (u) NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_adj_u, u, KK * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_TRY(adj_run(ctx, ev, ctx->d_adj_rho, 0.0, u ? ctx->d_adj_u : nullptr, seed, counter, ctx->d_adj_A, col_begin, col_stride));
    NHP_CUDA(ctx, cudaMemcpyAsync(A_inout, ctx->d_adj_A, KK * sizeof(double), cudaMemcpyDeviceToHost, s));
    // the new adjacency becomes the context's A (device to device; the masked tables are rebuilt)
    if (ctx->has_A) NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_A, ctx->d_adj_A, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return adj_commit(ctx);
}

extern "C" int nhp_cont_resample_adjacency_dev(nhp_ctx *ctx, nhp_events *ev, double rho, uint64_t seed, uint64_t counter, int64_t col_begin, int64_t col_stride,
                                               int commit) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "continuous parameters not set (call nhp_cont_params_set)");
    NHP_CHECK(ctx, ctx->has_A, NHP_ERR_STATE, "nhp_cont_resample_adjacency_dev: the process has no adjacency matrix");
    if (rho < 0.0) rho = ctx->rho;
    NHP_CHECK(ctx, rho >= 0.0 && rho <= 1.0, NHP_ERR_INVALID, "nhp_cont_resample_adjacency_dev: link probability outside [0, 1] (set it, or call nhp_cont_resample_network first)");
    NHP_TRY(adj_run(ctx, ev, nullptr, rho, nullptr, seed, counter, ctx->d_A, col_begin, col_stride));
    return commit ? adj_commit(ctx) : NHP_OK;
}

extern "C" int nhp_cont_adjacency_commit(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set && ctx->has_A, NHP_ERR_STATE, "nhp_cont_adjacency_commit: no network process parameters on the device");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    return adj_commit(ctx);
}

extern "C" int nhp_cont_adjacency_info(const nhp_ctx *ctx, double *out8) {
    if (!ctx || !out8) return NHP_ERR_INVALID;
    for (int i = 0; i < 8; i++) out8[i] = ctx->adj_info[i];
    return NHP_OK;
}
