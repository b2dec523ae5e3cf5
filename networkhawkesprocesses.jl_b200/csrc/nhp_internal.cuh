// nhp_internal.cuh -- shared declarations of libnhp (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <math.h>
#include <string>
#include <vector>
#include "../../include/nhp.h"
#include "../../include/nhp_devel.h"
#include "fastmath.cuh"

#define NHP_VERSION 100

// ---------------------------------------------------------------------------------------
// error plumbing
// ---------------------------------------------------------------------------------------
int nhp_fail(nhp_ctx *ctx, int code, const char *fmt, ...);

#define NHP_CUDA(ctx, call)                                                                               \
    do {                                                                                                  \
        cudaError_t e__ = (call);                                                                         \
        if (e__ != cudaSuccess) return nhp_fail((ctx), NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call,       \
                                                cudaGetErrorString(e__), __FILE__, __LINE__);             \
    } while (0)

#define NHP_CHECK(ctx, cond, code, ...)                                  \
    do {                                                                 \
        if (!(cond)) return nhp_fail((ctx), (code), __VA_ARGS__);        \
    } while (0)

#define NHP_TRY(expr)                 \
    do {                              \
        int rc__ = (expr);            \
        if (rc__ != NHP_OK) return rc__; \
    } while (0)

// ---------------------------------------------------------------------------------------
// per-(parent, child) parameter table entries.  Layout in HBM: child-major,
// table[child * K + parent], so a child's parents are contiguous (one 32 B / 16 B sector per pair).
// ---------------------------------------------------------------------------------------
struct __align__(32) EntryLN {  // LogitNormal: value = cf * exp(-h (z - mu)^2) / (dt (D - dt)),  z = log(dt/(D-dt))
    double cf;                  // [A] * W * sqrt(tau) * invsqrt2pi * D^2
    double mu;
    double h;                   // tau / 2
    double pad;
};
struct __align__(16) EntryEX {  // Exponential: value = wt * exp(-theta dt)
    double wt;                  // [A] * W * theta
    double theta;
};
template <int KIND> struct EntryOf;
template <> struct EntryOf<NHP_EXPONENTIAL> { typedef EntryEX type; };
template <> struct EntryOf<NHP_LOGITNORMAL> { typedef EntryLN type; };

// stats buffer layout (phase 0): [ll_logsum, ll_rowsum, M0[K], Mn[K], Mnm[K*K], S1[K*K]]
struct StatsLayout {
    int64_t K;
    __host__ __device__ int64_t off_ll() const { return 0; }
    __host__ __device__ int64_t off_M0() const { return 2; }
    __host__ __device__ int64_t off_Mn() const { return 2 + K; }
    __host__ __device__ int64_t off_Mnm() const { return 2 + 2 * K; }
    __host__ __device__ int64_t off_S1() const { return 2 + 2 * K + K * K; }
    __host__ __device__ int64_t total() const { return 2 + 2 * K + 2 * K * K; }
};

struct nhp_events {
    int64_t n = 0;          // events passed (halo + own)
    int64_t n_halo = 0;     // leading read-only predecessors
    int64_t index_base = 0; // global 0-based index of event 0
    int flags = 1;
    double duration = 0.0;
    int64_t K = 0;
    double *d_t = nullptr;      // [n + pad]
    int *d_c = nullptr;         // [n + pad] 0-based nodes
    int *d_poff = nullptr;      // [n] parent offset i - j (>0) | 0 baseline | -1 unset
    double *d_Mn = nullptr;     // [K] own-event counts per node
    int64_t n_t0 = 0;           // number of leading events with t == 0.0 exactly (quirk Q6)
    // tile window-start cache (depends on the look-back horizon)
    double cache_horizon = -1.0;
    int *d_tile_lo = nullptr;   // [ceil((n - n_halo)/64)]
    int64_t n_bound = 0;
    unsigned short *d_wlen = nullptr;  // [n - n_halo] window length of every own event (saturated at 65535), same cache
    // by-node order of the own events + work items of the child-major sweep (cont_child.cu), built on first use
    int *d_order = nullptr, *d_node_ptr = nullptr, *d_item_node = nullptr, *d_item_e0 = nullptr;
    double *d_lam0ev = nullptr;     // [n] baseline rate at every event for the context's grid baseline (version below), built on first use
    uint64_t lam0ev_version = 0;
    // the same rates in the by-node order (d_order) and their minimum per node, for the adjacency sampler (same curve version rule)
    double *d_lam0bn = nullptr;     // [n - n_halo] lam0ev[order[e]]
    double *d_lam0min = nullptr;    // [K] min over the node's own events (+Inf for a node without events)
    std::vector<double> lam0min;    // host copy of d_lam0min
    uint64_t lam0bn_version = 0;
    int64_t n_items = 0;
    // elliptical-slice update of the curves (cont_slice.cu): baseline-event records in by-node order, work items, partial sums
    int *d_sl_g = nullptr, *d_sl_item = nullptr;
    double *d_sl_t = nullptr, *d_sl_part = nullptr;
    // cached structure of the adjacency sampler (cont_adjacency.cu): every (child event, window predecessor) pair, grouped by
    // virtual column = (child column, time chunk of at most adj_chunk_cap of the column's events) and bucketed by parent node,
    // stably ordered (event, window position) inside a bucket.  The pairs depend on the data and the look-back horizon; the
    // payload also on the impulse kind it was built for (lags, or LogitNormal terms of the build-time dtmax), so a model of another
    // kind, or a LogitNormal model of another dtmax, must not read it
    double adj_horizon = -1.0;       // horizon the structure was built with
    int adj_impulse = -1;            // impulse kind (NHP_EXPONENTIAL / NHP_LOGITNORMAL) it was built for
    double adj_D = 0.0;              // dtmax it was built for (the LogitNormal payload holds logit(dt / D), 1 / (dt (D - dt)))
    int adj_cb = 0, adj_cs = 1;      // column partition it was built for
    int adj_chunk_cap = 0;           // chunk capacity (child events) it was built with
    int adj_chunk_max = 0;           // largest chunk actually present (sizes the sweep's shared memory)
    int64_t adj_nv = 0;              // number of virtual columns
    int *d_adj_vstart = nullptr;     // [K+1] first virtual column of every column
    int *d_adj_vnode = nullptr;      // [nv] child column of every virtual column
    int *d_adj_corder = nullptr;     // [owned columns] sweep order: most child events first
    int64_t *d_adj_vbase = nullptr;  // [nv+1] first entry of every virtual column
    int *d_adj_boff = nullptr;       // [nv][2K+1] section offsets inside a virtual column: singles of parent p at [2p], its runs at [2p+1]
    unsigned short *d_adj_i = nullptr;  // [adj_total] child event index inside its chunk | bit 15: same (event, parent) as the previous entry
    double *d_adj_dt = nullptr;      // [adj_total] t_i - t_j, or [2 adj_total] with the LogitNormal payload: (logit(dt / D), 1 / (dt (D - dt))) per entry, (0, 0) outside the support
    double *d_adj_q = nullptr;       // unused (the payload is interleaved in d_adj_dt)
    int adj_cluster = 0;             // CTAs per column (thread-block cluster size; 0: single-CTA streaming form)
    int adj_kind = 0;                // 1: LogitNormal payload
    double *d_adj_lam = nullptr;     // [n] per-event intensity in by-node order (work array of the sweep)
    size_t adj_bytes_i = 0, adj_bytes_dt = 0;  // sizes of the two entry arrays (they come from, and return to, the context's block cache)
    int64_t adj_total = 0;           // entries allocated (pairs + section padding)
    int64_t adj_pairs = 0;           // (child event, window predecessor) pairs
    int64_t max_win = 0;        // max over boundaries of (i0 - lo)
    double mean_win = 0.0;
};

struct nhp_disc {
    int64_t N = 0, T = 0, t_halo = 0;
    int *d_data = nullptr;      // [T][N] counts as int32, time-major (t outer, n inner) == Julia data[n + N*t]
    double *d_conv = nullptr;   // [B][N][T]  conv[t + T*(n + N*b)]
    int64_t L = 0, B = 0;
    int64_t total_events = 0;
    int64_t *d_scan = nullptr;  // exclusive scan of data in memory order (uniform index of each bin's first draw)
};

// the model shape a trace was begun for, compared whole: continuous Gibbs (K, kind, has_A, G), discrete Gibbs (N, B, has_A, 0),
// VB (N | K, B | kind, network, 0)
struct TraceShape {
    int64_t n = 0, b = 0, a = 0, g = 0;
    bool operator==(const TraceShape &o) const { return n == o.n && b == o.b && a == o.a && g == o.g; }
};

// a device-side trace (cont_trace.cu): cap slots, each of `doubles` doubles, `words` bit-packed adjacency words and `curve_doubles`
// doubles of curves (the last two optional), filled by device-to-device copies on the context's stream and read back at the end
struct DeviceTrace {
    double *d = nullptr;
    uint32_t *bits = nullptr;
    double *curves = nullptr;
    size_t doubles = 0, words = 0, curve_doubles = 0;  // per slot
    int64_t cap = 0, len = 0;
    TraceShape shape;
    // the doubles of the next slot, or nullptr when the trace is closed or full
    double *next() const { return len < cap ? d + (size_t)len * doubles : nullptr; }
};

// a mean-field VB state (vb_state.cu) of the discrete (disc_vb.cu) or the continuous (cont_vb.cu) model and its trace
struct VbState {
    bool set = false, network = false;
    int64_t n = 0, b = 0;  // N and B (discrete), K and the impulse kind (continuous)
    double dt = 1.0;
    double hyper[12] = {0};
    double *q = nullptr;
    size_t doubles = 0, cap = 0;  // doubles of the state, doubles allocated
    DeviceTrace trace;
};

struct nhp_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t own_stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    std::string err;
    int64_t launches = 0;
    double last_ms = 0.0;
    int sm_count = 148;
    int smem_optin = 0;
    // multi-GB blocks (adjacency structure) kept across events handles: cudaMalloc / cudaFree of 100 GB cost 0.1-0.7 s and a device-wide
    // synchronisation each, a first-time cudaMallocAsync of that size several seconds; a freed block serves the next structure
    std::vector<std::pair<void *, size_t>> big_cache;

    // ---- continuous parameters
    bool cont_set = false;
    int kind = 0;
    int64_t K = 0;
    double dtmax = 0.0;
    bool has_A = false;
    bool grad_valid = false;    // the statistics buffers hold a gradient (nhp_cont_loglik_grad_dev)
    double density = 1.0;       // fraction of non-zero effective weights
    double theta_min = 0.0, wt_max = 0.0, lambda0_min = 0.0; // Exponential cut-off horizon inputs (links with A*W != 0)
    double theta_min_all = 0.0, wt_max_all = 0.0;            // the same over all K^2 entries with W != 0 (adjacency sampler: it evaluates inactive links too)
    double lambda0_sum = 0.0;
    double a_sum = 0.0;           // sum of the adjacency matrix (number of links), refreshed with the tables
    double *d_lambda0 = nullptr;  // [K]
    // inhomogeneous baseline (LogGaussianCoxProcess, baselines.jl:187-336): lambda0_k(t) piecewise linear on a grid (cont_baseline.cu)
    double *d_bgrid_x = nullptr, *d_bgrid_v = nullptr;  // [bgrid_n] grid, [K][bgrid_n] values
    int64_t bgrid_n = 0; uint64_t bgrid_version = 0;     // 0 points: homogeneous lambda0
    double baseline_integral = 0.0;                      // sum_k integrate(lambda0_k) over the grid (trapezoid)
    double bgrid_min = 0.0;                              // smallest curve value: lambda0_min while the grid is active
    double bgrid_lo = 0.0, bgrid_hi = 0.0;               // x[0], x[bgrid_n-1] on the host (the simulator's coverage check)
    // GP prior of the log-curves, log lambda0_k = m + y_k, y_k ~ N(0, L L^T) (nhp_cont_baseline_prior; cont_slice.cu): [bprior_n^2] L
    double *d_bprior_L = nullptr; int64_t bprior_n = 0, bprior_cap = 0; double bprior_m = 0.0;  // 0 points: no prior
    void *d_slice = nullptr; size_t slice_cap = 0;       // work buffers of the elliptical-slice update
    double slice_info[4] = {0};                          // last update: list build ms, rounds + commit ms, rounds, work items
    double *d_W = nullptr, *d_A = nullptr, *d_p1 = nullptr, *d_p2 = nullptr; // raw [K*K] parent-major as passed
    void *d_table = nullptr;      // EntryLN/EntryEX [K*K] child-major
    double *d_rowsum = nullptr;   // [K] sum_c [A]W[p,c]
    double *d_rowsum_w = nullptr; // [K] sum_c W[p,c] (recursive Network quirk Q3)
    uint32_t *d_abits = nullptr;  // adjacency/non-zero bitmask, child-major rows of abits_words words
    int64_t abits_words = 0;
    int64_t cap_K = 0;            // allocated for this K
    // adjacency sampler work buffers (allocated on first use, sized by cap_K)
    void *d_adj_tw = nullptr;     // EntryLN/EntryEX [K*K] child-major, without the adjacency factor
    double *d_adj_rho = nullptr, *d_adj_u = nullptr, *d_adj_A = nullptr;  // [K*K] staging of host arguments
    double4 *d_adj_dec = nullptr; // [K*K] decision inputs of the adjacency sweep (k_adj_prep)
    int *d_adj_ctl = nullptr;     // [8] dynamic work counters of the build / sweep kernels
    unsigned long long *d_adj_stat = nullptr;  // [8] sweep diagnostics (steps, batches, flips, recomputed steps)
    double *d_save = nullptr;     // nhp_cont_params_save: [K + 4 K^2] copy of lambda0, W, A, p1, p2
    double rho = -1.0;            // link probability of the Bernoulli network kept with the context (nhp_cont_resample_network)
    // sample trace: slots of (rho, lambda0, W, p1 [, p2]) + bit-packed adjacency matrices, and the curves [K][G] for a trace begun
    // with curves and a prior
    DeviceTrace cont_trace;
    double sweep_info[8] = {0};   // last nhp_cont_gibbs_sweep: ms of the parent sweep, of (second pass + draws + tables), of the adjacency kernel, of the curves' slice update, its rounds
    double adj_info[8] = {0};     // last adjacency sweep: steps, batches, flips, recomputed steps, entries, chunks, kernel ms, build ms

    // ---- statistics
    double *d_stats0 = nullptr;   // StatsLayout
    double *d_stats1 = nullptr;   // [K*K] S2
    double *d_xbar = nullptr;     // [K*K] S1/Mnm scratch
    int *d_flag = nullptr;        // device error flag
    bool parents_valid = false;
    bool opt_sweep_ll = false;     // NHP_OPT_SWEEP_LOGLIK
    bool sweep_ll_valid = false;   // stats0[0..1] hold the log-likelihood terms of the last parent sweep

    // ---- scratch
    double *d_partials = nullptr;
    int64_t partials_cap = 0;
    void *d_scratch = nullptr;
    size_t scratch_cap = 0;
    int64_t *d_winstat = nullptr; // [2]: max window, sum window

    // ---- multi-GPU (comm.cu): NCCL communicator of this rank, staging buffer
    void *comm = nullptr;
    int rank = 0, nranks = 1;
    double *d_comm_buf = nullptr;
    size_t comm_buf_cap = 0;

    // ---- discrete parameters
    bool disc_set = false;
    int64_t dN = 0, dB = 0;
    double ddt = 1.0;
    bool d_has_A = false;
    double *dd_lambda0 = nullptr, *dd_W = nullptr, *dd_A = nullptr, *dd_theta = nullptr;
    double *dd_bump = nullptr;    // [N*B][N] row k=(p*B+b), col c: [A]W theta dt
    int *dd_klist = nullptr, *dd_kptr = nullptr;  // per child: ascending k = p*B+b of the structurally non-zero entries
    double *dd_btc = nullptr;     // bumpT values at dd_klist
    int *dd_kcnt = nullptr;       // [N] non-zero effective weights per child (table refresh work array)
    double *dd_ksum = nullptr;    // [4]: list length, longest child list, non-zero effective weights, sum of A (table refresh results)
    size_t dd_klist_cap = 0;      // entries allocated in dd_klist / dd_btc
    bool dd_lists = false;        // dd_klist / dd_kptr / dd_btc describe the current parameters (density <= 0.5)
    double dd_density = 1.0;
    double dd_a_sum = 0.0;        // sum of the discrete adjacency matrix, refreshed with the tables
    double dd_rho = -1.0;         // link probability of the discrete Bernoulli network (nhp_disc_network_set); the continuous model keeps its own
    double *dd_counts = nullptr;  // [N * (1 + N B)] counts of the last discrete Gibbs parent sweep (counts[c + N k]), kept for the device-side draws
    size_t dd_counts_cap = 0; int64_t dd_counts_N = 0, dd_counts_B = 0;
    int64_t dd_maxNA = 0;
    // discrete sample trace: slots of (rho, lambda0, W, theta) + bit-packed adjacency matrices
    DeviceTrace disc_trace;

    // ---- discrete mean-field VB (disc_vb.cu): q = [alphav(N); betav(N); gammav(N^2 B); kappav(N^2); nuv(N^2)]; a network state
    // appends [kappa0v(N^2); nu0v(N^2); pv(N^2); alpharhov; betarhov].  hyper: alpha0, beta0, kappa, nu, gamma (+ kappa0, nu0,
    // alpha_rho, beta_rho for a network state)
    VbState dvb;

    // ---- continuous mean-field VB (cont_vb.cu): q = [alphav(K); betav(K); kappav(K^2); nuv(K^2)], then Exponential atheta(K^2);
    // btheta(K^2) | LogitNormal mv(K^2); lambdav(K^2); av(K^2); bv(K^2); the kind and K of the parameters at nhp_cont_vb_set; a network
    // state appends [kappa0v(K^2); nu0v(K^2); pv(K^2); alpharhov; betarhov].  hyper: alpha0, beta0, kappa, nu, then alpha, beta, 0, 0 |
    // mumu, kappamu, a0, b0; then kappa0, nu0, alpha_rho, beta_rho (network).  Allocated behind q: one change slot, and for a network
    // state lrho and the block sums of pv
    VbState cvb;
};

// launch bookkeeping
#define NHP_LAUNCHED(ctx) ((ctx)->launches++)

int nhp_scratch(nhp_ctx *ctx, size_t bytes, void **out);
int nhp_partials(nhp_ctx *ctx, int64_t count, double **out);
int nhp_timer_begin(nhp_ctx *ctx);
int nhp_timer_end(nhp_ctx *ctx);  // synchronises the stream and stores last_ms

// device traces (cont_trace.cu).  begin: refuses capacity < 1, frees the trace, allocates capacity slots for shape (a failed
// allocation leaves it closed); free: synchronises the stream, releases the buffers and closes the trace
int nhp_trace_begin(nhp_ctx *ctx, DeviceTrace &tr, const char *fn, int64_t capacity, size_t doubles, size_t words, size_t curve_doubles,
                    TraceShape shape);
void nhp_trace_free(nhp_ctx *ctx, DeviceTrace &tr);
int nhp_trace_count(const DeviceTrace &tr, int64_t *count, int64_t *capacity);
int nhp_trace_check_range(nhp_ctx *ctx, const DeviceTrace &tr, const char *fn, int64_t first, int64_t count);  // slots [first, first + count) stored
// doubles [off, off + n) of slots [first, first + count) to the host, one slot after the other (nothing for out == NULL); stream-ordered
int nhp_trace_read_field(nhp_ctx *ctx, const DeviceTrace &tr, int64_t first, int64_t count, size_t off, size_t n, double *out);

// VB states (vb_state.cu).  set: every entry of q positive and finite, except [fin_lo, fin_hi) (finite) and [p_lo, p_hi) (a link
// probability in [0, 1]); refused before anything changes.  Then the buffer grows to alloc doubles, q is uploaded (synchronised: the
// caller may reuse q) and the state takes the shape (n, b, network); the caller adds dt and the hyper-parameters
int nhp_vb_state_set(nhp_ctx *ctx, VbState &st, const char *fn, const double *q, size_t doubles, size_t alloc, size_t fin_lo, size_t fin_hi,
                     size_t p_lo, size_t p_hi, int64_t n, int64_t b, bool network);
int nhp_vb_state_get(nhp_ctx *ctx, const VbState &st, const char *fn, const char *set_fn, double *q);
void nhp_vb_state_free(nhp_ctx *ctx, VbState &st);
int nhp_vb_trace_begin(nhp_ctx *ctx, VbState &st, const char *fn, const char *set_fn, int64_t capacity);  // slots of the state's q
int nhp_vb_trace_push(nhp_ctx *ctx, VbState &st);  // the state into the next slot of an open trace that is not full; stream-ordered
int nhp_vb_trace_read(nhp_ctx *ctx, const VbState &st, const char *fn, int64_t first, int64_t count, double *q_out);

// ---------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------
#define NHP_INVSQRT2PI 0.3989422804014327

// Philox4x32-10 (Salmon et al. 2011): counter (c0..c3), key (k0,k1)
__host__ __device__ inline void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1, uint32_t out[4]) {
    const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; r++) {
        uint64_t p0 = (uint64_t)M0 * c0, p1 = (uint64_t)M1 * c2;
        uint32_t hi0 = (uint32_t)(p0 >> 32), lo0 = (uint32_t)p0, hi1 = (uint32_t)(p1 >> 32), lo1 = (uint32_t)p1;
        uint32_t n0 = hi1 ^ c1 ^ k0, n1 = lo1, n2 = hi0 ^ c3 ^ k1, n3 = lo0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += W0; k1 += W1;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}
// uniform double in [0,1) with 53 random bits, keyed by (seed; index, counter)
__host__ __device__ inline double philox_uniform(uint64_t seed, uint64_t index, uint64_t counter) {
    uint32_t r[4];
    philox4x32_10((uint32_t)index, (uint32_t)(index >> 32), (uint32_t)counter, (uint32_t)(counter >> 32), (uint32_t)seed, (uint32_t)(seed >> 32), r);
    uint64_t x = (((uint64_t)r[0] << 32) | (uint64_t)r[1]) >> 11;
    return (double)x * 1.1102230246251565e-16; // 2^-53
}

#ifdef __CUDACC__
// out-of-line rare paths: subnormal arguments / overflowing exponent (libdevice arithmetic)
static __device__ __noinline__ double slow_pair_ln(double cf, double mu, double h, double dt, double D) {
    if (!(dt > 0.0 && dt < D)) return 0.0;
    double la = log(dt), lb = log(D - dt), dz = (la - lb) - mu;
    return cf * exp(-h * dz * dz - (la + lb));
}
// x in [2^-500, 2^500)?  (one integer compare on the high word; products and squares of such values stay normal)
__device__ __forceinline__ bool in_mid_range(double x) { return (unsigned)(__double2hiint(x) - 0x20B00000) < 0x3E800000u; }
// 1/x for mid-range x: MUFU seed (20 bits) + two Newton steps (full double precision, ~1 ulp)
__device__ __forceinline__ double fast_rcp_mid(double x) {
    double y;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x));
    double e = fma(-x, y, 1.0);
    y = fma(y, e, y);
    e = fma(-x, y, 1.0);
    return fma(y, e, y);
}
__device__ __forceinline__ double pair_value(const EntryLN &e, double dt, double D, const FastTables *ft) {
    // Distributions.pdf(LogitNormal(mu, tau^-1/2), dt/D): zero outside 0 < x < 1 (impulses.jl:174-178)
    //   = cf exp(-h (z - mu)^2) / (dt (D - dt)),  z = logit(dt/D) = log(dt / (D - dt)),  cf carries D^2.
    // One reciprocal q = 1/(dt b) serves both the Jacobian and the logit argument dt/b = dt^2 q, so the pair costs one
    // table-driven log and one exp (the two-log form needed a second shared-memory table look-up per pair).
    const double b = D - dt;
    if (in_mid_range(dt) && in_mid_range(b)) {  // => 0 < dt < D
        const double q = fast_rcp_mid(dt * b);
        const double dz = fast_log_n(dt * dt * q, ft) - e.mu;
        return e.cf * q * fast_exp_c(-(e.h * dz) * dz, ft);  // the exponent is <= 0: no overflow branch
    }
    return slow_pair_ln(e.cf, e.mu, e.h, dt, D);
}
__device__ __forceinline__ double pair_value(const EntryEX &e, double dt, double, const FastTables *ft) {
    // Distributions.pdf(Exponential(1/theta), dt): theta exp(-theta dt), zero for dt < 0 (impulses.jl:106-108)
    const double x = -e.theta * dt;
    if (__double2hiint(dt) < 0) return dt < 0.0 ? 0.0 : e.wt;  // dt < 0 (or -0.0)
    if (__double2hiint(x) >= 0x40862800) return e.wt * slow_exp(x);
    return e.wt * fast_exp_c(x, ft);
}
// log_duration(parent, child, dtmax)  impulses.jl:228
__device__ __forceinline__ double log_duration_dev(double dt, double D) { return log(dt / (D - dt)); }

__device__ __forceinline__ void red_add_f64(double *addr, double v) { atomicAdd(addr, v); }
#endif

// internal entry points shared between translation units
int nhp_cont_prepare_windows(nhp_ctx *ctx, nhp_events *ev, double horizon);
int nhp_cont_run_loglik(nhp_ctx *ctx, nhp_events *ev, int recursive);
double nhp_cont_horizon_value(const nhp_ctx *ctx, int64_t n_total, int recursive);
int nhp_events_build_node_index(nhp_ctx *ctx, nhp_events *ev);  // d_order / d_node_ptr (cont_child.cu)
int nhp_cont_event_baseline(nhp_ctx *ctx, nhp_events *ev, const double **lam0ev);  // cont_baseline.cu: NULL for a homogeneous baseline
int nhp_cont_event_baseline_bynode(nhp_ctx *ctx, nhp_events *ev, const double **lam0bn, const double **lam0min);  // the same in by-node order + per-node minima
double nhp_cont_baseline_term(const nhp_ctx *ctx, const nhp_events *ev);             // sum(integrated_intensity(baseline, duration)) of the log-likelihood
struct SweepArgs;
int nhp_cont_try_adj_loglik(nhp_ctx *ctx, nhp_events *ev, SweepArgs &sa, int *grid_out, int cb = 0, int cs = 1);  // cont_adjacency.cu: 1 = does not apply
void nhp_events_free_adjacency(nhp_ctx *ctx, nhp_events *ev, cudaStream_t s);
void *nhp_big_alloc(nhp_ctx *ctx, size_t bytes);              // nullptr when the device cannot provide it
void nhp_big_free(nhp_ctx *ctx, void *p, size_t bytes);       // ctx == nullptr: cudaFree
size_t nhp_big_cached_bytes(const nhp_ctx *ctx);
void nhp_big_flush(nhp_ctx *ctx);                 // cached structure of the adjacency sampler (nhp_context.cu)
int nhp_events_from_device(nhp_ctx *ctx, const double *d_t, const int *d_c, int64_t n, double duration, int64_t K, nhp_events **out);  // nhp_context.cu
// disc.cu: the handle of an int32 count grid d_data[t*N + n] already on the device (non-zero bins, draw scan, per-child CSR, row sums,
// total_events, longest column); takes ownership of d_data, also on failure
int nhp_disc_from_device(nhp_ctx *ctx, int *d_data, int64_t N, int64_t T, int64_t t_halo, nhp_disc **out);
// discrete chain pieces shared between translation units
int nhp_disc_tables_refresh(nhp_ctx *ctx);        // disc.cu: bump table, compact parent lists, density, sum of A from the device-resident parameters
const double *nhp_disc_rowsum(nhp_disc *dd);      // disc.cu: [N] events per node (device)
// disc.cu: VB statistics of the bins t_lo <= t < t_hi added into zeroed sums; the events of each node over those bins added into events[N]
int nhp_disc_vb_reduce(nhp_ctx *ctx, nhp_disc *dd, int64_t t_lo, int64_t t_hi, const double *e0, const double *ET, double *alpha_sum, double *gammaT);
int nhp_disc_range_events(nhp_ctx *ctx, nhp_disc *dd, int64_t t_lo, int64_t t_hi, double *events);
int nhp_disc_draw_params(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *d_Mn, const double *hyper);  // cont_conjugate.cu
int nhp_disc_draw_network(nhp_ctx *ctx, uint64_t seed, uint64_t counter, double alpha, double beta);  // cont_conjugate.cu: ctx->dd_rho ~ Beta
