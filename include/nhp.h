/*
 * nhp.h -- C ABI of libnhp, the B200 (sm_100a) implementation of the event-history hot path
 * of NetworkHawkesProcesses.jl.  This is the drop-in boundary: the Julia package keeps its
 * API and forwards the methods cited below to these entry points with `ccall`
 * (INTEGRATION.md shows the stubs).  Plain pointers and sizes only; no torch / CUDA types.
 *
 * Conventions (identical to the Julia arrays so no reshaping happens at the boundary):
 *   - Float64 everywhere; matrices column-major, X[parent + K*child] (0-based offsets);
 *   - nodes are 1-based Int64; parent indices are 1-based Int64 with 0 = baseline;
 *   - every pointer argument is a HOST pointer unless its name ends in `_dev`; the library
 *     copies in/out and never keeps a host pointer past the call;
 *   - every function returns NHP_OK (0) or a negative nhp_status; nhp_last_error() gives the
 *     message.  There is NO CPU fallback: without a usable sm_100 GPU nhp_create fails.
 *   - calls on one context are synchronous (stream-synchronised before return) and must not
 *     be issued concurrently from several threads; use one context per host thread.
 *
 * Reference citations are file:line under /root/reference/src/.
 */
#ifndef NHP_H
#define NHP_H
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

typedef enum {
    NHP_OK = 0,
    NHP_ERR_INVALID = -1,     /* bad argument (the reference would throw error()/DomainError) */
    NHP_ERR_CUDA = -2,        /* CUDA runtime failure */
    NHP_ERR_NO_DEVICE = -3,   /* no sm_100 device: the library has no CPU path */
    NHP_ERR_STATE = -4,       /* call sequence error (e.g. parameters not set) */
    NHP_ERR_NUMERIC = -5,     /* NaN / negative intensities where the reference's Categorical/Poisson would throw */
    NHP_ERR_UNSUPPORTED = -6
} nhp_status;

#define NHP_EXPONENTIAL 0 /* ExponentialImpulseResponse  impulses.jl:30-37  */
#define NHP_LOGITNORMAL 1 /* LogitNormalImpulseResponse  impulses.jl:138-148 */

typedef struct nhp_ctx nhp_ctx;       /* one device + one stream + parameter/statistic buffers */
typedef struct nhp_events nhp_events; /* device-resident continuous data (times, nodes, duration) */
typedef struct nhp_disc nhp_disc;     /* device-resident discrete data (N x T counts) + convolution */

/* ---- context ------------------------------------------------------------------------- */
int nhp_create(int device, nhp_ctx **out);
int nhp_destroy(nhp_ctx *ctx);
const char *nhp_last_error(const nhp_ctx *ctx); /* ctx may be NULL: last error of a failed nhp_create */
int nhp_version(void);
/* device-time (CUDA events on the context stream) of the kernels of the most recent call, ms */
double nhp_last_kernel_ms(const nhp_ctx *ctx);

/* Context options. */
#define NHP_OPT_SWEEP_LOGLIK 1 /* value != 0: nhp_cont_resample_parents also accumulates the log-likelihood terms */
int nhp_set_option(nhp_ctx *ctx, int option, int64_t value);
/* Run every later call of this context on the caller's CUDA stream (a cudaStream_t passed as
 * void*; NULL restores the context's own stream), e.g. torch.cuda.current_stream().cuda_stream so
 * that the caller's CUDA events and NCCL collectives order with the library's kernels. */
int nhp_set_stream(nhp_ctx *ctx, void *cuda_stream);
/* ---- continuous data: data = (events, nodes, duration) of continuous.jl:14 ------------- */
/* Upload once; mle!/mcmc! call the likelihood thousands of times on the same data
 * (continuous.jl:146-149, inference.jl:55-62).
 * Time sharding (multi-GPU): a shard passes its own events preceded by `n_halo` read-only
 * predecessor events (those within dtmax of its first event); `index_base` is the global
 * 0-based index of the first passed event, so parent indices stay global.  `flags` bit 0:
 * this shard adds the baseline integral term to the log-likelihood (set on exactly one
 * shard; pass 1 when not sharding). */
int nhp_events_upload(nhp_ctx *ctx, const double *times, const int64_t *nodes, int64_t n, double duration, int64_t K,
                      int64_t n_halo, int64_t index_base, int flags, nhp_events **out);
int nhp_events_free(nhp_ctx *ctx, nhp_events *ev);
int64_t nhp_events_count(const nhp_events *ev);
/* rand(process, duration)  continuous.jl:16-37, 131-142, 335-348: one sample of the process whose parameters the context
 * holds (nhp_cont_params_set), simulated on the device generation by generation (cluster representation: baseline events
 * baselines.jl:67-70, Poisson(W[p,c]) children per event and child node weights.jl:25-27, lags from the impulse response
 * impulses.jl:63-66, 196-202, truncated at `duration`), sorted by time and left device resident as an events handle -- no host
 * round trip for 1e8-event samples.  While LogGaussianCox curves are set (nhp_cont_baseline_grid), generation 0 of node k is the
 * inhomogeneous Poisson process of rate lambda0_k(t), the curve the sweeps evaluate; the grid must then cover [0, duration]
 * (x[0] <= 0 and x[n_grid-1] >= duration), NHP_ERR_INVALID otherwise, before anything is allocated.  Philox keyed by `seed`: the
 * sample is a deterministic function of the parameters, the curves, `duration` and `seed`; parity with the reference is
 * distributional.  Fails when the sample would exceed max_events.  nhp_events_download copies (events, nodes) of a handle to the host in Julia's conventions
 * (any pointer may be NULL). */
int nhp_cont_rand(nhp_ctx *ctx, double duration, uint64_t seed, int64_t max_events, nhp_events **out);
int nhp_events_download(nhp_ctx *ctx, nhp_events *ev, double *times, int64_t *nodes, double *duration);

/* ---- continuous parameters --------------------------------------------------------------
 * lambda0[K]  HomogeneousProcess.lambda (baselines.jl:27-39);  W[K*K] weights.W (weights.jl:47-55);
 * A[K*K] adjacency_matrix or NULL for ContinuousStandardHawkesProcess (continuous.jl:108-112, 315-321);
 * p1 = theta (Exponential) | mu (LogitNormal); p2 = tau (LogitNormal) | NULL; dtmax may be +Inf
 * for Exponential (impulses.jl:37).  Length checks mirror impulses.jl:44-45,155-156, weights.jl:10-11. */
int nhp_cont_params_set(nhp_ctx *ctx, int kind, int64_t K, const double *lambda0, const double *W, const double *A,
                        const double *p1, const double *p2, double dtmax);

/* Inhomogeneous baseline inside the sweeps: LogGaussianCoxProcess (baselines.jl:187-336), lambda0_k(t) = LinearInterpolator(x,
 * lambda[k])(t) (utils/interpolation.jl:27-36).  x[n_grid] strictly increasing, values[g + n_grid*k] >= 0.  After this call the
 * log-likelihood, intensity and parent sweeps of the context use lambda0_k(t_i) as the baseline rate of event i (parent weights:
 * "baseline last", parents.jl:25-46) and sum_k integrate(lambda0_k) (trapezoid, baselines.jl:336) as the baseline compensator; an
 * event or query time outside [x[0], x[n_grid-1]] is an error (the reference throws a DomainError).  n_grid = 0 returns to the
 * homogeneous lambda0; nhp_cont_params_set also does (re-apply the curves after it).  The adjacency sampler and the structure
 * log-likelihood of a network process read lambda0_k(t_i) as well (the sampler returns NHP_ERR_NUMERIC, before changing anything,
 * when a curve is zero at an event of a column it sweeps), and nhp_cont_rand draws the baseline events from the curves; the analytic gradient takes a homogeneous baseline (NHP_ERR_UNSUPPORTED
 * otherwise).  While the curves are set, the Exponential cut-off horizon measures the omitted tail against their smallest value. */
int nhp_cont_baseline_grid(nhp_ctx *ctx, int64_t n_grid, const double *x, const double *values);
/* The likelihood of the elliptical-slice update of the curves (baselines.jl:214-254: resample!(::LogGaussianCoxProcess) =
 * split_extract + loglikelihood per node), for all K nodes at once and for CANDIDATE curves `values` on grid `x`:
 *   ll[k] = -integrate(f_k) + sum over the events of node k that the last parent sweep attributed to the baseline of log f_k(t_i).
 * The parent assignment is the device-resident one of the last nhp_cont_resample_parents on `ev` (split_extract never
 * materialises).  Time shards return additive shares. */
int nhp_cont_baseline_loglik(nhp_ctx *ctx, nhp_events *ev, int64_t n_grid, const double *x, const double *values, double *ll);
/* The GP prior of the log-curves (baselines.jl:187-212): log lambda0_k = m + y_k, y_k ~ N(0, L L^T) on the grid.  L[g + n_grid*h]
 * is the lower-triangular Cholesky factor, column-major (its strictly upper triangle is ignored); n_grid must be that of the current
 * curves and at most 4096, L finite with a positive diagonal (NHP_ERR_INVALID otherwise).  nhp_cont_params_set, nhp_cont_baseline_grid
 * with n_grid = 0 and a grid of another size drop the prior.  With curves and a prior, nhp_cont_gibbs_sweep updates the curves. */
int nhp_cont_baseline_prior(nhp_ctx *ctx, int64_t n_grid, const double *L, double m);
/* resample!(process::LogGaussianCoxProcess, data, parents) (baselines.jl:214-326) for all K nodes on the device: one elliptical-slice
 * update per node [Murray, Adams & MacKay 2010] with the likelihood of nhp_cont_baseline_loglik, from the parents of the last parent
 * sweep on `ev` (a rank's time shard: the per-node sums are all-reduced, every rank reaches the same curves).  Random numbers:
 * z == NULL && u == NULL: Philox keyed by (seed; node, draw, counter); otherwise both are host arrays, z[g + n_grid*k] standard
 * normals (the prior draw is L z) and u[j + 101*k] uniforms, j = 0 the slice height, j = 1 + a the angle of attempt a (attempt 0:
 * theta = 2 pi u; after a rejection the bracket side theta is on shrinks to theta and theta = lo + u (hi - lo)).  attempts[K] (may be
 * NULL) receives the candidates each node evaluated.  NHP_ERR_STATE without curves, prior or parent assignment; NHP_ERR_NUMERIC for
 * a curve value <= 0 or when a node reaches 100 attempts (baselines.jl:316).  The curves change only when every node accepted; the
 * new ones invalidate the parent assignment, as nhp_cont_baseline_grid does. */
int nhp_cont_resample_baseline(nhp_ctx *ctx, nhp_events *ev, uint64_t seed, uint64_t counter, const double *z, const double *u, int64_t *attempts);
/* The current curves in the layout of nhp_cont_baseline_grid (values[g + n_grid*k]). */
int nhp_cont_baseline_get(nhp_ctx *ctx, double *values);

/* Look-back horizon the sweeps use for the current parameters: dtmax for LogitNormal; for
 * Exponential min(dtmax, H) where H is the cut-off beyond which the omitted tail of any event's
 * history is < 1e-14 of the smallest baseline rate (every omitted term <= max(W theta)
 * exp(-min(theta) H), fewer than n_total of them).  A time shard's halo must cover it. */
int nhp_cont_horizon(nhp_ctx *ctx, int64_t n_total, int recursive, double *horizon);

/* loglikelihood(process, data; recursive)  continuous.jl:210-239 / 360-389.  recursive != 0 with
 * an Exponential impulse selects the full-history semantics of recursive_loglikelihood
 * (continuous.jl:241-276 / 407-442, incl. quirks Q3/Q6/Q7 of SURVEY.md section 9).  For a shard
 * the result is the shard's additive share (sum over ranks = ll). */
int nhp_cont_loglik(nhp_ctx *ctx, nhp_events *ev, int recursive, double *ll);
/* Multi-GPU form: this rank's additive share (sum over ranks = ll).  ev_shard is the rank's time shard; when the replicated stream
 * ev_full (may be NULL) already carries the rank's columns of the adjacency structure, the share is taken from it instead (active
 * buckets of the columns c = rank mod nranks; rank 0 adds the baseline and compensator terms).  Single GPU: nhp_cont_loglik(ev_shard). */
int nhp_cont_loglik_dist(nhp_ctx *ctx, nhp_events *ev_shard, nhp_events *ev_full, int recursive, double *share);
/* Extension for mle! (continuous.jl:144-198; the reference gives Optim a gradient-free objective, i.e.
 * ~2P log-likelihood evaluations per finite-difference gradient): the log-likelihood of nhp_cont_loglik
 * together with its analytic gradient, from two sweeps over the events.  Layouts as the parameters:
 * dlambda0[K]; dW, dp1, dp2 [K*K] parent-major (X[parent + K*child]); Exponential: dp1 = d/d theta, dp2
 * untouched; LogitNormal: dp1 = d/d mu, dp2 = d/d tau.  Entries with A[p,c] = 0 get the derivative of the
 * compensator only.  Any output pointer may be NULL.  For a shard every output is the shard's additive share.
 * _dev leaves the result on the device in the statistics buffers (dlambda0 -> M0 slot, dW -> Mnm, dp1 -> S1 of
 * phase 0; dp2 -> phase 1 of nhp_cont_stats_dev) so the multi-GPU reduction is the two all-reduces of the Gibbs
 * statistics; _read copies it out.  Invalidates the parent-sweep statistics. */
int nhp_cont_loglik_grad(nhp_ctx *ctx, nhp_events *ev, int recursive, double *ll, double *dlambda0, double *dW, double *dp1, double *dp2);
int nhp_cont_loglik_grad_dev(nhp_ctx *ctx, nhp_events *ev, int recursive);
int nhp_cont_loglik_grad_read(nhp_ctx *ctx, nhp_events *ev, double *ll, double *dlambda0, double *dW, double *dp1, double *dp2);
/* total_intensity at every (non-halo) event  continuous.jl:286-300 / 391-405; out[n - n_halo] */
int nhp_cont_event_intensity(nhp_ctx *ctx, nhp_events *ev, double *out);
/* intensity(process, data, times::Vector{Float64})  continuous.jl:76-96; out[nq*K], out[q + nq*k] */
int nhp_cont_intensity(nhp_ctx *ctx, nhp_events *ev, const double *times, int64_t nq, double *out);

/* resample_parents(process, data)  parents.jl:1-46, fused with the counters and impulse
 * statistics of parents.jl:61-79, baselines.jl:87-96, impulses.jl:84-96,230-240 so parents need
 * not leave the GPU.  Uniforms: u != NULL -> u[i] is the uniform of (non-halo) event i (parity
 * tests); u == NULL -> Philox4x32-10 keyed by (seed; global event index, counter).
 * parents / parentnodes may be NULL (kept on device for nhp_cont_suffstats). */
int nhp_cont_resample_parents(nhp_ctx *ctx, nhp_events *ev, uint64_t seed, uint64_t counter, const double *u,
                              int64_t *parents, int64_t *parentnodes);
/* The parent sweep evaluates every event's total intensity anyway; with NHP_OPT_SWEEP_LOGLIK enabled it also
 * accumulates the log-likelihood terms of the parameters it ran with (one extra log per event), and this call
 * returns that log-likelihood (same value as nhp_cont_loglik with recursive = 0) without a second pass over the events.  For a shard: the shard's additive share; the terms
 * also sit in slots 0..1 of the phase-0 statistics buffer, so the multi-GPU all-reduce carries them. */
int nhp_cont_sweep_loglik(nhp_ctx *ctx, nhp_events *ev, double *ll);
/* The assignment the device currently holds, in the reference's format (parents.jl:1-23): what a caller that destructures
 * `parents, parentnodes = resample_parents(process, data)` gets, exported on demand.  Either pointer may be NULL. */
int nhp_cont_parents_get(nhp_ctx *ctx, nhp_events *ev, int64_t *parents, int64_t *parentnodes);
/* Import a parent assignment (1-based global indices, 0 = baseline) and rebuild the fused
 * statistics from it: the "statistics given identical parent assignments" entry. */
int nhp_cont_parents_set(nhp_ctx *ctx, nhp_events *ev, const int64_t *parents);
/* Sufficient statistics of the current parent assignment; any output may be NULL.
 *   M0[K]   baseline counts                node_counts(nodes,parentnodes,K)  baselines.jl:87-96
 *   Mn[K]   events per node                node_counts(nodes,K)              parents.jl:61-68
 *   Mnm[K*K] parent->child counts          parent_counts                     parents.jl:70-79
 *   S1[K*K] Exponential: sum of durations (duration_mean*Mnm, impulses.jl:84-96);
 *           LogitNormal: log_duration_sum  impulses.jl:230-240
 *   S2[K*K] LogitNormal: log_duration_variation around S1/Mnm  impulses.jl:242-252 (two-pass); Exponential: zeros.
 * Unsharded use only (sharded ranks go through the *_dev accessors below and allreduce). */
int nhp_cont_suffstats(nhp_ctx *ctx, nhp_events *ev, double *M0, double *Mn, double *Mnm, double *S1, double *S2);

/* resample_adjacency_matrix!(process, data)  continuous.jl:444-519: Gibbs over A[:,c], columns
 * independent, p sequential.  rho[K*K] = link_probability(network) (networks.jl:65-68);
 * u[K*K] uniforms (u[p + K*c]; Bernoulli draw is u <= p1) or NULL for Philox (seed, counter).
 * A_inout is read (current state), updated, and also becomes the context's A. */
int nhp_cont_resample_adjacency(nhp_ctx *ctx, nhp_events *ev, const double *rho, uint64_t seed, uint64_t counter,
                                const double *u, double *A_inout);
/* Multi-GPU form: columns are conditionally independent (the reference's Threads.@threads axis,
 * continuous.jl:462-464), so rank r of R resamples only the columns c with c % col_stride == col_begin
 * (events replicated on every rank) and leaves the others untouched; the host then exchanges the
 * owned columns (allgather / masked allreduce).  col_begin = 0, col_stride = 1 is the full sweep. */
int nhp_cont_resample_adjacency_cols(nhp_ctx *ctx, nhp_events *ev, const double *rho, uint64_t seed, uint64_t counter,
                                     const double *u, double *A_inout, int64_t col_begin, int64_t col_stride);
/* Device-resident form for chains (`resample!` of a network process, continuous.jl:350-358, without the K^2 matrices crossing
 * PCIe): the sweep runs in place on the context's adjacency matrix with the scalar link probability `rho` of a
 * BernoulliNetworkModel (networks.jl:65-68; rho < 0: the value kept by nhp_cont_network_set / nhp_cont_resample_network) and
 * Philox uniforms.  commit != 0 rebuilds the masked tables afterwards; a multi-GPU caller passes 0, exchanges the owned
 * columns (nhp_comm_allgather_adjacency) and commits once. */
int nhp_cont_resample_adjacency_dev(nhp_ctx *ctx, nhp_events *ev, double rho, uint64_t seed, uint64_t counter, int64_t col_begin,
                                    int64_t col_stride, int commit);
int nhp_cont_adjacency_commit(nhp_ctx *ctx);
/* resample!(network::BernoulliNetworkModel, data)  networks.jl:72-78: rho ~ Beta(alpha + sum(A), beta + K^2 - sum(A)) from the
 * device-resident adjacency matrix (Philox: seed, counter); the value stays with the context and is returned in *rho_out. */
int nhp_cont_network_set(nhp_ctx *ctx, double rho);
int nhp_cont_network_get(const nhp_ctx *ctx, double *rho);
int nhp_cont_resample_network(nhp_ctx *ctx, uint64_t seed, uint64_t counter, double alpha, double beta, double *rho_out);

/* Device-side conjugate draws of one Gibbs sweep (the `resample!` of baseline, weights and impulses:
 * baselines.jl:72-77, weights.jl:59-64, impulses.jl:68-73 / 204-214) from the statistics of the last parent sweep,
 * in place: the context's parameters are replaced and every derived table is rebuilt, so a chain can run without the
 * K^2 statistics or parameters crossing PCIe.  hyper: [alpha0, beta0 (baseline), kappa, nu (weights), then
 * Exponential: alpha, beta | LogitNormal: mumu, kappamu, alpha0, beta0]; `duration` is T of the whole data set.
 * flags bit 0: run the LogitNormal second pass (S2) first (single GPU); without it the caller has completed the
 * statistics (multi-GPU: all-reduce phase 0, nhp_cont_suffstats_second_pass, all-reduce phase 1) and every rank,
 * holding the same statistics, draws the same parameters (Philox keyed by seed, element, counter).
 * Parity with the reference is distributional. */
int nhp_cont_resample_params(nhp_ctx *ctx, nhp_events *ev, uint64_t seed, uint64_t counter, double duration, const double *hyper, int n_hyper, int flags);
/* Current parameters in the layouts of nhp_cont_params_set; any pointer may be NULL. */
int nhp_cont_params_get(nhp_ctx *ctx, double *lambda0, double *W, double *A, double *p1, double *p2);
/* Device-side sample trace of `mcmc!` (inference.jl:49-70; the reference pushes params(process) = [rho; lambda0; W; theta | mu, tau;
 * vec(A)] per sweep, continuous.jl:325-333).  _begin reserves `capacity` slots for the context's current model (real-valued
 * parameters as they are, the adjacency matrix bit-packed: K^2 / 8 bytes); _push appends the context's current parameters
 * (device-to-device on the context's stream, no host synchronisation) -- nhp_cont_gibbs_sweep does it by itself while a trace is
 * open; _read copies samples [first, first + count) to the host, one sample after the other in the layouts of
 * nhp_cont_params_get (rho[count], lambda0[count*K], W | A | p1 | p2 [count*K*K]; any pointer may be NULL).  A trace begun while the
 * context holds curves and their prior also keeps the K x n_grid curves of every sample (_read_curves: values[g + n_grid*(k + K*j)]
 * for sample first + j; NHP_ERR_STATE for a trace without curves); _push then refuses a grid of another size. */
int nhp_cont_trace_begin(nhp_ctx *ctx, int64_t capacity);
int nhp_cont_trace_push(nhp_ctx *ctx);
int nhp_cont_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity);
int nhp_cont_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *rho, double *lambda0, double *W, double *A, double *p1, double *p2);
int nhp_cont_trace_free(nhp_ctx *ctx);
int nhp_cont_trace_read_curves(nhp_ctx *ctx, int64_t first, int64_t count, double *values);
/* Mean-field VB of a continuous standard process with its state on the device (the reference's `vb!` is discrete only).  The model is
 * the one of the Gibbs sweep: lambda0_k ~ Gamma(alpha0, beta0), W[p,c] ~ Gamma(kappa, nu), Exponential theta ~ Gamma(alpha, beta) or
 * LogitNormal (mu, tau) ~ NormalGamma(mumu, kappamu, a0, b0) (all Gammas with rates), and the factorised posterior
 *   q = [alphav(K); betav(K); kappav(K*K); nuv(K*K)], then Exponential atheta(K*K); btheta(K*K)  (2 K + 4 K*K doubles)
 *                                                    or LogitNormal mv(K*K); lambdav(K*K); av(K*K); bv(K*K)  (2 K + 6 K*K doubles),
 * K*K planes parent-major (X[p + K*c]): q(lambda0_k) = Gamma(alphav, betav), q(W) = Gamma(kappav, nuv), q(theta) = Gamma(atheta, btheta),
 * q(mu, tau) = NormalGamma(mv, lambdav, av, bv).  _set takes the kind, K and dtmax of the current nhp_cont_params_set; hyper = [alpha0,
 * beta0, kappa, nu, then alpha, beta | mumu, kappamu, a0, b0] (n_hyper 6 or 8, that of the kind), every entry finite and > 0 except
 * mumu (finite); every entry of q finite and > 0 except mv (finite).  Otherwise NHP_ERR_INVALID (NHP_ERR_STATE without parameters)
 * and the kept state is as it was.  _get copies q back.
 * The E-step evaluates the parent probabilities at effective parameters, for which ln W_eff + ln h(dt) = E_q[ln W + ln h(dt)]:
 *   lambda0_eff = exp(psi(alphav) - ln betav); Exponential theta_eff = atheta / btheta, W_eff = exp(psi(kappav) - ln nuv + psi(atheta)
 *   - ln btheta) / theta_eff; LogitNormal mu_eff = mv, tau_eff = av / bv, W_eff = exp(psi(kappav) - ln nuv + (psi(av) - ln av) / 2
 *   - 1 / (2 lambdav));
 * with Z_i the total intensity at event i and u = W_eff h(t_i - t_j) / Z_i over the window of nhp_cont_resample_parents (dtmax for
 * LogitNormal, the cut-off horizon of nhp_cont_horizon for Exponential, both at the effective parameters):
 *   M0[k] = sum over the events of node k of lambda0_eff[k] / Z_i;  Mnm = sum u;  S1 = sum u (t_i - t_j) (Exponential) or sum u (y - mv)
 *   with y = logit((t_i - t_j) / dtmax) (LogitNormal);  S2 = sum u (y - mv)^2 (LogitNormal; zeros for Exponential).
 * nhp_cont_vb_stats runs the E-step only and returns those sums in the layouts of nhp_cont_suffstats (any output may be NULL); q does
 * not change.  nhp_cont_vb_step then updates q in place: alphav = alpha0 + M0, betav = beta0 + T (T the duration of ev), kappav =
 * kappa + Mnm, nuv = nu + Mn[p]; Exponential atheta = alpha + Mnm, btheta = beta + S1; LogitNormal, with n = Mnm, d = S1 / n (0 for
 * n = 0), ybar = mv + d, S = max(S2 - n d^2, 0): lambdav = kappamu + n, mv = (kappamu mumu + n ybar) / lambdav, av = a0 + n / 2,
 * bv = b0 + S / 2 + kappamu n (ybar - mumu)^2 / (2 lambdav) -- the textbook Normal-Gamma update, which keeps b0 where the Gibbs draw
 * of nhp_cont_resample_params does not (quirk Q5).  A pair with n = 0 gets its prior.  change (may be NULL) = the largest of
 * |new - old| / old over the positive entries and |new - old| over mv, the only value that crosses PCIe; then a push to the VB trace
 * while it has room.  After either call the context's parameters are the posterior means of q (alphav / betav, kappav / nuv, atheta /
 * btheta | mv, av / bv) with every table rebuilt, so nhp_cont_loglik, nhp_cont_intensity or nhp_cont_params_get see the fitted model;
 * the parent assignment and gradient of earlier calls are invalidated.  Refused before anything changes: a network process (A set),
 * LogGaussianCox curves set, a time shard (n_halo > 0) or a communicator of more than one rank (NHP_ERR_UNSUPPORTED); no parameters, no
 * VB state, or a kind or K that changed since _set (NHP_ERR_STATE); an events handle of another K (NHP_ERR_INVALID); for _step, an
 * open VB trace begun for another kind or K (NHP_ERR_STATE). */
int nhp_cont_vb_set(nhp_ctx *ctx, const double *hyper, int n_hyper, const double *q);
int nhp_cont_vb_get(nhp_ctx *ctx, double *q);
int nhp_cont_vb_stats(nhp_ctx *ctx, nhp_events *ev, double *M0, double *Mnm, double *S1, double *S2);
int nhp_cont_vb_step(nhp_ctx *ctx, nhp_events *ev, double *change);
/* Mean-field VB of a continuous network process with a BernoulliNetworkModel, the model of the discrete network VB
 * (nhp_disc_vb_network_set): A[p,c] ~ Bernoulli(rho), rho ~ Beta(alpha_rho, beta_rho), W | A=1 ~ Gamma(kappa, nu) (the slab), W | A=0 ~
 * Gamma(kappa0, nu0) (the spike), W entering the intensity directly; lambda0, theta | (mu, tau) with the priors of nhp_cont_vb_set.
 * The state extends the standard layout: q = [standard q; kappa0v(K*K); nu0v(K*K); pv(K*K); alpharhov; betarhov] (2 K + 7 K*K + 2
 * doubles for Exponential, 2 K + 9 K*K + 2 for LogitNormal), pv[p + K*c] = q(A[p,c] = 1); hyper = [hyper of nhp_cont_vb_set; kappa0,
 * nu0, alpha_rho, beta_rho] (10 or 12 entries).  _network_set validates (every hyper-parameter finite and > 0 except mumu; every entry
 * of q finite and > 0 except mv (finite) and pv (in [0, 1]); otherwise NHP_ERR_INVALID, NHP_ERR_STATE without parameters, and the kept
 * state is as it was) and keeps a state of network kind; nhp_cont_vb_set keeps a standard one, and the later call decides the kind.
 * nhp_cont_vb_get, _stats, _step and the VB trace serve both kinds.  On a network state the E-step is the standard one with
 * lW = pv (psi(kappav) - ln nuv) + (1 - pv) (psi(kappa0v) - ln nu0v) in place of psi(kappav) - ln nuv; no link has a zero effective
 * weight, so it sweeps the process as a standard one (no adjacency mask, and the events handle's cached pair structure is neither used
 * nor dropped).  The step's update is the standard one plus, with G = Mnm[p,c] and E = Mn[p], kappa0v = kappa0 + G, nu0v = nu0 + E,
 *   logit pv = psi(alpharhov) - psi(betarhov) + [lgamma(kappav) - kappav ln nuv] - [lgamma(kappa0v) - kappa0v ln nu0v]
 *              + [kappa ln nu - lgamma(kappa)] - [kappa0 ln nu0 - lgamma(kappa0)]
 * (the new kappav, nuv, kappa0v, nu0v; the old q(rho)) and, with S = sum of pv in a fixed order (the same state and statistics give the
 * same bits), alpharhov = alpha_rho + S, betarhov = beta_rho + K*K - S.  change also covers |new - old| over pv.  After either call
 * the context holds lambda0 = alphav / betav, W = kappav / nuv (the slab mean), A = [pv > 1/2], p1 and p2 as for the standard state,
 * and the rho of nhp_cont_network_set = alpharhov / (alpharhov + betarhov), so nhp_cont_loglik, nhp_cont_params_get and a following
 * nhp_cont_gibbs_sweep see a network process at the VB point estimate.  Refused before anything changes, for a network state:
 * parameters without an adjacency matrix, a kind or K changed since _set, or an open VB trace begun for the other kind of state
 * (NHP_ERR_STATE); LogGaussianCox curves, a time shard or more than one rank (NHP_ERR_UNSUPPORTED); events of another K
 * (NHP_ERR_INVALID).  A standard state still refuses a network process (NHP_ERR_UNSUPPORTED). */
int nhp_cont_vb_network_set(nhp_ctx *ctx, const double *hyper, int n_hyper, const double *q);
/* Device-side trace of the continuous VB state, independent of every other trace: one slot is q (laid out for the state at _begin,
 * standard or network); _read copies slots [first, first + count) one after the other. */
int nhp_cont_vb_trace_begin(nhp_ctx *ctx, int64_t capacity);
int nhp_cont_vb_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity);
int nhp_cont_vb_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *q_out);
int nhp_cont_vb_trace_free(nhp_ctx *ctx);

/* ---- multi-GPU (one process and one context per GPU; NCCL over NVLink, loaded with dlopen) ---------------------
 * SURVEY.md section 8e.  Time shards (nhp_events_upload with n_halo / index_base) carry the log-likelihood, the parent
 * sweep and the statistics; the adjacency sampler partitions the child columns over the ranks on a replicated stream.
 * The host distributes the 128-byte id of rank 0 (nhp_comm_unique_id) by any means it has (MPI.jl, Distributed.jl, a
 * file) and every rank calls nhp_comm_init; the collectives below then run on the context's stream.  On a context
 * without a communicator they are no-ops, so one call sequence serves 1..N GPUs:
 *   resample_parents -> nhp_comm_allreduce_stats(0) -> nhp_cont_suffstats_second_pass -> nhp_comm_allreduce_stats(1)
 *   -> nhp_cont_resample_params(flags = 0) | nhp_cont_suffstats_read
 *   -> nhp_cont_resample_adjacency_dev(col_begin = rank, col_stride = nranks, commit = 0) -> nhp_comm_allgather_adjacency
 * nhp_cont_gibbs_sweep runs exactly that sequence (the whole `resample!` of continuous.jl:202-208 / 350-358).
 * Statistics buffers (device, contiguous doubles):
 *   [ ll_logsum, ll_rowsum, M0[K], Mn[K], Mnm[K*K], S1[K*K] ]   (phase 0)
 *   [ S2[K*K] ]                                                 (phase 1) */
int nhp_comm_unique_id(void *id128);
int nhp_comm_init(nhp_ctx *ctx, const void *id128, int rank, int nranks);
int nhp_comm_destroy(nhp_ctx *ctx);
int nhp_comm_rank(const nhp_ctx *ctx, int *rank, int *nranks);
int nhp_comm_allreduce_stats(nhp_ctx *ctx, int phase);
/* sum of a small host vector over the ranks (log-likelihood shares of nhp_cont_loglik, ...) */
int nhp_comm_allreduce_host(nhp_ctx *ctx, double *inout, int64_t n);
int nhp_comm_allgather_adjacency(nhp_ctx *ctx);
/* The replicated stream from the time shards: every rank passes the shard it uploaded (consecutive pieces of one stream:
 * index_base of rank r = number of own events of the ranks before it) and receives an ordinary unsharded events handle with all
 * events -- the own events of the shards travel over NVLink (ncclBroadcast per rank) instead of every rank uploading the whole
 * stream through PCIe.  Needs a communicator; a single GPU uses its handle as is. */
int nhp_comm_allgather_events(nhp_ctx *ctx, nhp_events *ev_shard, nhp_events **out);
/* hyper as for nhp_cont_resample_params; net_alpha > 0: BernoulliNetworkModel with rho ~ Beta(net_alpha, net_beta) prior
 * (networks.jl:45-54, 72-78), else link probability 1 (DenseNetworkModel).  ev_full (the unsharded stream, replicated on
 * every rank) is only used by network processes; pass ev_shard itself on a single GPU.  With grid baseline curves and their prior
 * (nhp_cont_baseline_prior) the sweep runs nhp_cont_resample_baseline(seed, counter) after the conjugate draws and before the
 * adjacency sweep.  A network process with curves but no prior is refused with NHP_ERR_UNSUPPORTED before anything changes; a
 * standard process with curves but no prior keeps its curves. */
int nhp_cont_gibbs_sweep(nhp_ctx *ctx, nhp_events *ev_shard, nhp_events *ev_full, uint64_t seed, uint64_t counter, double duration,
                         const double *hyper, int n_hyper, double net_alpha, double net_beta);
/* Device pointer + length (in doubles) of a statistics buffer, for hosts that run their own collectives. */
int nhp_cont_stats_dev(nhp_ctx *ctx, int phase, void **ptr_dev, int64_t *count);
int nhp_cont_suffstats_second_pass(nhp_ctx *ctx, nhp_events *ev);
int nhp_cont_suffstats_read(nhp_ctx *ctx, double *M0, double *Mn, double *Mnm, double *S1, double *S2);
/* log-likelihood share left on the device in the phase-0 buffer slots 0..1 (no host sync) */
int nhp_cont_loglik_dev(nhp_ctx *ctx, nhp_events *ev, int recursive);

/* ---- discrete path -------------------------------------------------------------------- */
/* data::Matrix{Int64} N x T, data[n + N*t]  (discrete.jl:18).  Sharding: `t_halo` leading bins are
 * read-only history for the convolution. */
int nhp_disc_upload(nhp_ctx *ctx, const int64_t *data, int64_t N, int64_t T, int64_t t_halo, nhp_disc **out);
int nhp_disc_free(nhp_ctx *ctx, nhp_disc *dd);
/* rand(process::DiscreteHawkesProcess, T)  discrete.jl:20-38: one N x T sample of the discrete process whose parameters the context
 * holds (nhp_disc_params_set; standard, or network with A), simulated on the device and left there as an unsharded (t_halo = 0),
 * not yet convolved count handle -- the same handle nhp_disc_upload would make of the sample.  The law is the one nhp_disc_loglik
 * evaluates: given the earlier bins, data[c, t] ~ Poisson(lambda[t, c]) independently, lambda as nhp_disc_intensity returns it with
 * phi = nhp_disc_basis(L, B, dt) and no events before bin 0; it is drawn in the cluster representation (baseline events, then
 * Poisson children per event, generation by generation).  L is the impulse response's nlags.  Philox keyed by `seed`: the sample is a
 * deterministic function of (parameters, T, L, seed); parity with the reference is distributional.  Refused, with no handle and
 * nothing left allocated: no discrete parameters (NHP_ERR_STATE); T < 1, N*T >= 2^31, L < 1 or L*B > 4096, a negative or non-finite
 * lambda0, [A]W or theta, or a sample of more than max_events generated events, dropped children included (NHP_ERR_INVALID).
 * nhp_disc_download copies every bin of a handle (halo included) to the host as data[n + N*t]; nhp_disc_events_count gives the
 * events in its own bins. */
int nhp_disc_rand(nhp_ctx *ctx, int64_t T, int64_t L, uint64_t seed, int64_t max_events, nhp_disc **out);
int nhp_disc_download(nhp_ctx *ctx, nhp_disc *dd, int64_t *data);
int64_t nhp_disc_events_count(const nhp_disc *dd);
/* basis(impulse)  impulses.jl:321-335 -> phi[l + L*b] */
int nhp_disc_basis(int64_t L, int64_t B, double dt, double *phi);
/* convolve(process, data)  discrete.jl:146-151; result stays on the device; conv_out (T*N*B,
 * conv[t + T*(n + N*b)]) may be NULL */
int nhp_disc_convolve(nhp_ctx *ctx, nhp_disc *dd, const double *phi, int64_t L, int64_t B, double *conv_out);
/* the device-resident convolution in the reference's layout conv[t + T*(n + N*b)], for host code that indexes `convolved` */
int nhp_disc_conv_export(nhp_ctx *ctx, nhp_disc *dd, double *conv_out);
/* lambda0[N], W[N*N], A[N*N]|NULL, theta[N*N*B] (theta[p + N*(c + N*b)]), dt   discrete.jl:161-170, 395-402 */
int nhp_disc_params_set(nhp_ctx *ctx, int64_t N, int64_t B, const double *lambda0, const double *W, const double *A,
                        const double *theta, double dt);
/* intensity(process, convolved)  discrete.jl:115-129 -> lam[t + T*c] */
int nhp_disc_intensity(nhp_ctx *ctx, nhp_disc *dd, double *lam);
/* loglikelihood(process, data, convolved)  discrete.jl:91-102 */
int nhp_disc_loglik(nhp_ctx *ctx, nhp_disc *dd, double *ll);
/* Extension for the discrete `mle!` (discrete.jl:211-296; the reference differentiates numerically): the log-likelihood of
 * nhp_disc_loglik (ll may be NULL) and its analytic gradient in the layouts of nhp_disc_params_set -- dlambda0[N], dW[N*N]
 * (dW[p + N*c]), dtheta[N*N*B] (dtheta[p + N*(c + N*b)]); entries with A[p,c] = 0 get 0.  The T x N x (N B) contraction collapses to the
 * non-zero bins plus the conv column sums.  Time shards return additive shares. */
int nhp_disc_loglik_grad(nhp_ctx *ctx, nhp_disc *dd, double *ll, double *dlambda0, double *dW, double *dtheta);
/* resample_parents(process, data, convolved) reduced over t  parents.jl:82-134:
 * counts[c + N*k], k = 0 baseline, k = 1 + p*B + b.  u (one uniform per event, consumed in
 * (t outer, c inner, draw) order) or NULL for Philox. */
int nhp_disc_gibbs_counts(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *u, int64_t nu, double *counts);
/* The conjugate draws of the discrete `resample!` (discrete.jl:361-367 / 416-424) on the device, from the counts the last
 * nhp_disc_gibbs_counts left there (its `counts` argument may be NULL):  lambda0[c] ~ Gamma(alpha0 + counts[c,0], 1/(beta0 + T dt))
 * (baselines.jl:413-419, intended form), W[p,c] ~ Gamma(kappa + sum_b counts[c,p,b], 1/(nu + Mn[p])) (weights.jl:59-64),
 * theta[p,c,:] ~ Dirichlet(gamma + counts[c,p,:]) (impulses.jl:337-353).  Mn[N] = events per node; hyper = [alpha0, beta0, kappa, nu,
 * gamma]; Philox keyed (seed, element, counter).  The new parameters replace the context's (every derived table is rebuilt on the
 * device) and are returned in the layouts of nhp_disc_params_set.  Parity with the reference is distributional. */
int nhp_disc_resample_params(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *Mn, const double *hyper, int n_hyper,
                             double *lambda0, double *W, double *theta);
/* update_parents + the three VB reductions  parents.jl:136-177, baselines.jl:444-452,
 * weights.jl:70-91, impulses.jl:355-371.  e0[N], E[N*N*B] are the exp-expectations. */
int nhp_disc_vb_stats(nhp_ctx *ctx, nhp_disc *dd, const double *e0, const double *E, double *alpha_sum, double *kappa_sum,
                      double *nu_sum, double *gamma_sum);
/* resample_adjacency_matrix!(process, data, convolved)  discrete.jl:426-480 */
int nhp_disc_resample_adjacency(nhp_ctx *ctx, nhp_disc *dd, const double *rho, uint64_t seed, uint64_t counter, const double *u,
                                double *A_inout);
/* Current parameters in the layouts of nhp_disc_params_set; any pointer may be NULL (A: NHP_ERR_STATE for a standard process). */
int nhp_disc_params_get(nhp_ctx *ctx, double *lambda0, double *W, double *A, double *theta);
/* Device-resident form for chains (`resample_adjacency_matrix!` of discrete.jl:426-460 without the N^2 matrices crossing PCIe):
 * the sweep runs in place on the context's adjacency matrix with the scalar link probability `rho` of a BernoulliNetworkModel
 * (networks.jl:65-68; rho < 0: the value kept by nhp_disc_network_set / nhp_disc_gibbs_sweep) and Philox uniforms keyed
 * (seed, p + N c, counter), as nhp_disc_resample_adjacency with u = NULL; the derived tables follow the new matrix.  Unsharded
 * data only (NHP_ERR_UNSUPPORTED for t_halo > 0). */
int nhp_disc_resample_adjacency_dev(nhp_ctx *ctx, nhp_disc *dd, double rho, uint64_t seed, uint64_t counter);
/* Link probability of the discrete BernoulliNetworkModel (networks.jl:45-54) kept with the context, apart from the continuous
 * model's (nhp_cont_network_set). */
int nhp_disc_network_set(nhp_ctx *ctx, double rho);
int nhp_disc_network_get(const nhp_ctx *ctx, double *rho);
/* Device-side sample trace of the discrete `mcmc!` (inference.jl:49-70; the reference pushes params(process) per sweep,
 * discrete.jl:178-182 / 406-414).  Same semantics as nhp_cont_trace_*: one slot holds (rho, lambda0[N], W[N*N], theta[N*N*B]) and
 * the adjacency matrix bit-packed; _push appends the context's current discrete parameters and rho (nhp_disc_gibbs_sweep does it
 * while the trace has room) and refuses a model whose N or B changed, or that gained or lost A, since _begin; _read copies samples
 * [first, first + count) in the layouts of nhp_disc_params_get, one after the other (any pointer may be NULL).  The discrete trace
 * is independent of the continuous one. */
int nhp_disc_trace_begin(nhp_ctx *ctx, int64_t capacity);
int nhp_disc_trace_push(nhp_ctx *ctx);
int nhp_disc_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity);
int nhp_disc_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *rho, double *lambda0, double *W, double *A, double *theta);
int nhp_disc_trace_free(nhp_ctx *ctx);
/* One whole Gibbs sweep of the discrete `resample!` (discrete.jl:361-367 / 416-424) on the device, with no N^2-sized host transfer:
 * parent counts (Philox: seed, uniform index, counter), the conjugate draws of nhp_disc_resample_params from them (Mn = the events
 * per node kept with the data), and for a network process the in-place adjacency sweep (nhp_disc_resample_adjacency_dev with counter
 * + 2^40) followed, when net_alpha > 0, by rho ~ Beta(net_alpha + sum(A), net_beta + N^2 - sum(A)) (networks.jl:72-78; otherwise link
 * probability 1, DenseNetworkModel); then a push to the discrete trace while it has room.  Given the same (seed, counter) and state,
 * lambda0, W, theta and A equal those of nhp_disc_gibbs_counts + nhp_disc_resample_params + nhp_disc_resample_adjacency.  hyper as
 * for nhp_disc_resample_params (n_hyper = 5).  Time-sharded data or a communicator of more than one rank: NHP_ERR_UNSUPPORTED,
 * before anything changes. */
int nhp_disc_gibbs_sweep(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *hyper, int n_hyper, double net_alpha,
                         double net_beta);
/* Mean-field VB of a discrete standard process (`vb!`, inference.jl:153-181) with its state on the device.  The state is the
 * reference's variational_params vector (discrete.jl:204-209), q = [alphav(N); betav(N); vec(gammav)(N*N*B); vec(kappav)(N*N);
 * vec(nuv)(N*N)] with gammav[p + N*(c + N*b)], kappav[p + N*c], nuv[p + N*c].  _set validates (every entry of q and hyper finite and
 * > 0, dt > 0) and keeps q, hyper = [alpha0, beta0, kappa, nu, gamma] and dt with the context (buffers grow with N or B only, and are
 * freed by nhp_destroy); _get copies q back. */
int nhp_disc_vb_set(nhp_ctx *ctx, int64_t N, int64_t B, double dt, const double *hyper, int n_hyper, const double *q);
int nhp_disc_vb_get(nhp_ctx *ctx, double *q);
/* One `update!(process, data, convolved)` (discrete.jl:369-375) on the device: the exp-expectations from q (digamma on the device),
 * the statistics of nhp_disc_vb_stats, then in place alphav = alpha0 + alpha_sum, betav = 1/beta0 + T dt (baselines.jl:450 as
 * written), gammav = gamma + gamma_sum, kappav = kappa + kappa_sum, nuv = nu + events of the parent node; then a push to the VB trace
 * while it has room.  change (may be NULL) = max_i |q_new[i] - q_old[i]| / q_old[i], the only value that crosses PCIe.  Needs
 * nhp_disc_convolve.  Refused before anything changes: time-sharded data or a communicator of more than one rank
 * (NHP_ERR_UNSUPPORTED); no state or no convolution (NHP_ERR_STATE); N or B of the state not those of dd (NHP_ERR_INVALID); an open
 * VB trace whose slot size is not the state's (NHP_ERR_STATE). */
int nhp_disc_vb_step(nhp_ctx *ctx, nhp_disc *dd, double *change);
/* One step of stochastic variational inference (Hoffman et al. 2013; the reference's `svi!`, inference.jl:183-190, is an empty stub)
 * on the state of nhp_disc_vb_set, from the window of n_bins bins (t_begin + j) mod T, j = 0 .. n_bins - 1, of the T bins of dd; a
 * window may wrap around the end, so with t_begin uniform on [0, T) every bin is in it with probability n_bins / T and the scaled
 * statistics are unbiased.  With s = T / n_bins and the statistics of nhp_disc_vb_stats over the window's bins only (the convolution
 * still covers the whole series, so the window's responsibilities are exact), the targets are alphav* = alpha0 + s alpha_sum,
 * betav* = 1/beta0 + T dt (the full-data value, unscaled), gammav* = gamma + s gamma_sum, kappav* = kappa + s kappa_sum, nuv* = nu + s
 * (events of the parent node in the window), and in place q = (1 - step) q + step q*; then a push to the VB trace while it has room.
 * t_begin = 0, n_bins = T, step = 1 is the arithmetic of nhp_disc_vb_step.  The kernels visit only the window's non-zero bins.  change
 * (may be NULL) as for nhp_disc_vb_step.  Refused before anything changes, as nhp_disc_vb_step, and also: a window outside
 * 0 <= t_begin < T, 1 <= n_bins <= T, or step outside (0, 1] or not finite (NHP_ERR_INVALID). */
int nhp_disc_svi_step(nhp_ctx *ctx, nhp_disc *dd, int64_t t_begin, int64_t n_bins, double step, double *change);
/* Mean-field VB of a discrete network process with a BernoulliNetworkModel (the reference's update! for it, discrete.jl:494-502,
 * is non-functional, quirk Q10).  A true spike W = A W' gives E[ln W] = -inf whenever q(A=1) < 1, so the model is a Gamma mixture:
 * A[p,c] ~ Bernoulli(rho), rho ~ Beta(alpha_rho, beta_rho), W | A=1 ~ Gamma(kappa, nu) (the slab), W | A=0 ~ Gamma(kappa0, nu0) (the
 * spike), lambda0 and theta as for the standard process, W entering the intensity directly.  The state extends the standard layout:
 * q = [alphav(N); betav(N); gammav(N*N*B); kappav(N*N); nuv(N*N); kappa0v(N*N); nu0v(N*N); pv(N*N); alpharhov; betarhov]
 * (2 N + N*N*(B + 5) + 2 doubles), with q(W | A=1) = Gamma(kappav, nuv), q(W | A=0) = Gamma(kappa0v, nu0v), pv[p + N*c] = q(A[p,c] = 1),
 * q(rho) = Beta(alpharhov, betarhov); hyper = [alpha0, beta0, kappa, nu, gamma, kappa0, nu0, alpha_rho, beta_rho] (n_hyper = 9).
 * _network_set validates (every hyper-parameter and every entry of q finite and > 0, except pv: in [0, 1]; dt > 0; otherwise
 * NHP_ERR_INVALID and the kept state is as it was) and keeps a state of network kind; nhp_disc_vb_set keeps a standard one, and the
 * later of the two calls decides the kind.  nhp_disc_vb_get, nhp_disc_vb_step, nhp_disc_svi_step and the VB trace work on either.
 * On a network state a step over the window (s = T / n_bins; the VB step is s = 1, step = 1) takes the expectations from the old q,
 * with E[ln W] = pv (psi(kappav) - ln nuv) + (1 - pv) (psi(kappa0v) - ln nu0v), and the statistics of nhp_disc_vb_stats; with
 * G = s sum_b gamma_sum[p,c,b] and E = s (events of p in the window), the targets are those of the standard step, kappa0v* = kappa0 + G,
 * nu0v* = nu0 + E, and
 *   logit pv* = psi(alpharhov) - psi(betarhov) + [lgamma(kappav*) - lgamma(kappa) + kappa ln nu - kappav* ln nuv*]
 *                                              - [lgamma(kappa0v*) - lgamma(kappa0) + kappa0 ln nu0 - kappa0v* ln nu0v*]
 * (the log marginal likelihoods of the link's statistics under slab and spike), then with S = sum of pv* (a fixed-order two-stage
 * sum: the same state and statistics give the same bits) alpharhov* = alpha_rho + S, betarhov* = beta_rho + N*N - S (unscaled: N*N
 * counts links).  Every entry moves to (1 - step) q + step q* in place; then a push to the VB trace while it has room.  change = the
 * largest of |new - old| / old over the positive entries and |new - old| over pv.  Refusals as for the standard steps; a step on an
 * open VB trace begun for the other kind of state is NHP_ERR_STATE. */
int nhp_disc_vb_network_set(nhp_ctx *ctx, int64_t N, int64_t B, double dt, const double *hyper, int n_hyper, const double *q);
/* Device-side trace of the VB state, independent of the Gibbs traces: one slot is q (2 N + N*N*(B + 2) doubles for a standard state,
 * 2 N + N*N*(B + 5) + 2 for a network state, laid out for the state at _begin); _read copies slots [first, first + count) one after
 * the other. */
int nhp_disc_vb_trace_begin(nhp_ctx *ctx, int64_t capacity);
int nhp_disc_vb_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity);
int nhp_disc_vb_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *q_out);
int nhp_disc_vb_trace_free(nhp_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
