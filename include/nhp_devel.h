/*
 * nhp_devel.h -- measurement and test hooks of libnhp.  NOT part of the drop-in boundary (include/nhp.h): nothing a Julia
 * binding needs lives here.  bench.py and tests/ use these to measure roofline denominators, to count launches, to check the
 * table-driven log/exp, and to rewind the device-resident parameters between timed steps.
 */
#ifndef NHP_DEVEL_H
#define NHP_DEVEL_H
#include "nhp.h"
#ifdef __cplusplus
extern "C" {
#endif

/* kernels launched by this context since creation (bench.py's gpu_launches claim) */
int64_t nhp_launch_count(const nhp_ctx *ctx);
/* Roofline denominators measured on this device: which = 0 FP64 FMA peak [TFLOP/s], 1 LogitNormal / 2 Exponential
 * register-resident impulse evaluations [pairs/s], 3 FP64 tensor-core (mma.sync m8n8k4.f64) peak [TFLOP/s],
 * 4 adjacency-bit probes [probes/s] (one shared-memory node id + one shared-memory bit-row word per probe, the
 * inner loop of the sparse sweep's filter with nothing else around it). */
int nhp_bench_fp64(nhp_ctx *ctx, int which, double *result);
/* Test hook for the table-driven FP64 log (which = 0) / exp (which = 1) the impulse evaluation uses, and for the digamma of the
 * VB expectations (which = 2, x > 0): out[i] = f(x[i]), host pointers. */
int nhp_test_fastmath(nhp_ctx *ctx, int which, const double *x, int64_t n, double *out);
/* Last adjacency sweep of this context: out8 = [steps taken, batches, flips, recomputed steps, cached pairs,
 * virtual columns, sweep kernel ms, structure build ms]. */
int nhp_cont_adjacency_info(const nhp_ctx *ctx, double *out8);
/* Last nhp_cont_gibbs_sweep of this context: out8 = [parent sweep ms, second pass + conjugate draws + table rebuild ms,
 * adjacency sweep kernel ms, slice update of the curves ms, its rounds, 0...]. */
int nhp_cont_sweep_info(const nhp_ctx *ctx, double *out8);
/* Last nhp_cont_resample_baseline of this context: out4 = [list build ms (draws, prior draw, baseline-event records, work items),
 * rounds + commit ms, rounds, work items]. */
int nhp_cont_slice_info(const nhp_ctx *ctx, double *out4);
/* Keep / bring back a device-side copy of the continuous parameters (lambda0, W, A, p1, p2) and rebuild the tables:
 * bench.py rewinds a chain to the workload's parameters between timed steps without a host round trip. */
int nhp_cont_params_save(nhp_ctx *ctx);
int nhp_cont_params_restore(nhp_ctx *ctx);

#ifdef __cplusplus
}
#endif
#endif
