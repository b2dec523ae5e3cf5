// fastmath.cuh -- table-driven FP64 log/exp for the impulse evaluation.
//
// The continuous sweeps are bound by the FP64 pipe / instruction issue: with libdevice log/exp/div a
// LogitNormal pair costs ~80 DP instructions.  The parity contract is 1e-10 relative on intensities,
// so an implementation with ~1e-15 absolute error in log and ~2e-16 relative error in exp is exact
// for the purpose while costing 11 + 10 DP instructions (tables in shared memory, integer work on the
// ALU pipe, polynomial coefficients as constant-bank operands).
//   log(x)  = e ln2 + (-log c_i) + log1p(m c_i - 1),   c_i ~ 1/m on the i-th of 32 mantissa intervals
//             (32 x 16 B = four 128 B rows: a warp's lookup costs at most 4 shared-memory wavefronts)
//   exp(x)  = 2^(k/64) (1 + expm1(r)),                  k = round(64 x / ln2), r = x - k ln2/64
// Tables are correctly rounded (tools/gen_fastmath_tables.py).  Also here: the digamma of the discrete VB step (no tables).
#pragma once
#include <cuda_runtime.h>
#include "fastmath_tables.h"

struct FastTables {
    double2 logtab[32];   // {c, -log c}
    double exptab[64];    // 2^(j/64)
};

// polynomial coefficients and split constants live in the constant bank so a DFMA can take them as
// an operand (no per-use 64-bit immediate moves)
struct FastConsts {
    double l8, l7, l6, l5, l4, l3, l2;   // log1p: -1/8, 1/7, -1/6, 1/5, -1/4, 1/3, -1/2
    double ln2_hi, ln2_lo, emagic;       // e ln2 split; 2^52 + 2^31
    double e5, e4, e3, e2;               // expm1: 1/120, 1/24, 1/6, 1/2
    double inv, kmagic, l64_hi, l64_lo;  // 64/ln2; 1.5 * 2^52; -ln2/64 split
};
static __constant__ FastConsts c_fm = {-0.125, 1.0 / 7.0, -1.0 / 6.0,      0.2,        -0.25,          1.0 / 3.0,      -0.5,
                                       NHP_LN2_HI,      NHP_LN2_LO, 4503601774854144.0,
                                       1.0 / 120.0,     1.0 / 24.0, 1.0 / 6.0,      0.5,
                                       NHP_64_OVER_LN2, 6755399441055744.0, -NHP_LN2_64_HI, -NHP_LN2_64_LO};

// one copy per translation unit (1 KB), read once per CTA through L2
static __device__ unsigned long long g_nhp_logtab[64];
static __device__ unsigned long long g_nhp_exptab[64];
// host: copy the generated tables into this translation unit's device arrays (idempotent)
static inline cudaError_t fast_tables_upload(cudaStream_t s) {
    cudaError_t e = cudaMemcpyToSymbolAsync(g_nhp_logtab, NHP_LOGTAB_BITS, sizeof(NHP_LOGTAB_BITS), 0, cudaMemcpyHostToDevice, s);
    if (e != cudaSuccess) return e;
    return cudaMemcpyToSymbolAsync(g_nhp_exptab, NHP_EXPTAB_BITS, sizeof(NHP_EXPTAB_BITS), 0, cudaMemcpyHostToDevice, s);
}

// cooperative load of the tables into shared memory (1 KB); caller synchronises afterwards
__device__ __forceinline__ void fast_tables_load(FastTables *ft) {
    unsigned long long *dst = reinterpret_cast<unsigned long long *>(ft);
    for (int i = threadIdx.x; i < 64 + 64; i += blockDim.x) dst[i] = i < 64 ? g_nhp_logtab[i] : g_nhp_exptab[i - 64];
}

// rare-path fallbacks kept out of line so the hot loops stay small
static __device__ __noinline__ double slow_log(double x) { return log(x); }
static __device__ __noinline__ double slow_exp(double x) { return exp(x); }

// a positive, normal, finite double?  (one integer compare on the high word)
__device__ __forceinline__ bool is_pos_normal(double x) { return (unsigned)(__double2hiint(x) - 0x00100000) < 0x7fe00000u; }

// log of a positive normal finite double (unchecked: callers test is_pos_normal first)
__device__ __forceinline__ double fast_log_n(double x, const FastTables *ft) {
    const int hi = __double2hiint(x), lo = __double2loint(x);
    const int e = (hi >> 20) - 1023;
    const double m = __hiloint2double((hi & 0x000fffff) | 0x3ff00000, lo);
    const double2 t = ft->logtab[(hi >> 15) & 31];
    const double r = fma(m, t.x, -1.0);  // |r| <= 1/64: degree-8 log1p, truncation r^9/9 < 6e-18
    double q = fma(r, c_fm.l8, c_fm.l7);
    q = fma(r, q, c_fm.l6);
    q = fma(r, q, c_fm.l5);
    q = fma(r, q, c_fm.l4);
    q = fma(r, q, c_fm.l3);
    q = fma(r, q, c_fm.l2);
    const double p = fma(r * r, q, r);
    const double ed = __hiloint2double(0x43300000, e ^ 0x80000000) - c_fm.emagic;  // (double)e
    return fma(ed, c_fm.ln2_hi, t.y) + fma(ed, c_fm.ln2_lo, p);
}

// exp for x <= 709 (unchecked above; callers guarantee it); flushes to 0 below -707 (omitted mass < 1e-307)
__device__ __forceinline__ double fast_exp_c(double x, const FastTables *ft) {
    const double t = fma(x, c_fm.inv, c_fm.kmagic);
    const int k = __double2loint(t);
    const double kf = t - c_fm.kmagic;
    double r = fma(kf, c_fm.l64_hi, x);
    r = fma(kf, c_fm.l64_lo, r);
    const double T = ft->exptab[k & 63];
    double q = fma(r, c_fm.e5, c_fm.e4);
    q = fma(r, q, c_fm.e3);
    q = fma(r, q, c_fm.e2);
    const double p = fma(r * r, q, r);
    const double v = fma(T, p, T);
    // x < -707  <=>  sign set and magnitude >= 707  <=>  unsigned high word >= 0xC0861800
    const bool flush = (unsigned)__double2hiint(x) >= 0xC0861800u;
    return flush ? 0.0 : __hiloint2double(__double2hiint(v) + ((k >> 6) << 20), __double2loint(v));
}

// checked general-purpose wrappers (tests, non-critical paths)
__device__ __forceinline__ double fast_log(double x, const FastTables *ft) {
    if (!is_pos_normal(x)) return slow_log(x);
    return fast_log_n(x, ft);
}
__device__ __forceinline__ double fast_exp(double x, const FastTables *ft) {
    if (!(x >= -707.0)) return x < -707.0 ? 0.0 : x;  // NaN propagates
    if (x > 709.0) return slow_exp(x);
    return fast_exp_c(x, ft);
}

// digamma psi(x) for x > 0 (the VB expectations, baselines.jl:454-456, impulses.jl:373-375, weights.jl:95-97): the recurrence
// psi(x) = psi(x + 1) - 1/x up to x >= 10, then the asymptotic series log x - 1/(2x) - sum_k B_2k / (2k x^2k) with 7 terms (the
// first omitted term is below 5e-17 at x = 10).  Error 1.3e-15 * max(1, |psi|) against mpmath, measured on a B200 (libdevice log,
// IEEE division); the largest error is the cancellation near the root 1.4616...  NaN for x <= 0 or NaN.
__device__ inline double nhp_digamma(double x) {
    if (!(x > 0.0)) return __longlong_as_double(0x7ff8000000000000ll);
    double s = 0.0;
    while (x < 10.0) { s += 1.0 / x; x += 1.0; }
    const double r = 1.0 / x, z = r * r;
    double p = fma(z, 1.0 / 12.0, -691.0 / 32760.0);  // B_2k / 2k, k = 7 .. 1
    p = fma(z, p, 1.0 / 132.0);
    p = fma(z, p, -1.0 / 240.0);
    p = fma(z, p, 1.0 / 252.0);
    p = fma(z, p, -1.0 / 120.0);
    p = fma(z, p, 1.0 / 12.0);
    return (log(x) - 0.5 * r - z * p) - s;
}
