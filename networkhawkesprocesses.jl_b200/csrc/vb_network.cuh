// vb_network.cuh -- pieces of the mean-field VB steps shared by the discrete (disc_vb.cu) and continuous (cont_vb.cu) paths: the
// relative change and blend of an entry of q, the link probability's sigmoid, the end-of-kernel reduction of the update kernels, and
// the fixed-order reduction of the link probabilities into q(rho) of a network state.
#pragma once
#include "nhp_internal.cuh"

__device__ __forceinline__ double rel_change(double nw, double old) { return fabs(nw - old) / old; }

__device__ __forceinline__ double blend(double old, double target, double step) { return (1.0 - step) * old + step * target; }

// 1 / (1 + exp(-x)) without overflow for either sign of x
__device__ __forceinline__ double stable_sigmoid(double x) {
    if (x >= 0.0) return 1.0 / (1.0 + exp(-x));
    const double z = exp(x);
    return z / (1.0 + z);
}

// the end of an update kernel of 256-thread blocks: the block's largest mx into *change (an integer atomicMax per warp: the bit order
// of non-negative doubles is their numeric order); NET: also the block's sum of pt into psum[blockIdx.x] (a fixed shuffle tree, then
// the warps in order), so the same inputs give the same bits
template <bool NET>
__device__ __forceinline__ void vb_block_reduce(double mx, double pt, unsigned long long *change, double *psum) {
    __shared__ double warp_sum[8];
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) {
        mx = fmax(mx, __shfl_xor_sync(0xffffffffu, mx, d));
        if constexpr (NET) pt += __shfl_xor_sync(0xffffffffu, pt, d);
    }
    if ((threadIdx.x & 31) == 0) {
        if (mx > 0.0) atomicMax(change, (unsigned long long)__double_as_longlong(mx));
        if constexpr (NET) warp_sum[threadIdx.x >> 5] = pt;
    }
    if constexpr (NET) {
        __syncthreads();
        if (threadIdx.x == 0) {
            double t = 0.0;
            for (int w = 0; w < (int)(blockDim.x >> 5); w++) t += warp_sum[w];
            psum[blockIdx.x] = t;
        }
    }
}

// one block of 256: S = sum of the nblocks partial sums in a fixed order, then alpharhov* = alpha_rho + S, betarhov* = beta_rho + N^2 - S
// (N^2 counts links, not data: never scaled), blended, their relative change folded into change.  Static: each translation unit that
// launches it holds its own copy.
static __global__ void __launch_bounds__(256) k_vbn_finish(double *__restrict__ rho, const double *__restrict__ psum, int nblocks, double alpha_rho,
                                                           double beta_rho, double links, double step, unsigned long long *__restrict__ change) {
    __shared__ double sh[256];
    double a = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += 256) a += psum[i];
    sh[threadIdx.x] = a;
    __syncthreads();
    for (int w = 128; w > 0; w >>= 1) {
        if ((int)threadIdx.x < w) sh[threadIdx.x] += sh[threadIdx.x + w];
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        const double S = sh[0];
        const double an = blend(rho[0], alpha_rho + S, step), bn = blend(rho[1], (beta_rho + links) - S, step);
        const double mx = fmax(rel_change(an, rho[0]), rel_change(bn, rho[1]));
        rho[0] = an;
        rho[1] = bn;
        if (mx > 0.0) atomicMax(change, (unsigned long long)__double_as_longlong(mx));
    }
}
