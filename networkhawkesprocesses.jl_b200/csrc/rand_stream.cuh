// rand_stream.cuh -- pieces shared by the device simulators (cont_rand.cu, disc_rand.cu): a Philox stream with the Poisson sampler,
// and the per-row running sums of a non-negative K x K rate matrix that the child-node draws invert.
#pragma once
#include "nhp_internal.cuh"

// Philox4x32-10 keyed (seed ^ tag; element, gen | draw, 0); every simulator has its own tag
#define NHP_RAND_TAG_CONT 0x52414E444841574Bull  // "RANDHAWK"
#define NHP_RAND_TAG_DISC 0x444953434841574Bull  // "DISCHAWK"

struct RandStream {
    uint32_t k0, k1, c0, c1, c2, c3, buf[4];
    int have;
    __device__ RandStream(uint64_t seed, uint64_t element, uint32_t gen, uint64_t tag = NHP_RAND_TAG_CONT) {
        const uint64_t key = seed ^ tag;
        k0 = (uint32_t)key; k1 = (uint32_t)(key >> 32);
        c0 = (uint32_t)element; c1 = (uint32_t)(element >> 32); c2 = gen; c3 = 0u;
        have = 0;
    }
    __device__ double uniform() {  // (0, 1)
        if (have == 0) { philox4x32_10(c0, c1, c2, c3, k0, k1, buf); c3++; have = 2; }
        have--;
        const uint64_t x = (((uint64_t)buf[2 * have] << 32) | (uint64_t)buf[2 * have + 1]) >> 11;
        return ((double)x + 0.5) * 1.1102230246251565e-16;
    }
    __device__ double normal() {
        const double u1 = uniform(), u2 = uniform();
        return sqrt(-2.0 * log(u1)) * cospi(2.0 * u2);
    }
    // Poisson(mean): sequential inversion for small means, Hoermann's PTRS transformed rejection (1993) otherwise
    __device__ long long poisson(double mean) {
        if (!(mean > 0.0)) return 0;
        if (mean < 10.0) {
            double p = exp(-mean), cum = p;
            const double u = uniform();
            long long k = 0;
            while (u > cum && k < 1000) { k++; p *= mean / (double)k; cum += p; }
            return k;
        }
        const double slam = sqrt(mean), loglam = log(mean);
        const double b = 0.931 + 2.53 * slam, a = -0.059 + 0.02483 * b, invalpha = 1.1239 + 1.1328 / (b - 3.4), vr = 0.9277 - 3.6224 / (b - 2.0);
        for (int it = 0; it < 10000; it++) {
            const double U = uniform() - 0.5, V = uniform();
            const double us = 0.5 - fabs(U);
            const double kf = floor((2.0 * a / us + b) * U + mean + 0.43);
            if (us >= 0.07 && V <= vr) return (long long)kf;
            if (kf < 0.0 || (us < 0.013 && V > us)) continue;
            if (log(V) + log(invalpha) - log(a / (us * us) + b) <= -mean + kf * loglam - lgamma(kf + 1.0)) return (long long)kf;
        }
        return (long long)mean;
    }
};

// per parent node p: the child nodes with A W[p,c] != 0 and the running sums of their weights (one warp per row)
static __global__ void k_rand_rows(int K, const double *__restrict__ W, const double *__restrict__ A, int *__restrict__ row_n, int *__restrict__ row_c,
                                   double *__restrict__ row_cum) {
    const int p = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    if (p >= K) return;
    int cnt = 0;
    double run = 0.0;
    for (int c0 = 0; c0 < K; c0 += 32) {
        const int c = c0 + lane;
        double w = 0.0;
        if (c < K) { w = W[p + (int64_t)K * c]; if (A) w *= A[p + (int64_t)K * c]; }
        const bool nz = w != 0.0;
        const unsigned m = __ballot_sync(0xffffffffu, nz);
        double x = w;  // inclusive scan of the weights across the lanes
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { const double y = __shfl_up_sync(0xffffffffu, x, d); if (lane >= d) x += y; }
        if (nz) {
            const int pos = cnt + __popc(m & ((1u << lane) - 1u));
            row_c[(int64_t)p * K + pos] = c;
            row_cum[(int64_t)p * K + pos] = run + x;
        }
        cnt += __popc(m);
        run += __shfl_sync(0xffffffffu, x, 31);
    }
    if (lane == 0) row_n[p] = cnt;
}
