// microbench.cu -- in-library roofline denominators that MEASURED_PEAKS.json does not carry:
// the FP64 FMA peak and the register-resident pairs/s ceiling of each impulse function
// (SURVEY.md section 8d asks the builder to measure both and quote % roofline against them).
#include "nhp_internal.cuh"

// 8 independent DFMA chains per thread, no memory traffic
__global__ void __launch_bounds__(256) k_dfma_peak(double *out, int iters, double a, double b) {
    double x0 = threadIdx.x, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
        x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
        x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
    }
    double s = x0 + x1 + x2 + x3 + x4 + x5 + x6 + x7;
    if (s == 12345.678) out[0] = s;
}

// FP64 tensor-core rate: mma.sync.aligned.m8n8k4.f64 (DMMA), 4 independent accumulator tiles per warp
__global__ void __launch_bounds__(256) k_dmma_peak(double *out, int iters) {
    double a = 1.0 + threadIdx.x * 1e-3, b = 0.5 - threadIdx.x * 1e-3;
    double c0 = 0, c1 = 0, d0 = 0, d1 = 0, e0 = 0, e1 = 0, f0 = 0, f1 = 0;
    for (int i = 0; i < iters; i++) {
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(d0), "+d"(d1) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(e0), "+d"(e1) : "d"(a), "d"(b));
        asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(f0), "+d"(f1) : "d"(a), "d"(b));
    }
    double s = c0 + c1 + d0 + d1 + e0 + e1 + f0 + f1;
    if (s == 12345.678) out[0] = s;
}

// the device impulse function on register inputs (dt marches through the support)
template <typename E> __global__ void __launch_bounds__(256) k_pair_peak(double *out, int iters, E e, double D) {
    __shared__ FastTables s_ft;
    fast_tables_load(&s_ft);
    __syncthreads();
    const FastTables *ft = &s_ft;
    double dt0 = (threadIdx.x + 1) * (D / 300.0), acc = 0.0, step = D * 1e-7;
    double dt1 = dt0 * 0.5;
    for (int i = 0; i < iters; i++) {
        acc += pair_value(e, dt0, D, ft);
        acc += pair_value(e, dt1, D, ft);
        dt0 += step; dt1 += step;
    }
    if (acc == 12345.678) out[0] = acc;
}

// Adjacency-bit probe rate of the sparse sweep's filter with nothing around it: every thread owns a 1024-bit row in its own
// shared-memory bank (word w of lane l at [w * 32 + l], as in k_sweep_sparse) and walks a shared window of node ids eight
// probes per trip: one LDS for the node id, one LDS for the row word, shift / mask / merge -- the instruction sequence of
// cont_sparse.cu's phase 1.  probes/s of this loop is the ceiling the sweep's filter phase is compared with.
__global__ void __launch_bounds__(256) k_probe_peak(unsigned long long *out, int iters, unsigned seed) {
    __shared__ uint32_t rows[8 * 32 * 32];  // [warp][word][lane]
    __shared__ int sc[512 + 8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t x = seed ^ (threadIdx.x * 2654435761u) ^ (blockIdx.x * 40503u);
    for (int w = 0; w < 32; w++) { x = x * 1664525u + 1013904223u; rows[(warp * 32 + w) * 32 + lane] = x & (x >> 3) & (x >> 7) & (x >> 11); }  // ~6 % of the bits set
    for (int i = threadIdx.x; i < 520; i += 256) { x = x * 1664525u + 1013904223u; sc[i] = (int)((x >> 8) & 1023u); }
    __syncthreads();
    const uint32_t *myrow = rows + warp * 32 * 32 + lane;
    unsigned long long acc = 0ull;
    int pos = 64 + (threadIdx.x & 63);
    for (int it = 0; it < iters; it++) {
        unsigned long long hits = 0ull;
        const int *src = sc + pos;
#pragma unroll 1
        for (int m = 0; m < 64; m += 8) {
            const int p0 = src[-m], p1 = src[-m - 1], p2 = src[-m - 2], p3 = src[-m - 3];
            const int p4 = src[-m - 4], p5 = src[-m - 5], p6 = src[-m - 6], p7 = src[-m - 7];
            const uint32_t w0 = myrow[p0 & ~31], w1 = myrow[p1 & ~31], w2 = myrow[p2 & ~31], w3 = myrow[p3 & ~31];
            const uint32_t w4 = myrow[p4 & ~31], w5 = myrow[p5 & ~31], w6 = myrow[p6 & ~31], w7 = myrow[p7 & ~31];
            const uint32_t b8 = ((w0 >> (p0 & 31)) & 1u) | (((w1 >> (p1 & 31)) & 1u) << 1) | (((w2 >> (p2 & 31)) & 1u) << 2) |
                                (((w3 >> (p3 & 31)) & 1u) << 3) | (((w4 >> (p4 & 31)) & 1u) << 4) | (((w5 >> (p5 & 31)) & 1u) << 5) |
                                (((w6 >> (p6 & 31)) & 1u) << 6) | (((w7 >> (p7 & 31)) & 1u) << 7);
            hits |= (unsigned long long)b8 << m;
        }
        acc += __popcll(hits);
        pos = 64 + ((pos + 37 + (int)(hits & 7ull)) & 255);
    }
    if (acc == 0x7fffffffffffull) out[0] = acc;
}

// which: 0 = DFMA TFLOP/s (2 flops per FMA), 1 = LogitNormal pairs/s, 2 = Exponential pairs/s, 3 = DMMA m8n8k4 TFLOP/s
extern "C" int nhp_bench_fp64(nhp_ctx *ctx, int which, double *result) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, result != nullptr && which >= 0 && which <= 4, NHP_ERR_INVALID, "nhp_bench_fp64: bad argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, 64, &scratch));
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    const int blocks = ctx->sm_count * 8, iters = which == 0 ? 20000 : 2000;
    double best = 1e30;
    for (int rep = 0; rep < 4; rep++) {
        NHP_TRY(nhp_timer_begin(ctx));
        if (which == 0) k_dfma_peak<<<blocks, 256, 0, ctx->stream>>>((double *)scratch, iters, 0.999999, 1e-9);
        else if (which == 3) k_dmma_peak<<<blocks, 256, 0, ctx->stream>>>((double *)scratch, iters);
        else if (which == 4) k_probe_peak<<<blocks, 256, 0, ctx->stream>>>((unsigned long long *)scratch, iters, 12345u);
        else if (which == 1) { EntryLN e{0.3, 0.1, 0.6, 0.0}; k_pair_peak<EntryLN><<<blocks, 256, 0, ctx->stream>>>((double *)scratch, iters, e, 1.0); }
        else { EntryEX e{0.3, 1.1}; k_pair_peak<EntryEX><<<blocks, 256, 0, ctx->stream>>>((double *)scratch, iters, e, 1.0); }
        NHP_LAUNCHED(ctx);
        NHP_TRY(nhp_timer_end(ctx));
        if (rep > 0 && ctx->last_ms < best) best = ctx->last_ms;
    }
    double work = (double)blocks * 256.0 * iters * (which == 0 ? 16.0 : 2.0);
    if (which == 3) work = (double)blocks * 8.0 * iters * 4.0 * 512.0;  // 8 warps x 4 DMMA x (8*8*4*2 flops)
    if (which == 4) work = (double)blocks * 256.0 * iters * 64.0;       // 64 probes per thread and iteration
    *result = work / (best * 1e-3) / ((which == 0 || which == 3) ? 1e12 : 1.0);
    return NHP_OK;
}

// test hook: out[i] = fast_log(x[i]) (which = 0), fast_exp(x[i]) (which = 1) or nhp_digamma(x[i]) (which = 2); HOST pointers
__global__ void k_fastmath_eval(const double *x, double *out, int64_t n, int which) {
    __shared__ FastTables s_ft;
    fast_tables_load(&s_ft);
    __syncthreads();
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) out[i] = which == 0 ? fast_log(x[i], &s_ft) : which == 1 ? fast_exp(x[i], &s_ft) : nhp_digamma(x[i]);
}
extern "C" int nhp_test_fastmath(nhp_ctx *ctx, int which, const double *x, int64_t n, double *out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, x && out && n > 0 && which >= 0 && which <= 2, NHP_ERR_INVALID, "nhp_test_fastmath: bad argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)n * 16, &scratch));
    double *dx = (double *)scratch, *dout = dx + n;
    NHP_CUDA(ctx, cudaMemcpyAsync(dx, x, (size_t)n * 8, cudaMemcpyHostToDevice, ctx->stream));
    k_fastmath_eval<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dx, dout, n, which);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaMemcpyAsync(out, dout, (size_t)n * 8, cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}
