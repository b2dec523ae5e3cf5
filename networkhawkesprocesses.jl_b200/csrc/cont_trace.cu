// cont_trace.cu -- device-side sample traces of `mcmc!` (inference.jl:49-70; continuous.jl:325-333, discrete.jl:178-182 / 406-414).
//
// The reference pushes `params(process)` = [rho; lambda0; W; theta | mu, tau; vec(A)] as a fresh Vector{Float64} per sweep
// (32 MB per sweep at K = 1000, adjacency as Float64).  With the whole sweep on the device (nhp_cont_gibbs_sweep) the sample
// would be the only thing that still crosses PCIe every sweep; the trace keeps it on the device instead: one slot per stored
// sweep, the real-valued parameters as they are (device-to-device copies on the context's stream, no host synchronisation) and
// the adjacency matrix bit-packed (K^2 / 8 bytes instead of 8 K^2), read back in one piece when the chain is done.
#include "nhp_internal.cuh"
#include <algorithm>

__global__ void k_trace_pack_bits(const double *__restrict__ A, int64_t n, uint32_t *__restrict__ out) {
    const int64_t w = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (w * 32 >= n) return;
    const int64_t e = w * 32 + lane;
    const unsigned m = __ballot_sync(0xffffffffu, e < n && A[e] != 0.0);
    if (lane == 0) out[w] = m;
}
__global__ void k_trace_unpack_bits(const uint32_t *__restrict__ in, int64_t n, double *__restrict__ A) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < n) A[e] = (in[e >> 5] >> (e & 31)) & 1u ? 1.0 : 0.0;
}

static size_t trace_slot_doubles(const nhp_ctx *ctx) {  // rho, lambda0, W, p1 (, p2)
    const size_t K = (size_t)ctx->K;
    return 1 + K + K * K * (ctx->kind == NHP_LOGITNORMAL ? 3 : 2);
}
static size_t trace_slot_words(const nhp_ctx *ctx) { return ctx->has_A ? ((size_t)ctx->K * ctx->K + 31) / 32 : 0; }

extern "C" int nhp_cont_trace_free(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->d_trace); cudaFree(ctx->d_trace_bits); cudaFree(ctx->d_trace_curves);
    ctx->d_trace = nullptr; ctx->d_trace_bits = nullptr; ctx->d_trace_curves = nullptr; ctx->trace_cap = ctx->trace_len = 0; ctx->trace_G = 0;
    return NHP_OK;
}

extern "C" int nhp_cont_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "nhp_cont_trace_begin: continuous parameters not set (the slot layout follows the model)");
    NHP_CHECK(ctx, capacity >= 1, NHP_ERR_INVALID, "nhp_cont_trace_begin: capacity must be positive");
    NHP_TRY(nhp_cont_trace_free(ctx));
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t sd = trace_slot_doubles(ctx), sw = trace_slot_words(ctx);
    // curves with a prior move with the sweep (nhp_cont_gibbs_sweep): every slot also keeps them
    const int64_t G = ctx->bgrid_n > 0 && ctx->bprior_n == ctx->bgrid_n ? ctx->bgrid_n : 0;
    const size_t sc = (size_t)(ctx->K * G);
    if (cudaMalloc(&ctx->d_trace, (size_t)capacity * sd * sizeof(double)) != cudaSuccess ||
        (sw && cudaMalloc(&ctx->d_trace_bits, (size_t)capacity * sw * sizeof(uint32_t)) != cudaSuccess) ||
        (sc && cudaMalloc(&ctx->d_trace_curves, (size_t)capacity * sc * sizeof(double)) != cudaSuccess)) {
        cudaGetLastError();
        cudaFree(ctx->d_trace); cudaFree(ctx->d_trace_bits); ctx->d_trace = nullptr; ctx->d_trace_bits = nullptr;
        return nhp_fail(ctx, NHP_ERR_CUDA, "nhp_cont_trace_begin: cannot allocate %lld slots of %.1f MB", (long long)capacity, 1e-6 * (double)(sd * 8 + sw * 4 + sc * 8));
    }
    ctx->trace_G = G;
    ctx->trace_cap = capacity; ctx->trace_len = 0; ctx->trace_K = ctx->K; ctx->trace_kind = ctx->kind; ctx->trace_has_A = ctx->has_A;
    return NHP_OK;
}

// append the context's current parameters (after a sweep: the new sample); stream-ordered, no host synchronisation
extern "C" int nhp_cont_trace_push(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->trace_cap > 0, NHP_ERR_STATE, "nhp_cont_trace_push: no trace (call nhp_cont_trace_begin)");
    NHP_CHECK(ctx, ctx->cont_set && ctx->trace_K == ctx->K && ctx->trace_kind == ctx->kind && ctx->trace_has_A == ctx->has_A, NHP_ERR_STATE,
              "nhp_cont_trace_push: the model changed since nhp_cont_trace_begin");
    NHP_CHECK(ctx, ctx->trace_len < ctx->trace_cap, NHP_ERR_STATE, "nhp_cont_trace_push: the trace is full (%lld slots)", (long long)ctx->trace_cap);
    NHP_CHECK(ctx, ctx->trace_G == 0 || ctx->bgrid_n == ctx->trace_G, NHP_ERR_STATE, "nhp_cont_trace_push: the curves' grid changed since nhp_cont_trace_begin (%lld -> %lld points)",
              (long long)ctx->trace_G, (long long)ctx->bgrid_n);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t K = (size_t)ctx->K, KK = K * K, sd = trace_slot_doubles(ctx), sw = trace_slot_words(ctx);
    cudaStream_t s = ctx->stream;
    double *slot = ctx->d_trace + (size_t)ctx->trace_len * sd;
    const double rho = ctx->rho;
    NHP_CUDA(ctx, cudaMemcpyAsync(slot, &rho, sizeof(double), cudaMemcpyHostToDevice, s));  // 8 bytes from pageable memory: staged by the runtime before the call returns
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1, ctx->d_lambda0, K * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + K, ctx->d_W, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + K + KK, ctx->d_p1, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (ctx->kind == NHP_LOGITNORMAL) NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + K + 2 * KK, ctx->d_p2, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (ctx->trace_G > 0) {
        const size_t sc = K * (size_t)ctx->trace_G;
        NHP_CUDA(ctx, cudaMemcpyAsync(ctx->d_trace_curves + (size_t)ctx->trace_len * sc, ctx->d_bgrid_v, sc * sizeof(double), cudaMemcpyDeviceToDevice, s));
    }
    if (sw) {
        const int64_t warps = (int64_t)sw;
        k_trace_pack_bits<<<(unsigned)((warps + 7) / 8), 256, 0, s>>>(ctx->d_A, (int64_t)KK, ctx->d_trace_bits + (size_t)ctx->trace_len * sw);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
    }
    ctx->trace_len++;
    return NHP_OK;
}

extern "C" int nhp_cont_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    if (count) *count = ctx->trace_len;
    if (capacity) *capacity = ctx->trace_cap;
    return NHP_OK;
}

// samples [first, first + count) in the layouts of nhp_cont_params_get, one sample after the other: rho[count], lambda0[count*K],
// W / A / p1 / p2 [count*K*K]; any pointer may be NULL (A, p2 are ignored by models without them)
extern "C" int nhp_cont_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *rho, double *lambda0, double *W, double *A, double *p1, double *p2) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, first >= 0 && count >= 0 && first + count <= ctx->trace_len, NHP_ERR_INVALID, "nhp_cont_trace_read: samples [%lld, %lld) outside the %lld stored",
              (long long)first, (long long)(first + count), (long long)ctx->trace_len);
    if (count == 0) return NHP_OK;
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t K = (size_t)ctx->trace_K, KK = K * K;
    const size_t sd = 1 + K + KK * (ctx->trace_kind == NHP_LOGITNORMAL ? 3 : 2), sw = ctx->trace_has_A ? (KK + 31) / 32 : 0;
    cudaStream_t s = ctx->stream;
    const double *base = ctx->d_trace + (size_t)first * sd;
    const size_t pitch = sd * sizeof(double);
    if (rho) NHP_CUDA(ctx, cudaMemcpy2DAsync(rho, sizeof(double), base, pitch, sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (lambda0) NHP_CUDA(ctx, cudaMemcpy2DAsync(lambda0, K * sizeof(double), base + 1, pitch, K * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (W) NHP_CUDA(ctx, cudaMemcpy2DAsync(W, KK * sizeof(double), base + 1 + K, pitch, KK * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (p1) NHP_CUDA(ctx, cudaMemcpy2DAsync(p1, KK * sizeof(double), base + 1 + K + KK, pitch, KK * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (p2 && ctx->trace_kind == NHP_LOGITNORMAL)
        NHP_CUDA(ctx, cudaMemcpy2DAsync(p2, KK * sizeof(double), base + 1 + K + 2 * KK, pitch, KK * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (A && sw) {
        void *scratch = nullptr;
        NHP_TRY(nhp_scratch(ctx, KK * sizeof(double), &scratch));
        for (int64_t k = 0; k < count; k++) {  // expanded one sample at a time through the context's scratch buffer
            k_trace_unpack_bits<<<(unsigned)((KK + 255) / 256), 256, 0, s>>>(ctx->d_trace_bits + (size_t)(first + k) * sw, (int64_t)KK, (double *)scratch);
            NHP_LAUNCHED(ctx);
            NHP_CUDA(ctx, cudaMemcpyAsync(A + (size_t)k * KK, scratch, KK * sizeof(double), cudaMemcpyDeviceToHost, s));
        }
    }
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// the curves of samples [first, first + count): values[g + G (k + K j)] is curve point g of node k in sample first + j
extern "C" int nhp_cont_trace_read_curves(nhp_ctx *ctx, int64_t first, int64_t count, double *values) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->trace_G > 0, NHP_ERR_STATE, "nhp_cont_trace_read_curves: the trace holds no curves (begin it with curves and their prior set)");
    NHP_CHECK(ctx, first >= 0 && count >= 0 && first + count <= ctx->trace_len, NHP_ERR_INVALID, "nhp_cont_trace_read_curves: samples [%lld, %lld) outside the %lld stored",
              (long long)first, (long long)(first + count), (long long)ctx->trace_len);
    if (count == 0) return NHP_OK;
    NHP_CHECK(ctx, values != nullptr, NHP_ERR_INVALID, "nhp_cont_trace_read_curves: NULL argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t sc = (size_t)ctx->trace_K * (size_t)ctx->trace_G;
    NHP_CUDA(ctx, cudaMemcpyAsync(values, ctx->d_trace_curves + (size_t)first * sc, (size_t)count * sc * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// discrete trace (discrete.jl:178-182 / 406-414): the same scheme for the discrete model, with its own state on the context.
// One slot: rho, lambda0[N], W[N^2], theta[N^2 B] (+ the adjacency matrix bit-packed, N^2 / 8 bytes): 2.24 MB at N = 200, B = 6.
// ---------------------------------------------------------------------------------------
static size_t disc_slot_doubles(int64_t N, int64_t B) { return 1 + (size_t)N + (size_t)(N * N) * (size_t)(1 + B); }
static size_t disc_slot_words(int64_t N, bool has_A) { return has_A ? ((size_t)(N * N) + 31) / 32 : 0; }

extern "C" int nhp_disc_trace_free(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(ctx->dd_trace); cudaFree(ctx->dd_trace_bits);
    ctx->dd_trace = nullptr; ctx->dd_trace_bits = nullptr; ctx->dd_trace_cap = ctx->dd_trace_len = 0;
    return NHP_OK;
}

extern "C" int nhp_disc_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->disc_set, NHP_ERR_STATE, "nhp_disc_trace_begin: discrete parameters not set (the slot layout follows the model)");
    NHP_CHECK(ctx, capacity >= 1, NHP_ERR_INVALID, "nhp_disc_trace_begin: capacity must be positive");
    NHP_TRY(nhp_disc_trace_free(ctx));
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t sd = disc_slot_doubles(ctx->dN, ctx->dB), sw = disc_slot_words(ctx->dN, ctx->d_has_A);
    if (cudaMalloc(&ctx->dd_trace, (size_t)capacity * sd * sizeof(double)) != cudaSuccess ||
        (sw && cudaMalloc(&ctx->dd_trace_bits, (size_t)capacity * sw * sizeof(uint32_t)) != cudaSuccess)) {
        cudaGetLastError();
        cudaFree(ctx->dd_trace); ctx->dd_trace = nullptr;
        return nhp_fail(ctx, NHP_ERR_CUDA, "nhp_disc_trace_begin: cannot allocate %lld slots of %.2f MB", (long long)capacity, 1e-6 * (double)(sd * 8 + sw * 4));
    }
    ctx->dd_trace_cap = capacity; ctx->dd_trace_len = 0; ctx->dd_trace_N = ctx->dN; ctx->dd_trace_B = ctx->dB; ctx->dd_trace_has_A = ctx->d_has_A;
    return NHP_OK;
}

// append the context's current discrete parameters and rho; stream-ordered, no host synchronisation
extern "C" int nhp_disc_trace_push(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->dd_trace_cap > 0, NHP_ERR_STATE, "nhp_disc_trace_push: no trace (call nhp_disc_trace_begin)");
    NHP_CHECK(ctx, ctx->disc_set && ctx->dd_trace_N == ctx->dN && ctx->dd_trace_B == ctx->dB && ctx->dd_trace_has_A == ctx->d_has_A, NHP_ERR_STATE,
              "nhp_disc_trace_push: the model changed since nhp_disc_trace_begin");
    NHP_CHECK(ctx, ctx->dd_trace_len < ctx->dd_trace_cap, NHP_ERR_STATE, "nhp_disc_trace_push: the trace is full (%lld slots)", (long long)ctx->dd_trace_cap);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t N = (size_t)ctx->dN, NN = N * N, sd = disc_slot_doubles(ctx->dN, ctx->dB), sw = disc_slot_words(ctx->dN, ctx->d_has_A);
    cudaStream_t s = ctx->stream;
    double *slot = ctx->dd_trace + (size_t)ctx->dd_trace_len * sd;
    const double rho = ctx->dd_rho;
    NHP_CUDA(ctx, cudaMemcpyAsync(slot, &rho, sizeof(double), cudaMemcpyHostToDevice, s));  // 8 bytes from pageable memory: staged before the call returns
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1, ctx->dd_lambda0, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + N, ctx->dd_W, NN * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + N + NN, ctx->dd_theta, NN * (size_t)ctx->dB * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (sw) {
        k_trace_pack_bits<<<(unsigned)((sw + 7) / 8), 256, 0, s>>>(ctx->dd_A, (int64_t)NN, ctx->dd_trace_bits + (size_t)ctx->dd_trace_len * sw);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
    }
    ctx->dd_trace_len++;
    return NHP_OK;
}

extern "C" int nhp_disc_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    if (count) *count = ctx->dd_trace_len;
    if (capacity) *capacity = ctx->dd_trace_cap;
    return NHP_OK;
}

// samples [first, first + count) in the layouts of nhp_disc_params_get, one sample after the other: rho[count], lambda0[count*N],
// W / A [count*N*N], theta[count*N*N*B]; any pointer may be NULL (A is ignored for a model without it)
extern "C" int nhp_disc_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *rho, double *lambda0, double *W, double *A, double *theta) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, first >= 0 && count >= 0 && first + count <= ctx->dd_trace_len, NHP_ERR_INVALID, "nhp_disc_trace_read: samples [%lld, %lld) outside the %lld stored",
              (long long)first, (long long)(first + count), (long long)ctx->dd_trace_len);
    if (count == 0) return NHP_OK;
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t N = (size_t)ctx->dd_trace_N, NN = N * N, NNB = NN * (size_t)ctx->dd_trace_B;
    const size_t sd = disc_slot_doubles(ctx->dd_trace_N, ctx->dd_trace_B), sw = disc_slot_words(ctx->dd_trace_N, ctx->dd_trace_has_A);
    cudaStream_t s = ctx->stream;
    const double *base = ctx->dd_trace + (size_t)first * sd;
    const size_t pitch = sd * sizeof(double);
    if (rho) NHP_CUDA(ctx, cudaMemcpy2DAsync(rho, sizeof(double), base, pitch, sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (lambda0) NHP_CUDA(ctx, cudaMemcpy2DAsync(lambda0, N * sizeof(double), base + 1, pitch, N * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (W) NHP_CUDA(ctx, cudaMemcpy2DAsync(W, NN * sizeof(double), base + 1 + N, pitch, NN * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (theta) NHP_CUDA(ctx, cudaMemcpy2DAsync(theta, NNB * sizeof(double), base + 1 + N + NN, pitch, NNB * sizeof(double), (size_t)count, cudaMemcpyDeviceToHost, s));
    if (A && sw) {
        void *scratch = nullptr;
        NHP_TRY(nhp_scratch(ctx, NN * sizeof(double), &scratch));
        for (int64_t k = 0; k < count; k++) {  // expanded one sample at a time through the context's scratch buffer
            k_trace_unpack_bits<<<(unsigned)((NN + 255) / 256), 256, 0, s>>>(ctx->dd_trace_bits + (size_t)(first + k) * sw, (int64_t)NN, (double *)scratch);
            NHP_LAUNCHED(ctx);
            NHP_CUDA(ctx, cudaMemcpyAsync(A + (size_t)k * NN, scratch, NN * sizeof(double), cudaMemcpyDeviceToHost, s));
        }
    }
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}
