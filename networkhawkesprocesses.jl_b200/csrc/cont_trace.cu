// cont_trace.cu -- device-side traces (DeviceTrace, nhp_internal.cuh) and the sample traces of `mcmc!` (inference.jl:49-70;
// continuous.jl:325-333, discrete.jl:178-182 / 406-414).
//
// The reference pushes `params(process)` = [rho; lambda0; W; theta | mu, tau; vec(A)] as a fresh Vector{Float64} per sweep
// (32 MB per sweep at K = 1000, adjacency as Float64).  With the whole sweep on the device (nhp_cont_gibbs_sweep) the sample
// would be the only thing that still crosses PCIe every sweep; the trace keeps it on the device instead: one slot per stored
// sweep, the real-valued parameters as they are (device-to-device copies on the context's stream, no host synchronisation) and
// the adjacency matrix bit-packed (K^2 / 8 bytes instead of 8 K^2), read back in one piece when the chain is done.  The VB steps
// keep their states in the same kind of trace (vb_state.cu).
#include "nhp_internal.cuh"

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

void nhp_trace_free(nhp_ctx *ctx, DeviceTrace &tr) {
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    cudaFree(tr.d); cudaFree(tr.bits); cudaFree(tr.curves);
    tr = DeviceTrace();
}

int nhp_trace_begin(nhp_ctx *ctx, DeviceTrace &tr, const char *fn, int64_t capacity, size_t doubles, size_t words, size_t curve_doubles,
                    TraceShape shape) {
    NHP_CHECK(ctx, capacity >= 1, NHP_ERR_INVALID, "%s: capacity must be positive", fn);
    nhp_trace_free(ctx, tr);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t c = (size_t)capacity;
    if (cudaMalloc(&tr.d, c * doubles * sizeof(double)) != cudaSuccess ||
        (words && cudaMalloc(&tr.bits, c * words * sizeof(uint32_t)) != cudaSuccess) ||
        (curve_doubles && cudaMalloc(&tr.curves, c * curve_doubles * sizeof(double)) != cudaSuccess)) {
        cudaGetLastError();
        nhp_trace_free(ctx, tr);
        return nhp_fail(ctx, NHP_ERR_CUDA, "%s: cannot allocate %lld slots of %.2f MB", fn, (long long)capacity,
                        1e-6 * (double)(doubles * 8 + words * 4 + curve_doubles * 8));
    }
    tr.doubles = doubles; tr.words = words; tr.curve_doubles = curve_doubles;
    tr.cap = capacity; tr.len = 0; tr.shape = shape;
    return NHP_OK;
}

int nhp_trace_count(const DeviceTrace &tr, int64_t *count, int64_t *capacity) {
    if (count) *count = tr.len;
    if (capacity) *capacity = tr.cap;
    return NHP_OK;
}

int nhp_trace_check_range(nhp_ctx *ctx, const DeviceTrace &tr, const char *fn, int64_t first, int64_t count) {
    NHP_CHECK(ctx, first >= 0 && count >= 0 && first + count <= tr.len, NHP_ERR_INVALID, "%s: slots [%lld, %lld) outside the %lld stored", fn,
              (long long)first, (long long)(first + count), (long long)tr.len);
    return NHP_OK;
}

int nhp_trace_read_field(nhp_ctx *ctx, const DeviceTrace &tr, int64_t first, int64_t count, size_t off, size_t n, double *out) {
    if (!out) return NHP_OK;
    const double *src = tr.d + (size_t)first * tr.doubles + off;
    if (n == tr.doubles)  // whole slots: one contiguous copy
        NHP_CUDA(ctx, cudaMemcpyAsync(out, src, (size_t)count * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    else
        NHP_CUDA(ctx, cudaMemcpy2DAsync(out, n * sizeof(double), src, tr.doubles * sizeof(double), n * sizeof(double), (size_t)count,
                                        cudaMemcpyDeviceToHost, ctx->stream));
    return NHP_OK;
}

// the adjacency matrix A[n] into the bits of the next slot
static int trace_pack_bits(nhp_ctx *ctx, DeviceTrace &tr, const double *A, int64_t n) {
    k_trace_pack_bits<<<(unsigned)((tr.words + 7) / 8), 256, 0, ctx->stream>>>(A, n, tr.bits + (size_t)tr.len * tr.words);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaGetLastError());
    return NHP_OK;
}

// the adjacency matrices of slots [first, first + count), n entries each, expanded one sample at a time through the context's scratch buffer
static int trace_unpack_bits(nhp_ctx *ctx, const DeviceTrace &tr, int64_t first, int64_t count, int64_t n, double *A) {
    void *scratch = nullptr;
    NHP_TRY(nhp_scratch(ctx, (size_t)n * sizeof(double), &scratch));
    for (int64_t k = 0; k < count; k++) {
        k_trace_unpack_bits<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(tr.bits + (size_t)(first + k) * tr.words, n, (double *)scratch);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaMemcpyAsync(A + (size_t)k * n, scratch, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    }
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// continuous trace: one slot is rho, lambda0[K], W[K^2], p1[K^2] (, p2[K^2]), the adjacency matrix bit-packed, and with curves and
// their prior set at begin, the curves [K][G] (they move with the sweep)
// ---------------------------------------------------------------------------------------
extern "C" int nhp_cont_trace_free(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    nhp_trace_free(ctx, ctx->cont_trace);
    return NHP_OK;
}

extern "C" int nhp_cont_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->cont_set, NHP_ERR_STATE, "nhp_cont_trace_begin: continuous parameters not set (the slot layout follows the model)");
    const size_t K = (size_t)ctx->K, KK = K * K;
    const int64_t G = ctx->bgrid_n > 0 && ctx->bprior_n == ctx->bgrid_n ? ctx->bgrid_n : 0;
    return nhp_trace_begin(ctx, ctx->cont_trace, "nhp_cont_trace_begin", capacity, 1 + K + KK * (ctx->kind == NHP_LOGITNORMAL ? 3 : 2),
                           ctx->has_A ? (KK + 31) / 32 : 0, K * (size_t)G, TraceShape{ctx->K, ctx->kind, ctx->has_A, G});
}

// append the context's current parameters (after a sweep: the new sample); stream-ordered, no host synchronisation
extern "C" int nhp_cont_trace_push(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    DeviceTrace &tr = ctx->cont_trace;
    NHP_CHECK(ctx, tr.cap > 0, NHP_ERR_STATE, "nhp_cont_trace_push: no trace (call nhp_cont_trace_begin)");
    NHP_CHECK(ctx, ctx->cont_set && (tr.shape == TraceShape{ctx->K, ctx->kind, ctx->has_A, tr.shape.g}), NHP_ERR_STATE,
              "nhp_cont_trace_push: the model changed since nhp_cont_trace_begin");
    NHP_CHECK(ctx, tr.len < tr.cap, NHP_ERR_STATE, "nhp_cont_trace_push: the trace is full (%lld slots)", (long long)tr.cap);
    NHP_CHECK(ctx, tr.shape.g == 0 || ctx->bgrid_n == tr.shape.g, NHP_ERR_STATE, "nhp_cont_trace_push: the curves' grid changed since nhp_cont_trace_begin (%lld -> %lld points)",
              (long long)tr.shape.g, (long long)ctx->bgrid_n);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t K = (size_t)ctx->K, KK = K * K;
    cudaStream_t s = ctx->stream;
    double *slot = tr.next();
    const double rho = ctx->rho;
    NHP_CUDA(ctx, cudaMemcpyAsync(slot, &rho, sizeof(double), cudaMemcpyHostToDevice, s));  // 8 bytes from pageable memory: staged by the runtime before the call returns
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1, ctx->d_lambda0, K * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + K, ctx->d_W, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + K + KK, ctx->d_p1, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (ctx->kind == NHP_LOGITNORMAL) NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + K + 2 * KK, ctx->d_p2, KK * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (tr.curve_doubles)
        NHP_CUDA(ctx, cudaMemcpyAsync(tr.curves + (size_t)tr.len * tr.curve_doubles, ctx->d_bgrid_v, tr.curve_doubles * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (tr.words) NHP_TRY(trace_pack_bits(ctx, tr, ctx->d_A, (int64_t)KK));
    tr.len++;
    return NHP_OK;
}

extern "C" int nhp_cont_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    return nhp_trace_count(ctx->cont_trace, count, capacity);
}

// samples [first, first + count) in the layouts of nhp_cont_params_get, one sample after the other: rho[count], lambda0[count*K],
// W / A / p1 / p2 [count*K*K]; any pointer may be NULL (A, p2 are ignored by models without them)
extern "C" int nhp_cont_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *rho, double *lambda0, double *W, double *A, double *p1, double *p2) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    const DeviceTrace &tr = ctx->cont_trace;
    NHP_TRY(nhp_trace_check_range(ctx, tr, "nhp_cont_trace_read", first, count));
    if (count == 0) return NHP_OK;
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t K = (size_t)tr.shape.n, KK = K * K;
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 0, 1, rho));
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1, K, lambda0));
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1 + K, KK, W));
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1 + K + KK, KK, p1));
    if (tr.shape.b == NHP_LOGITNORMAL) NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1 + K + 2 * KK, KK, p2));
    if (A && tr.words) NHP_TRY(trace_unpack_bits(ctx, tr, first, count, (int64_t)KK, A));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

// the curves of samples [first, first + count): values[g + G (k + K j)] is curve point g of node k in sample first + j
extern "C" int nhp_cont_trace_read_curves(nhp_ctx *ctx, int64_t first, int64_t count, double *values) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    const DeviceTrace &tr = ctx->cont_trace;
    NHP_CHECK(ctx, tr.curve_doubles > 0, NHP_ERR_STATE, "nhp_cont_trace_read_curves: the trace holds no curves (begin it with curves and their prior set)");
    NHP_TRY(nhp_trace_check_range(ctx, tr, "nhp_cont_trace_read_curves", first, count));
    if (count == 0) return NHP_OK;
    NHP_CHECK(ctx, values != nullptr, NHP_ERR_INVALID, "nhp_cont_trace_read_curves: NULL argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t sc = tr.curve_doubles;
    NHP_CUDA(ctx, cudaMemcpyAsync(values, tr.curves + (size_t)first * sc, (size_t)count * sc * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// discrete trace (discrete.jl:178-182 / 406-414): the same scheme for the discrete model, with its own trace on the context.
// One slot: rho, lambda0[N], W[N^2], theta[N^2 B] (+ the adjacency matrix bit-packed, N^2 / 8 bytes): 2.24 MB at N = 200, B = 6.
// ---------------------------------------------------------------------------------------
extern "C" int nhp_disc_trace_free(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    nhp_trace_free(ctx, ctx->disc_trace);
    return NHP_OK;
}

extern "C" int nhp_disc_trace_begin(nhp_ctx *ctx, int64_t capacity) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->disc_set, NHP_ERR_STATE, "nhp_disc_trace_begin: discrete parameters not set (the slot layout follows the model)");
    const size_t N = (size_t)ctx->dN, NN = N * N;
    return nhp_trace_begin(ctx, ctx->disc_trace, "nhp_disc_trace_begin", capacity, 1 + N + NN * (size_t)(1 + ctx->dB), ctx->d_has_A ? (NN + 31) / 32 : 0,
                           0, TraceShape{ctx->dN, ctx->dB, ctx->d_has_A, 0});
}

// append the context's current discrete parameters and rho; stream-ordered, no host synchronisation
extern "C" int nhp_disc_trace_push(nhp_ctx *ctx) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    DeviceTrace &tr = ctx->disc_trace;
    NHP_CHECK(ctx, tr.cap > 0, NHP_ERR_STATE, "nhp_disc_trace_push: no trace (call nhp_disc_trace_begin)");
    NHP_CHECK(ctx, ctx->disc_set && (tr.shape == TraceShape{ctx->dN, ctx->dB, ctx->d_has_A, 0}), NHP_ERR_STATE,
              "nhp_disc_trace_push: the model changed since nhp_disc_trace_begin");
    NHP_CHECK(ctx, tr.len < tr.cap, NHP_ERR_STATE, "nhp_disc_trace_push: the trace is full (%lld slots)", (long long)tr.cap);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t N = (size_t)ctx->dN, NN = N * N;
    cudaStream_t s = ctx->stream;
    double *slot = tr.next();
    const double rho = ctx->dd_rho;
    NHP_CUDA(ctx, cudaMemcpyAsync(slot, &rho, sizeof(double), cudaMemcpyHostToDevice, s));  // 8 bytes from pageable memory: staged before the call returns
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1, ctx->dd_lambda0, N * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + N, ctx->dd_W, NN * sizeof(double), cudaMemcpyDeviceToDevice, s));
    NHP_CUDA(ctx, cudaMemcpyAsync(slot + 1 + N + NN, ctx->dd_theta, NN * (size_t)ctx->dB * sizeof(double), cudaMemcpyDeviceToDevice, s));
    if (tr.words) NHP_TRY(trace_pack_bits(ctx, tr, ctx->dd_A, (int64_t)NN));
    tr.len++;
    return NHP_OK;
}

extern "C" int nhp_disc_trace_count(const nhp_ctx *ctx, int64_t *count, int64_t *capacity) {
    if (!ctx) return NHP_ERR_INVALID;
    return nhp_trace_count(ctx->disc_trace, count, capacity);
}

// samples [first, first + count) in the layouts of nhp_disc_params_get, one sample after the other: rho[count], lambda0[count*N],
// W / A [count*N*N], theta[count*N*N*B]; any pointer may be NULL (A is ignored for a model without it)
extern "C" int nhp_disc_trace_read(nhp_ctx *ctx, int64_t first, int64_t count, double *rho, double *lambda0, double *W, double *A, double *theta) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    const DeviceTrace &tr = ctx->disc_trace;
    NHP_TRY(nhp_trace_check_range(ctx, tr, "nhp_disc_trace_read", first, count));
    if (count == 0) return NHP_OK;
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const size_t N = (size_t)tr.shape.n, NN = N * N;
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 0, 1, rho));
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1, N, lambda0));
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1 + N, NN, W));
    NHP_TRY(nhp_trace_read_field(ctx, tr, first, count, 1 + N + NN, NN * (size_t)tr.shape.b, theta));
    if (A && tr.words) NHP_TRY(trace_unpack_bits(ctx, tr, first, count, (int64_t)NN, A));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}
