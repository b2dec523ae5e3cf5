// disc_rand.cu -- rand(process::DiscreteHawkesProcess, T) (discrete.jl:20-38) on the device.
//
// The sample has the law nhp_disc_loglik evaluates: given every bin before t, the counts data[c, t] are independent
// Poisson(lambda[t, c]), lambda[t, c] = lambda0_c dt + sum_{p, b, l = 1..L} data[p, t - l] phi_b[l] [A]W[p, c] theta[p, c, b] dt
// (nhp_disc_intensity, phi from nhp_disc_basis), with no events before bin 0.  It is simulated in its cluster representation,
// generation by generation as in cont_rand.cu:
//   generation 0    n_c ~ Poisson(lambda0_c dt T) per node, bins uniform on 0..T-1: i.i.d. Poisson(lambda0_c dt) bin counts;
//   generation g+1  every event (t, p) of generation g draws its total number of children m ~ Poisson(s_p), s_p = sum_c e[p, c] with
//                   e[p, c] = [A]W[p, c] sum_b theta[p, c, b] sum_l phi_b[l] dt, then every child its node from Categorical(e[p, :] / s_p)
//                   and its lag l in 1..L from q_l ~ sum_b theta[p, c, b] phi_b[l]; children at t + l >= T are dropped and do not
//                   reproduce.
// By Poisson splitting the event (t, p) adds independent Poisson(sum_b phi_b[l] [A]W[p, c] theta[p, c, b] dt) counts to the cells
// (c, t + l): the conditional law above.  e is computed from the parameters as written: neither sum_b theta = 1 nor sum_l phi dt = 1
// is assumed.  The lag probabilities are formed on the fly from phi in shared memory (no N^2 L table).  Counts accumulate in the
// handle's int32 grid with integer atomics, which is order independent, so the sample is a deterministic function of (parameters,
// T, L, seed).  Random numbers: Philox4x32-10 keyed (seed ^ "DISCHAWK"; element, generation | draw, 0) (rand_stream.cuh).
#include "rand_stream.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <vector>

// e[p + N c] = [A]W[p, c] sum_b theta[p, c, b] sb[b]  (sb[b] = sum_l phi_b[l] dt); flag bit 0: a negative or non-finite [A]W, theta or
// lambda0
__global__ void k_drand_rates(int N, int B, const double *__restrict__ lambda0, const double *__restrict__ W, const double *__restrict__ A,
                              const double *__restrict__ theta, const double *__restrict__ sb, double *__restrict__ e, int *flag) {
    const int64_t NN = (int64_t)N * N;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= NN) return;
    bool bad = false;
    if (i < N) bad = !(lambda0[i] >= 0.0 && lambda0[i] < INFINITY);
    const double w = A ? A[i] * W[i] : W[i];
    bad |= !(w >= 0.0 && w < INFINITY);
    double acc = 0.0;
    for (int b = 0; b < B; b++) {
        const double th = theta[i + NN * b];
        bad |= !(th >= 0.0 && th < INFINITY);
        acc += th * sb[b];
    }
    if (bad) atomicOr(flag, 1);
    e[i] = w != 0.0 ? w * acc : 0.0;
}
__global__ void k_drand_base_counts(int N, const double *__restrict__ lambda0, double dtT, uint64_t seed, long long *__restrict__ counts) {
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= N) return;
    RandStream r(seed, (uint64_t)k, 0x80000000u, NHP_RAND_TAG_DISC);
    counts[k] = r.poisson(lambda0[k] * dtT);
}
// first event index of every node -> (bin, node) of generation 0, counted into the grid
__global__ void k_drand_base_emit(int N, const long long *__restrict__ off, int64_t T, uint64_t seed, int *__restrict__ ev_t, int *__restrict__ ev_c, long long n0,
                                  int *__restrict__ data) {
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= n0) return;
    int lo = 0, hi = N;  // node k with off[k] <= e < off[k+1]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (off[mid] <= e) lo = mid; else hi = mid; }
    RandStream r(seed, (uint64_t)e, 0u, NHP_RAND_TAG_DISC);
    const int64_t t = min((int64_t)(r.uniform() * (double)T), T - 1);
    ev_t[e] = (int)t;
    ev_c[e] = lo;
    atomicAdd(data + t * N + lo, 1);
}
// number of children of every event of the current generation: Poisson(s_p), s_p the last running sum of row p
__global__ void k_drand_child_counts(const int *__restrict__ ev_c, long long g0, long long ng, int N, const int *__restrict__ row_n, const double *__restrict__ row_cum,
                                     uint64_t seed, uint32_t gen, long long *__restrict__ counts) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= ng) return;
    const int p = ev_c[g0 + i];
    long long m = 0;
    if (p >= 0 && row_n[p] > 0) {
        RandStream r(seed, (uint64_t)(g0 + i), gen * 2u + 1u, NHP_RAND_TAG_DISC);
        m = r.poisson(row_cum[(int64_t)p * N + row_n[p] - 1]);
    }
    counts[i] = m;
}
// every child: its parent by the offsets, its node by inversion on the parent's running sums, its lag by inversion on
// q_l = sum_b theta[p, c, b] phi_b[l] (phi and s[b] = sum_l phi_b[l] in shared memory); children past the last bin get node -1
__global__ void k_drand_child_emit(int *__restrict__ ev_t, int *__restrict__ ev_c, long long g0, long long ng, const long long *__restrict__ off, long long total,
                                   long long out0, int N, int B, int L, int64_t T, const int *__restrict__ row_n, const int *__restrict__ row_c,
                                   const double *__restrict__ row_cum, const double *__restrict__ theta, const double *__restrict__ phi_s, uint64_t seed,
                                   uint32_t gen, int *__restrict__ data) {
    extern __shared__ double s_phi[];  // [L * B] phi[l + L b] | [B] sum_l phi[l + L b]
    for (int i = threadIdx.x; i < L * B + B; i += blockDim.x) s_phi[i] = phi_s[i];
    __syncthreads();
    const double *s_sum = s_phi + L * B;
    const long long s = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= total) return;
    long long lo = 0, hi = ng;  // parent i with off[i] <= s < off[i+1]
    while (hi - lo > 1) { const long long mid = (lo + hi) >> 1; if (off[mid] <= s) lo = mid; else hi = mid; }
    const int tp = ev_t[g0 + lo];
    const int p = ev_c[g0 + lo];
    RandStream r(seed, (uint64_t)(out0 + s), gen * 2u + 2u, NHP_RAND_TAG_DISC);
    // child node: Categorical(e[p, :] / s_p)
    const int nr = row_n[p];
    const double *cum = row_cum + (int64_t)p * N;
    const double target = r.uniform() * cum[nr - 1];
    int a = 0, b = nr - 1;
    while (a < b) { const int mid = (a + b) >> 1; if (cum[mid] > target) b = mid; else a = mid + 1; }
    const int c = row_c[(int64_t)p * N + a];
    // lag: Categorical(q / sum q), the entries of (p, c) at stride N^2
    const int64_t NN = (int64_t)N * N;
    const double *th = theta + p + (int64_t)N * c;
    double Q = 0.0;
    for (int k = 0; k < B; k++) Q += __ldg(th + NN * k) * s_sum[k];
    const double lt = r.uniform() * Q;
    double run = 0.0;
    int lag = -1, last = 0;
    for (int l = 0; l < L; l++) {
        double q = 0.0;
        for (int k = 0; k < B; k++) q += __ldg(th + NN * k) * s_phi[l + L * k];
        if (q > 0.0) last = l;
        run += q;
        if (run > lt) { lag = l; break; }
    }
    if (lag < 0) lag = last;  // rounding left the running sum at or below the target: the last lag with a positive q
    const int64_t tc = (int64_t)tp + lag + 1;
    if (tc < T) {
        ev_t[out0 + s] = (int)tc;
        ev_c[out0 + s] = c;
        atomicAdd(data + tc * N + c, 1);
    } else {
        ev_c[out0 + s] = -1;  // dropped: no count, no children
    }
}

#define R_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fin(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__)); } while (0)

extern "C" int nhp_disc_rand(nhp_ctx *ctx, int64_t T, int64_t L, uint64_t seed, int64_t max_events, nhp_disc **out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, out != nullptr, NHP_ERR_INVALID, "nhp_disc_rand: out is NULL");
    *out = nullptr;
    NHP_CHECK(ctx, ctx->disc_set, NHP_ERR_STATE, "nhp_disc_rand: discrete parameters not set (call nhp_disc_params_set)");
    const int64_t N = ctx->dN, B = ctx->dB, NN = N * N;
    NHP_CHECK(ctx, T >= 1 && T < (int64_t)2147483000 && N * T < (int64_t)2147483000, NHP_ERR_INVALID,
              "nhp_disc_rand: T = %lld must be >= 1 with N*T below 2^31 (N = %lld)", (long long)T, (long long)N);
    NHP_CHECK(ctx, L >= 1 && L <= 4096 && L * B <= 4096, NHP_ERR_INVALID, "nhp_disc_rand: nlags L = %lld must be >= 1 with L*B <= 4096 (B = %lld)", (long long)L, (long long)B);
    NHP_CHECK(ctx, max_events >= 1 && max_events < (int64_t)2147483000, NHP_ERR_INVALID, "nhp_disc_rand: max_events outside [1, 2^31)");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    // phi[l + L b] (impulses.jl:321-335), then s[b] = sum_l phi_b[l] and s[b] dt
    std::vector<double> ph((size_t)(L * B + 2 * B), 0.0);
    NHP_CHECK(ctx, nhp_disc_basis(L, B, ctx->ddt, ph.data()) == NHP_OK, NHP_ERR_INVALID, "nhp_disc_rand: bad basis dimensions");
    for (int64_t b = 0; b < B; b++) {
        double sum = 0.0;
        for (int64_t l = 0; l < L; l++) sum += ph[l + L * b];
        ph[L * B + b] = sum;
        ph[L * B + B + b] = sum * ctx->ddt;
    }
    const int64_t cap = max_events;
    cudaStream_t s = ctx->stream;
    double *d_phi = nullptr, *d_e = nullptr, *row_cum = nullptr;
    int *row_n = nullptr, *row_c = nullptr, *d_data = nullptr, *ev_t = nullptr, *ev_c = nullptr;
    long long *d_cnt = nullptr, *d_off = nullptr;
    void *d_tmp = nullptr;
    auto fin = [&](int rc) {
        cudaStreamSynchronize(s);
        cudaFree(d_phi); cudaFree(d_e); cudaFree(row_cum); cudaFree(row_n); cudaFree(row_c); cudaFree(d_data); cudaFree(ev_t); cudaFree(ev_c);
        cudaFree(d_cnt); cudaFree(d_off); cudaFree(d_tmp);
        return rc;
    };
    R_CUDA(cudaMalloc(&d_phi, ph.size() * sizeof(double)));
    R_CUDA(cudaMemcpyAsync(d_phi, ph.data(), ph.size() * sizeof(double), cudaMemcpyHostToDevice, s));
    R_CUDA(cudaMalloc(&d_e, (size_t)NN * sizeof(double)));
    R_CUDA(cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
    k_drand_rates<<<(unsigned)((NN + 255) / 256), 256, 0, s>>>((int)N, (int)B, ctx->dd_lambda0, ctx->dd_W, ctx->d_has_A ? ctx->dd_A : nullptr, ctx->dd_theta,
                                                              d_phi + L * B + B, d_e, ctx->d_flag);
    NHP_LAUNCHED(ctx);
    int flag = 0;
    R_CUDA(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    R_CUDA(cudaStreamSynchronize(s));
    if (flag) return fin(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_disc_rand: lambda0, [A]W and theta must be finite and non-negative"));
    R_CUDA(cudaMalloc(&row_n, (size_t)N * sizeof(int)));
    R_CUDA(cudaMalloc(&row_c, (size_t)NN * sizeof(int)));
    R_CUDA(cudaMalloc(&row_cum, (size_t)NN * sizeof(double)));
    k_rand_rows<<<(unsigned)((N + 7) / 8), 256, 0, s>>>((int)N, d_e, nullptr, row_n, row_c, row_cum);
    NHP_LAUNCHED(ctx);
    R_CUDA(cudaMalloc(&d_data, (size_t)(N * T) * sizeof(int)));
    R_CUDA(cudaMemsetAsync(d_data, 0, (size_t)(N * T) * sizeof(int), s));
    R_CUDA(cudaMalloc(&ev_t, (size_t)cap * sizeof(int)));
    R_CUDA(cudaMalloc(&ev_c, (size_t)cap * sizeof(int)));
    // ---- generation 0
    int64_t cnt_len = std::max<int64_t>(N, 1 << 20);
    R_CUDA(cudaMalloc(&d_cnt, (size_t)(cnt_len + 1) * sizeof(long long)));
    R_CUDA(cudaMalloc(&d_off, (size_t)(cnt_len + 1) * sizeof(long long)));
    size_t tmp_bytes = 0, need = 0;
    auto ensure_tmp = [&](size_t bytes) -> cudaError_t {
        if (bytes <= tmp_bytes) return cudaSuccess;
        cudaStreamSynchronize(s);
        cudaFree(d_tmp); d_tmp = nullptr; tmp_bytes = 0;
        cudaError_t e = cudaMalloc(&d_tmp, bytes);
        if (e == cudaSuccess) tmp_bytes = bytes;
        return e;
    };
    auto ensure_cnt = [&](int64_t len) -> cudaError_t {
        if (len <= cnt_len) return cudaSuccess;
        cudaStreamSynchronize(s);
        cudaFree(d_cnt); cudaFree(d_off); d_cnt = d_off = nullptr;
        cnt_len = len;
        cudaError_t e = cudaMalloc(&d_cnt, (size_t)(len + 1) * sizeof(long long));
        if (e == cudaSuccess) e = cudaMalloc(&d_off, (size_t)(len + 1) * sizeof(long long));
        return e;
    };
    // exclusive scan of d_cnt[0..len) into d_off[0..len]; returns the total
    auto scan_total = [&](int64_t len, long long *total) -> int {
        R_CUDA(cudaMemsetAsync(d_cnt + len, 0, sizeof(long long), s));
        cub::DeviceScan::ExclusiveSum(nullptr, need, d_cnt, d_off, (int)(len + 1), s);
        R_CUDA(ensure_tmp(need));
        R_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tmp_bytes, d_cnt, d_off, (int)(len + 1), s));
        NHP_LAUNCHED(ctx);
        R_CUDA(cudaMemcpyAsync(total, d_off + len, sizeof(long long), cudaMemcpyDeviceToHost, s));
        R_CUDA(cudaStreamSynchronize(s));
        return NHP_OK;
    };
    k_drand_base_counts<<<(unsigned)((N + 127) / 128), 128, 0, s>>>((int)N, ctx->dd_lambda0, ctx->ddt * (double)T, seed, d_cnt);
    NHP_LAUNCHED(ctx);
    long long n0 = 0;
    { int rc = scan_total(N, &n0); if (rc != NHP_OK) return rc; }
    if (n0 > cap) return fin(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_disc_rand: the sample needs more than max_events = %lld events (generation 0 alone has %lld)", (long long)cap, n0));
    if (n0 > 0) {
        k_drand_base_emit<<<(unsigned)((n0 + 255) / 256), 256, 0, s>>>((int)N, d_off, T, seed, ev_t, ev_c, n0, d_data);
        NHP_LAUNCHED(ctx);
    }
    // ---- later generations
    const size_t smem = (size_t)(L * B + B) * sizeof(double);
    if (smem > 48 * 1024) R_CUDA(cudaFuncSetAttribute(k_drand_child_emit, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    long long g0 = 0, ng = n0, total_n = n0;
    for (uint32_t gen = 1; ng > 0 && gen < 100000u; gen++) {
        R_CUDA(ensure_cnt(ng));
        k_drand_child_counts<<<(unsigned)((ng + 255) / 256), 256, 0, s>>>(ev_c, g0, ng, (int)N, row_n, row_cum, seed, gen, d_cnt);
        NHP_LAUNCHED(ctx);
        long long nchild = 0;
        { int rc = scan_total(ng, &nchild); if (rc != NHP_OK) return rc; }
        if (total_n + nchild > cap)
            return fin(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_disc_rand: the sample needs more than max_events = %lld events (is the process stable?)", (long long)cap));
        if (nchild > 0) {
            k_drand_child_emit<<<(unsigned)((nchild + 255) / 256), 256, smem, s>>>(ev_t, ev_c, g0, ng, d_off, nchild, total_n, (int)N, (int)B, (int)L, T, row_n, row_c,
                                                                                   row_cum, ctx->dd_theta, d_phi, seed, gen, d_data);
            NHP_LAUNCHED(ctx);
        }
        g0 = total_n; ng = nchild; total_n += nchild;
    }
    R_CUDA(cudaGetLastError());
    int *grid = d_data;
    d_data = nullptr;  // the handle owns the grid from here on
    fin(NHP_OK);
    return nhp_disc_from_device(ctx, grid, N, T, 0, out);
}

// data[n + N*t] (Julia's Matrix{Int64}) of every bin of the handle, halo included
__global__ void k_disc_widen(const int *__restrict__ src, int64_t n, int64_t *__restrict__ dst) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) dst[i] = (int64_t)src[i];
}
extern "C" int nhp_disc_download(nhp_ctx *ctx, nhp_disc *dd, int64_t *data) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr && data != nullptr, NHP_ERR_INVALID, "nhp_disc_download: NULL argument");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t n = dd->N * dd->T;
    cudaStream_t s = ctx->stream;
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)n * sizeof(int64_t), &scratch));
    k_disc_widen<<<(unsigned)((n + 255) / 256), 256, 0, s>>>(dd->d_data, n, (int64_t *)scratch);
    NHP_LAUNCHED(ctx);
    NHP_CUDA(ctx, cudaMemcpyAsync(data, scratch, (size_t)n * sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    NHP_CUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}
extern "C" int64_t nhp_disc_events_count(const nhp_disc *dd) { return dd ? dd->total_events : 0; }
