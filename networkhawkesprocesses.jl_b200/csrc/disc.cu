// disc.cu -- discrete-time path (discrete.jl, parents.jl:82-177, impulses.jl:310-371, weights.jl:70-91,
// baselines.jl:402-456).
//
// Device layout: counts d_data[t*N + n] (int32; same order as Julia's data[n + N*t]); the
// convolution is kept as convT[t*(N*B) + p*B + b] (the (p,b) axis contiguous) so that the
// contraction  lambda = conv * bump  is a row-major GEMM and the Gibbs / VB / adjacency consumers
// read one contiguous row per non-zero bin.  The reference's dense T x N x (1+N*B) `parents` / `u`
// arrays (1.9 TB at config 3) are never materialised: every downstream statistic is weighted by
// data[c,t], so only the ~4 % non-zero bins are visited (CSR by child node, built at upload).
#include "nhp_internal.cuh"
#include <cub/cub.cuh>
#include <algorithm>
#include <vector>

struct DiscExtra {  // hangs off nhp_disc (kept here so the public struct stays small)
    int64_t nnz = 0;
    int *nz_t = nullptr;        // [nnz] time bin, grouped by child, time order inside a child
    int *nz_s = nullptr;        // [nnz] count
    int64_t *nz_off = nullptr;  // [nnz] index of the bin's first uniform ((t outer, c inner, draw) order)
    int *child_ptr = nullptr;   // [N+1]
    double *rowsum = nullptr;   // [N] sum_t data[p,t] over own bins
    double *phi = nullptr;      // [L*B]
    double *csum = nullptr;     // [N*B] sum over own bins of convT[:, k]
    int max_ne = 0;             // most non-zero bins of one child (grid of the streaming adjacency sweep)
};
static DiscExtra *extra_of(nhp_disc *dd) { return reinterpret_cast<DiscExtra *>(dd->d_scan); }

#define DCUDA(ctx, call) NHP_CUDA(ctx, call)

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) v += __shfl_xor_sync(0xffffffffu, v, d);
    return v;
}

// ---------------------------------------------------------------------------------------
// upload
// ---------------------------------------------------------------------------------------
__global__ void k_disc_ingest(const int64_t *__restrict__ src, int *__restrict__ dst, int64_t total, int *flag) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int64_t v = src[i];
    if (v < 0 || v > 2147483647) atomicOr(flag, 1);
    dst[i] = (int)v;
}
__global__ void k_disc_flags(const int *__restrict__ data, int64_t total, int64_t first, unsigned char *__restrict__ flags, int64_t *__restrict__ cnt64) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    int v = i >= first ? data[i] : 0;
    flags[i] = v > 0;
    cnt64[i] = v;
}
__global__ void k_disc_gather(const int64_t *__restrict__ idx, const int64_t *__restrict__ scan, const int *__restrict__ data, int64_t nnz, int N,
                              int *__restrict__ key_c, int *__restrict__ pos) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    key_c[i] = (int)(idx[i] % N);
    pos[i] = (int)i;
}
__global__ void k_disc_fill(const int *__restrict__ pos_sorted, const int *__restrict__ key_sorted, const int64_t *__restrict__ idx, const int64_t *__restrict__ scan,
                            const int *__restrict__ data, int64_t nnz, int N, int *__restrict__ nz_t, int *__restrict__ nz_s, int64_t *__restrict__ nz_off,
                            int *__restrict__ child_cnt) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    int64_t lin = idx[pos_sorted[i]];
    nz_t[i] = (int)(lin / N);
    nz_s[i] = data[lin];
    nz_off[i] = scan[lin];
    atomicAdd(&child_cnt[key_sorted[i] + 1], 1);
}
__global__ void k_disc_rowsum(const int *__restrict__ data, int N, int64_t T, int64_t t0, double *__restrict__ rowsum) {
    // one block per slab of time bins; threads over nodes
    for (int n = threadIdx.x; n < N; n += blockDim.x) {
        long long s = 0;
        for (int64_t t = t0 + blockIdx.x; t < T; t += gridDim.x) s += data[t * N + n];
        if (s) atomicAdd(&rowsum[n], (double)s);
    }
}
__global__ void k_prefix_small(int *v, int n) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        int run = 0;
        for (int i = 0; i <= n; i++) { run += v[i]; v[i] = run; }
    }
}

extern "C" int nhp_disc_free(nhp_ctx *ctx, nhp_disc *dd) {
    if (!dd) return NHP_OK;
    if (ctx) { cudaSetDevice(ctx->device); cudaStreamSynchronize(ctx->stream); }
    DiscExtra *ex = extra_of(dd);
    if (ex) {
        cudaFree(ex->nz_t); cudaFree(ex->nz_s); cudaFree(ex->nz_off); cudaFree(ex->child_ptr); cudaFree(ex->rowsum); cudaFree(ex->phi); cudaFree(ex->csum);
        delete ex;
    }
    cudaFree(dd->d_data); cudaFree(dd->d_conv);
    delete dd;
    return NHP_OK;
}

extern "C" int nhp_disc_upload(nhp_ctx *ctx, const int64_t *data, int64_t N, int64_t T, int64_t t_halo, nhp_disc **out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, out != nullptr && data != nullptr, NHP_ERR_INVALID, "nhp_disc_upload: NULL argument");
    *out = nullptr;
    NHP_CHECK(ctx, N >= 1 && N <= 32768 && T >= 1 && t_halo >= 0 && t_halo < T, NHP_ERR_INVALID, "nhp_disc_upload: bad dimensions N=%lld T=%lld t_halo=%lld", (long long)N, (long long)T, (long long)t_halo);
    NHP_CHECK(ctx, N * T < (int64_t)2147483000, NHP_ERR_INVALID, "nhp_disc_upload: N*T must stay below 2^31 per handle (shard the time axis)");
    DCUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int64_t total = N * T;
    int *d_data = nullptr;
    auto fail = [&](int rc) { cudaStreamSynchronize(s); cudaFree(d_data); return rc; };
#define IN_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__))); } while (0)
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)total * sizeof(int64_t), &scratch));
    IN_CUDA(cudaMalloc(&d_data, (size_t)total * sizeof(int)));
    IN_CUDA(cudaMemcpyAsync(scratch, data, (size_t)total * sizeof(int64_t), cudaMemcpyHostToDevice, s));
    IN_CUDA(cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
    unsigned blocks = (unsigned)((total + 255) / 256);
    k_disc_ingest<<<blocks, 256, 0, s>>>((const int64_t *)scratch, d_data, total, ctx->d_flag);
    NHP_LAUNCHED(ctx);
    int flag = 0;
    IN_CUDA(cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    IN_CUDA(cudaStreamSynchronize(s));
#undef IN_CUDA
    if (flag & 1) return fail(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_disc_upload: counts must be in [0, 2^31)"));
    return nhp_disc_from_device(ctx, d_data, N, T, t_halo, out);
}

// Everything a handle derives from its counts, for a grid already on the device (the upload's, the simulator's): the non-zero own
// bins in memory order, the running draw index, the per-child CSR, the row sums, total_events and the longest column.  Takes
// ownership of d_data (freed with the handle, or here on failure).
int nhp_disc_from_device(nhp_ctx *ctx, int *d_data, int64_t N, int64_t T, int64_t t_halo, nhp_disc **out) {
    *out = nullptr;
    cudaStream_t s = ctx->stream;
    const int64_t total = N * T, first = t_halo * N;
    nhp_disc *dd = new nhp_disc();
    DiscExtra *ex = new DiscExtra();
    dd->N = N; dd->T = T; dd->t_halo = t_halo; dd->d_scan = reinterpret_cast<int64_t *>(ex);
    dd->d_data = d_data;
    unsigned char *d_flags = nullptr; int64_t *d_cnt = nullptr, *d_scan = nullptr, *d_idx = nullptr, *d_nnz = nullptr; void *d_tmp = nullptr;
    int *d_key = nullptr, *d_pos = nullptr, *d_key2 = nullptr, *d_pos2 = nullptr;
    auto fin = [&](int rc) {
        cudaStreamSynchronize(s);
        cudaFree(d_flags); cudaFree(d_cnt); cudaFree(d_scan); cudaFree(d_idx); cudaFree(d_nnz); cudaFree(d_tmp); cudaFree(d_key); cudaFree(d_pos); cudaFree(d_key2); cudaFree(d_pos2);
        if (rc != NHP_OK) nhp_disc_free(ctx, dd);
        return rc;
    };
#define UP_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fin(nhp_fail(ctx, NHP_ERR_CUDA, "%s failed: %s", #call, cudaGetErrorString(e__))); } while (0)
    unsigned blocks = (unsigned)((total + 255) / 256);
    // non-zero bins (own bins only) in memory order + the running draw index
    UP_CUDA(cudaMalloc(&d_flags, (size_t)total));
    UP_CUDA(cudaMalloc(&d_cnt, (size_t)total * sizeof(int64_t)));
    UP_CUDA(cudaMalloc(&d_scan, (size_t)total * sizeof(int64_t)));
    UP_CUDA(cudaMalloc(&d_idx, (size_t)total * sizeof(int64_t)));
    UP_CUDA(cudaMalloc(&d_nnz, 2 * sizeof(int64_t)));
    k_disc_flags<<<blocks, 256, 0, s>>>(dd->d_data, total, first, d_flags, d_cnt);
    NHP_LAUNCHED(ctx);
    size_t tb1 = 0, tb2 = 0;
    cub::DeviceScan::ExclusiveSum(nullptr, tb1, d_cnt, d_scan, (int)total, s);
    cub::CountingInputIterator<int64_t> iota(0);
    cub::DeviceSelect::Flagged(nullptr, tb2, iota, d_flags, d_idx, d_nnz, (int)total, s);
    size_t tb = std::max(tb1, tb2);
    UP_CUDA(cudaMalloc(&d_tmp, tb));
    UP_CUDA(cub::DeviceScan::ExclusiveSum(d_tmp, tb, d_cnt, d_scan, (int)total, s));
    UP_CUDA(cub::DeviceSelect::Flagged(d_tmp, tb, iota, d_flags, d_idx, d_nnz, (int)total, s));
    NHP_LAUNCHED(ctx); NHP_LAUNCHED(ctx);
    int64_t h_nnz = 0, h_last[2] = {0, 0};
    UP_CUDA(cudaMemcpyAsync(&h_nnz, d_nnz, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    UP_CUDA(cudaMemcpyAsync(&h_last[0], d_scan + total - 1, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    UP_CUDA(cudaMemcpyAsync(&h_last[1], d_cnt + total - 1, sizeof(int64_t), cudaMemcpyDeviceToHost, s));
    UP_CUDA(cudaStreamSynchronize(s));
    if (h_nnz >= (int64_t)2147483000) return fin(nhp_fail(ctx, NHP_ERR_INVALID, "nhp_disc: too many non-zero bins"));
    ex->nnz = h_nnz;
    dd->total_events = h_last[0] + h_last[1];
    UP_CUDA(cudaMalloc(&ex->child_ptr, (size_t)(N + 1) * sizeof(int)));
    UP_CUDA(cudaMemsetAsync(ex->child_ptr, 0, (size_t)(N + 1) * sizeof(int), s));
    UP_CUDA(cudaMalloc(&ex->rowsum, (size_t)N * sizeof(double)));
    UP_CUDA(cudaMemsetAsync(ex->rowsum, 0, (size_t)N * sizeof(double), s));
    k_disc_rowsum<<<(unsigned)std::min<int64_t>(T - t_halo, 1024), 128, 0, s>>>(dd->d_data, (int)N, T, t_halo, ex->rowsum);
    NHP_LAUNCHED(ctx);
    if (h_nnz > 0) {
        UP_CUDA(cudaMalloc(&d_key, (size_t)h_nnz * sizeof(int))); UP_CUDA(cudaMalloc(&d_pos, (size_t)h_nnz * sizeof(int)));
        UP_CUDA(cudaMalloc(&d_key2, (size_t)h_nnz * sizeof(int))); UP_CUDA(cudaMalloc(&d_pos2, (size_t)h_nnz * sizeof(int)));
        UP_CUDA(cudaMalloc(&ex->nz_t, (size_t)h_nnz * sizeof(int))); UP_CUDA(cudaMalloc(&ex->nz_s, (size_t)h_nnz * sizeof(int)));
        UP_CUDA(cudaMalloc(&ex->nz_off, (size_t)h_nnz * sizeof(int64_t)));
        unsigned nb = (unsigned)((h_nnz + 255) / 256);
        k_disc_gather<<<nb, 256, 0, s>>>(d_idx, d_scan, dd->d_data, h_nnz, (int)N, d_key, d_pos);
        NHP_LAUNCHED(ctx);
        int bits = 1;
        while ((1 << bits) < N) bits++;
        size_t tb3 = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tb3, d_key, d_key2, d_pos, d_pos2, (int)h_nnz, 0, bits, s);
        if (tb3 > tb) { cudaFree(d_tmp); d_tmp = nullptr; UP_CUDA(cudaMalloc(&d_tmp, tb3)); tb = tb3; }
        UP_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tb3, d_key, d_key2, d_pos, d_pos2, (int)h_nnz, 0, bits, s));  // stable: time order kept per child
        NHP_LAUNCHED(ctx);
        k_disc_fill<<<nb, 256, 0, s>>>(d_pos2, d_key2, d_idx, d_scan, dd->d_data, h_nnz, (int)N, ex->nz_t, ex->nz_s, ex->nz_off, ex->child_ptr);
        NHP_LAUNCHED(ctx);
    }
    k_prefix_small<<<1, 32, 0, s>>>(ex->child_ptr, (int)N);
    NHP_LAUNCHED(ctx);
    UP_CUDA(cudaGetLastError());
    {  // the longest column depends on the data only: kept here so that no adjacency sweep synchronises to find it
        std::vector<int> cp((size_t)N + 1);
        UP_CUDA(cudaMemcpyAsync(cp.data(), ex->child_ptr, (size_t)(N + 1) * sizeof(int), cudaMemcpyDeviceToHost, s));
        UP_CUDA(cudaStreamSynchronize(s));
        for (int64_t c = 0; c < N; c++) ex->max_ne = std::max(ex->max_ne, cp[c + 1] - cp[c]);
    }
#undef UP_CUDA
    int rc = fin(NHP_OK);
    if (rc == NHP_OK) *out = dd;
    return rc;
}

// ---------------------------------------------------------------------------------------
// basis (host; impulses.jl:321-335) and convolution (discrete.jl:146-151)
// ---------------------------------------------------------------------------------------
extern "C" int nhp_disc_basis(int64_t L, int64_t B, double dt, double *phi) {
    if (L < 1 || B < 1 || !phi || !(dt > 0.0)) return NHP_ERR_INVALID;
    double sigma = (double)L / (double)(B - 1);
    for (int64_t b = 0; b < B; b++) {
        // means: LinRange(1, L, B+2)[2:end-1] when B < L, else LinRange(1, L, B)
        int64_t len = B < L ? B + 2 : B, j = B < L ? b + 1 : b;
        double tt = len == 1 ? 0.0 : (double)j / (double)(len - 1);
        double mu = len == 1 ? 1.0 : (1.0 - tt) * 1.0 + tt * (double)L;
        double s = 0.0;
        for (int64_t l = 0; l < L; l++) {
            double d = (double)(l + 1) - mu;
            double v = exp(-1.0 / 2.0 * (1.0 / sigma) / 2.0 * (d * d));  // exp(-1/2 * sigma^-1 / 2 * (lag - mu)^2)
            phi[l + L * b] = v;
            s += v;
        }
        for (int64_t l = 0; l < L; l++) phi[l + L * b] = phi[l + L * b] / (s * dt);
    }
    return NHP_OK;
}

// convT[t][p*B + b] = max(0, sum_{l=1..L, t-l>=0} phi[l-1 + L*b] * data[t-l][p]); lags ascending as in the FIR restatement
__global__ void __launch_bounds__(256) k_convolve(const int *__restrict__ data, int N, int64_t T, const double *__restrict__ phi, int L, int B,
                                                  double *__restrict__ convT) {
    extern __shared__ double s_phi[];
    for (int i = threadIdx.x; i < L * B; i += blockDim.x) s_phi[i] = phi[i];
    __syncthreads();
    const int NB = N * B;
    for (int64_t t = blockIdx.x; t < T; t += gridDim.x) {
        for (int k = threadIdx.x; k < NB; k += blockDim.x) {
            int p = k / B, b = k - p * B;
            double s = 0.0;
            for (int l = 1; l <= L; l++) {
                if (t - l < 0) break;
                int v = __ldg(data + (t - l) * N + p);
                if (v) s += s_phi[(l - 1) + L * b] * (double)v;
            }
            convT[t * NB + k] = s > 0.0 ? s : 0.0;
        }
    }
}
// Same arithmetic (lags ascending), one thread per (t, p) producing all B basis outputs from L coalesced count loads;
// the (t, p)-major thread order makes a warp's stores one contiguous 32*B*8-byte span of convT.
template <int BMAX>
__global__ void __launch_bounds__(256) k_convolve_tp(const int *__restrict__ data, int N, int64_t T, const double *__restrict__ phi, int L, int B,
                                                     double *__restrict__ convT) {
    extern __shared__ double s_phi[];
    for (int i = threadIdx.x; i < L * B; i += blockDim.x) s_phi[i] = phi[i];
    __syncthreads();
    const int64_t total = T * N;
    for (int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; e < total; e += (int64_t)gridDim.x * blockDim.x) {
        const int64_t t = e / N;
        const int p = (int)(e - t * N);
        double acc[BMAX];
#pragma unroll
        for (int b = 0; b < BMAX; b++) acc[b] = 0.0;
        for (int l = 1; l <= L; l++) {
            if (t - l < 0) break;
            const int v = __ldg(data + (t - l) * N + p);
            if (v) {
                const double dv = (double)v;
#pragma unroll
                for (int b = 0; b < BMAX; b++)
                    if (b < B) acc[b] += s_phi[(l - 1) + L * b] * dv;
            }
        }
        double *dst = convT + e * B;
#pragma unroll
        for (int b = 0; b < BMAX; b++)
            if (b < B) dst[b] = acc[b] > 0.0 ? acc[b] : 0.0;
    }
}

// HBM-bound form (B <= 8, L <= 64, N <= 256): a thread owns one node p and walks SEGMENTS of consecutive time rows, so
//  (i)   the non-zero lags of its window live in a bit mask that slides with t and the last RS >= L counts in a per-thread ring in
//        shared memory (one global count load per (t, p) instead of L; the counts are sparse, 4 % non-zero bins at config 3); only
//        the non-zero lags take the B multiply-adds, lags ascending as before (same rounding),
//  (ii)  the column sums sum_t convT[t][p*B + b] over the own bins accumulate in registers and the separate pass that re-read all of
//        convT (9.6 GB at config 3) is gone,
//  (iii) a warp's 32 (t, p..p+31) results -- one contiguous span of 32*B doubles of convT -- go through a per-warp staging buffer
//        (pitch B + 1 for even B: conflict-free) and leave as fully coalesced stores (the thread-per-(t,p) stores were 8 bytes at a
//        8*B-byte stride).
// PW = N rounded up to whole warps, R = row groups per CTA (blockDim = PW * R); CONV_TT = rows per segment; RS = ring slots (power of 2).
constexpr int CONV_TT = 128;
template <typename M> __device__ __forceinline__ int conv_ffs(M m);
template <> __device__ __forceinline__ int conv_ffs<unsigned>(unsigned m) { return __ffs((int)m); }
template <> __device__ __forceinline__ int conv_ffs<unsigned long long>(unsigned long long m) { return __ffsll((long long)m); }
template <int B, typename M>  // M: the lag mask, 32 bits when L <= 32
__global__ void __launch_bounds__(256, 4) k_convolve_rows(const int *__restrict__ data, int N, int64_t T, int64_t t_own, const double *__restrict__ phi, int L,
                                                          int PW, int R, int RS, double *__restrict__ convT, double *__restrict__ csum) {
    constexpr int PITCH = (B & 1) ? B : B + 1;
    extern __shared__ double s_cv[];  // [L * B] phi | per warp: [32 * PITCH] staging | [RS][blockDim] ring of counts
    double *s_phi = s_cv;
    for (int i = threadIdx.x; i < L * B; i += blockDim.x) s_phi[i] = phi[i];
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
    double *stg = s_cv + L * B + warp * 32 * PITCH;
    int *ring = reinterpret_cast<int *>(s_cv + L * B + nwarp * 32 * PITCH) + threadIdx.x;  // slot k of this thread: ring[k * blockDim.x]
    const int bd = blockDim.x, rmask = RS - 1;
    const int r = threadIdx.x / PW, p = threadIdx.x - r * PW;  // warps never straddle row groups: PW is a multiple of 32
    const int p0 = p - lane;                                  // first node of this warp
    const int nq = max(0, min(32, N - p0)) * B;               // doubles this warp writes per row
    const int NB = N * B;
    const bool live = p < N;
    const M lmask = L >= (int)(8 * sizeof(M)) ? ~(M)0 : (M)(((M)1 << L) - (M)1);
    int rd[B];  // staged position of the m-th double this lane stores: element q = lane + 32 m sits at (q / B) * PITCH + q % B
#pragma unroll
    for (int m = 0; m < B; m++) { const int q = lane + 32 * m; rd[m] = (q / B) * PITCH + q % B; }
    double cs[B];
#pragma unroll
    for (int b = 0; b < B; b++) cs[b] = 0.0;
    const int64_t nseg = (T + CONV_TT - 1) / CONV_TT;
    for (int64_t seg = (int64_t)blockIdx.x * R + r; seg < nseg; seg += (int64_t)gridDim.x * R) {
        const int64_t tb = seg * CONV_TT;
        const int nt = (int)min((int64_t)CONV_TT, T - tb);
        M nz = 0;  // bit l - 1: data[t - l][p] != 0
        const int *col = data + tb * N + (live ? p : 0);
        if (live) {
            const int lmax = (int)min((int64_t)L, tb);
            for (int l = 1; l <= lmax; l++) {
                const int v = __ldg(col - l * N);
                ring[((int)(tb & rmask) - l & rmask) * bd] = v;
                nz |= (M)(v != 0) << (l - 1);
            }
        }
        int slot = (int)(tb & rmask);  // ring slot of row t
        double *dst = convT + tb * NB + (int64_t)p0 * B;
        for (int it = 0; it < nt; it++, col += N, dst += NB, slot = (slot + 1) & rmask) {
            double acc[B];
#pragma unroll
            for (int b = 0; b < B; b++) acc[b] = 0.0;
            const int cur = live ? __ldg(col) : 0;  // enters the window of row t + 1
            for (M m = nz; m;) {
                const int l1 = conv_ffs<M>(m) - 1;  // lag - 1
                m &= m - 1;
                const double dv = (double)ring[((slot - 1 - l1) & rmask) * bd];
                const double *ph = s_phi + l1;
#pragma unroll
                for (int b = 0; b < B; b++) acc[b] += ph[L * b] * dv;
            }
            ring[slot * bd] = cur;
            nz = ((nz << 1) | (M)(cur != 0)) & lmask;
            const double ownf = tb + it >= t_own ? 1.0 : 0.0;
#pragma unroll
            for (int b = 0; b < B; b++) {
                const double v = __double2hiint(acc[b]) < 0 ? 0.0 : acc[b];  // max(0, .): negative sums (a basis with negative lobes) clamp to zero
                stg[lane * PITCH + b] = v;
                cs[b] = fma(ownf, v, cs[b]);
            }
            __syncwarp();
            if (nq == 32 * B) {
#pragma unroll
                for (int m = 0; m < B; m++) dst[lane + 32 * m] = stg[rd[m]];
            } else {
#pragma unroll
                for (int m = 0; m < B; m++)
                    if (lane + 32 * m < nq) dst[lane + 32 * m] = stg[rd[m]];
            }
            __syncwarp();
        }
    }
    if (live) {
#pragma unroll
        for (int b = 0; b < B; b++)
            if (cs[b] != 0.0) atomicAdd(&csum[p * B + b], cs[b]);
    }
}
typedef void (*conv_rows_fn)(const int *, int, int64_t, int64_t, const double *, int, int, int, int, double *, double *);
template <typename M> static conv_rows_fn conv_rows_kernel_m(int B) {
    switch (B) {
        case 1: return k_convolve_rows<1, M>; case 2: return k_convolve_rows<2, M>; case 3: return k_convolve_rows<3, M>; case 4: return k_convolve_rows<4, M>;
        case 5: return k_convolve_rows<5, M>; case 6: return k_convolve_rows<6, M>; case 7: return k_convolve_rows<7, M>; default: return k_convolve_rows<8, M>;
    }
}
static conv_rows_fn conv_rows_kernel(int B, int L) { return L <= 32 ? conv_rows_kernel_m<unsigned>(B) : conv_rows_kernel_m<unsigned long long>(B); }

// Julia layout export: out[t + T*(n + N*b)] = convT[t][n*B + b]   (tiled transpose)
__global__ void k_conv_export(const double *__restrict__ convT, int N, int B, int64_t T, double *__restrict__ out) {
    __shared__ double tile[32][33];
    const int NB = N * B;
    int64_t t0 = (int64_t)blockIdx.x * 32;
    int k0 = blockIdx.y * 32;
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int64_t t = t0 + r; int k = k0 + threadIdx.x;
        tile[r][threadIdx.x] = (t < T && k < NB) ? convT[t * NB + k] : 0.0;
    }
    __syncthreads();
    for (int r = threadIdx.y; r < 32; r += blockDim.y) {
        int k = k0 + r; int64_t t = t0 + threadIdx.x;
        if (t < T && k < NB) { int p = k / B, b = k - p * B; out[t + T * (p + (int64_t)N * b)] = tile[threadIdx.x][r]; }
    }
}
// csum[k] = sum over own bins of convT[t][k]
__global__ void k_conv_colsum(const double *__restrict__ convT, int NB, int64_t T, int64_t t0, double *__restrict__ csum) {
    for (int k = threadIdx.x; k < NB; k += blockDim.x) {
        double s = 0.0;
        for (int64_t t = t0 + blockIdx.x; t < T; t += gridDim.x) s += convT[t * NB + k];
        atomicAdd(&csum[k], s);
    }
}

extern "C" int nhp_disc_convolve(nhp_ctx *ctx, nhp_disc *dd, const double *phi, int64_t L, int64_t B, double *conv_out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd && phi && L >= 1 && B >= 1 && L * B <= 4096, NHP_ERR_INVALID, "nhp_disc_convolve: bad argument");
    DCUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    DiscExtra *ex = extra_of(dd);
    const int64_t NB = dd->N * B;
    if (dd->B != B || !dd->d_conv) {
        DCUDA(ctx, cudaStreamSynchronize(s));
        cudaFree(dd->d_conv); dd->d_conv = nullptr;
        cudaFree(ex->csum); ex->csum = nullptr;
        DCUDA(ctx, cudaMalloc(&dd->d_conv, (size_t)dd->T * NB * sizeof(double)));
        DCUDA(ctx, cudaMalloc(&ex->csum, (size_t)NB * sizeof(double)));
    }
    cudaFree(ex->phi); ex->phi = nullptr;
    DCUDA(ctx, cudaMalloc(&ex->phi, (size_t)(L * B) * sizeof(double)));
    DCUDA(ctx, cudaMemcpyAsync(ex->phi, phi, (size_t)(L * B) * sizeof(double), cudaMemcpyHostToDevice, s));
    dd->L = L; dd->B = B;
    NHP_TRY(nhp_timer_begin(ctx));
    int grid = (int)std::min<int64_t>(dd->T, (int64_t)ctx->sm_count * 16);
    const char *envr = getenv("NHP_DISC_CONV_ROWS");
    if (B <= 8 && L <= 64 && dd->N <= 256 && !(envr && atoi(envr) == 0)) {
        // rows kernel: stores through a staging buffer, column sums fused (no second pass over convT)
        const int PW = (int)((dd->N + 31) / 32) * 32, R = std::max(1, 256 / PW), threads = PW * R;
        int RS = 1;
        while (RS < L) RS <<= 1;
        const int pitch = (B & 1) ? (int)B : (int)B + 1;
        const size_t smem = ((size_t)(L * B) + (size_t)(threads / 32) * 32 * pitch) * sizeof(double) + (size_t)RS * threads * sizeof(int);
        conv_rows_fn kern = conv_rows_kernel((int)B, (int)L);
        DCUDA(ctx, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));
        int per_sm = 1;
        DCUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, threads, smem));
        per_sm = std::max(per_sm, 1);
        const int64_t nseg = (dd->T + CONV_TT - 1) / CONV_TT;
        const int g3 = (int)std::min<int64_t>((nseg + R - 1) / R, (int64_t)ctx->sm_count * per_sm);
        DCUDA(ctx, cudaMemsetAsync(ex->csum, 0, (size_t)NB * sizeof(double), s));
        kern<<<g3, threads, smem, s>>>(dd->d_data, (int)dd->N, dd->T, dd->t_halo, ex->phi, (int)L, PW, R, RS, dd->d_conv, ex->csum);
        NHP_LAUNCHED(ctx);
        DCUDA(ctx, cudaGetLastError());
        NHP_TRY(nhp_timer_end(ctx));
        goto exported;
    }
    if (B <= 8) {
        int g2 = (int)std::min<int64_t>((dd->T * dd->N + 255) / 256, (int64_t)ctx->sm_count * 32);
        k_convolve_tp<8><<<g2, 256, (size_t)(L * B) * sizeof(double), s>>>(dd->d_data, (int)dd->N, dd->T, ex->phi, (int)L, (int)B, dd->d_conv);
    } else
    k_convolve<<<grid, 256, (size_t)(L * B) * sizeof(double), s>>>(dd->d_data, (int)dd->N, dd->T, ex->phi, (int)L, (int)B, dd->d_conv);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaMemsetAsync(ex->csum, 0, (size_t)NB * sizeof(double), s));
    k_conv_colsum<<<(unsigned)std::min<int64_t>(dd->T - dd->t_halo, 2048), 256, 0, s>>>(dd->d_conv, (int)NB, dd->T, dd->t_halo, ex->csum);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaGetLastError());
    NHP_TRY(nhp_timer_end(ctx));
exported:
    if (conv_out) {
        void *scratch;
        NHP_TRY(nhp_scratch(ctx, (size_t)dd->T * NB * sizeof(double), &scratch));
        dim3 g((unsigned)((dd->T + 31) / 32), (unsigned)((NB + 31) / 32)), b(32, 8);
        k_conv_export<<<g, b, 0, s>>>(dd->d_conv, (int)dd->N, (int)B, dd->T, (double *)scratch);
        NHP_LAUNCHED(ctx);
        DCUDA(ctx, cudaMemcpyAsync(conv_out, scratch, (size_t)dd->T * NB * sizeof(double), cudaMemcpyDeviceToHost, s));
        DCUDA(ctx, cudaStreamSynchronize(s));
    }
    return NHP_OK;
}

// the device-resident convolution of a handle in the reference's layout conv[t + T*(n + N*b)] (what `convolve` returns in Julia);
// only needed when host code looks inside it -- the sweeps read it on the device
extern "C" int nhp_disc_conv_export(nhp_ctx *ctx, nhp_disc *dd, double *conv_out) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr && conv_out != nullptr, NHP_ERR_INVALID, "nhp_disc_conv_export: NULL argument");
    NHP_CHECK(ctx, dd->d_conv != nullptr && dd->B > 0, NHP_ERR_STATE, "nhp_disc_conv_export: call nhp_disc_convolve first");
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int64_t NB = dd->N * dd->B;
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)dd->T * NB * sizeof(double), &scratch));
    dim3 g((unsigned)((dd->T + 31) / 32), (unsigned)((NB + 31) / 32)), b(32, 8);
    k_conv_export<<<g, b, 0, s>>>(dd->d_conv, (int)dd->N, (int)dd->B, dd->T, (double *)scratch);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaMemcpyAsync(conv_out, scratch, (size_t)dd->T * NB * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// parameters: bump[p,c,b] = [A] W theta dt  (discrete.jl:381-385, 511-516)
// ---------------------------------------------------------------------------------------
__global__ void k_bump(int N, int B, const double *__restrict__ W, const double *__restrict__ A, const double *__restrict__ theta, double dt,
                       double *__restrict__ bumpM /* [k][c] */, double *__restrict__ bumpT /* [c][k] */) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t NB = (int64_t)N * B;
    if (e >= NB * N) return;
    int c = (int)(e / NB), k = (int)(e % NB);
    int p = k / B, b = k - p * B;
    int64_t pc = p + (int64_t)N * c;
    double w = W[pc], th = theta[pc + (int64_t)N * N * b];
    double v = A ? A[pc] * w * th * dt : w * th * dt;
    bumpT[e] = v;
    bumpM[(int64_t)k * N + c] = v;
}

// btc[i] = bumpT[c][klist[i]] for the entries of child c
__global__ void k_compact_bump(int NB, const double *__restrict__ bumpT, const int *__restrict__ klist, const int *__restrict__ kptr, double *__restrict__ btc) {
    const int c = blockIdx.x;
    for (int i = kptr[c] + threadIdx.x; i < kptr[c + 1]; i += blockDim.x) btc[i] = bumpT[(int64_t)c * NB + klist[i]];
}

// Compact per-child lists of the structurally non-zero (parent, basis) entries, k = p*B + b with [A]W[p,c] != 0, built on the
// device from the resident parameters: a count per child, one scan over the children, then every child writes its list in
// ascending k.  Only sparse effective weights (<= 50 % non-zero) get lists; dense models keep the full parent scan.
__global__ void __launch_bounds__(256) k_disc_klist_count(int N, const double *__restrict__ W, const double *__restrict__ A, int *__restrict__ kcnt,
                                                          double *__restrict__ acol) {
    __shared__ int s_n[8];
    __shared__ double s_a[8];
    const int c = blockIdx.x, lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    int n = 0;
    double a = 0.0;
    for (int p = threadIdx.x; p < N; p += 256) {
        const int64_t e = p + (int64_t)N * c;
        const double av = A ? A[e] : 1.0;
        n += (A ? av * W[e] : W[e]) != 0.0;
        a += av;
    }
    n = __reduce_add_sync(0xffffffffu, n);
    a = warp_sum_d(a);
    if (lane == 0) { s_n[warp] = n; s_a[warp] = a; }
    __syncthreads();
    if (threadIdx.x == 0) {  // fixed order: the same sum of A on every call
        int tn = 0;
        double ta = 0.0;
        for (int w = 0; w < 8; w++) { tn += s_n[w]; ta += s_a[w]; }
        kcnt[c] = tn;
        acol[c] = ta;
    }
}
// kptr[c] = B * (non-zero entries of the children before c); out = [list length, longest list, non-zero entries, sum of A]
__global__ void __launch_bounds__(1024) k_disc_klist_scan(int N, int B, const int *__restrict__ kcnt, const double *__restrict__ acol, int *__restrict__ kptr,
                                                          double *__restrict__ out) {
    typedef cub::BlockScan<int, 1024> Scan;
    typedef cub::BlockReduce<double, 1024> Red;
    __shared__ union { typename Scan::TempStorage scan; typename Red::TempStorage red; } tmp;
    __shared__ int s_max;
    if (threadIdx.x == 0) s_max = 0;
    __syncthreads();
    int carry = 0;
    double asum = 0.0;  // thread 0
    for (int c0 = 0; c0 < N; c0 += 1024) {
        const int c = c0 + threadIdx.x;
        const int v = c < N ? kcnt[c] : 0;
        int excl, tot;
        Scan(tmp.scan).ExclusiveSum(v, excl, tot);
        if (c < N) kptr[c] = (carry + excl) * B;
        carry += tot;
        if (v) atomicMax(&s_max, v);
        __syncthreads();
        const double a = Red(tmp.red).Sum(c < N ? acol[c] : 0.0);
        if (threadIdx.x == 0) asum += a;
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        kptr[N] = carry * B;
        out[0] = (double)carry * B; out[1] = (double)s_max * B; out[2] = (double)carry; out[3] = asum;
    }
}
__global__ void __launch_bounds__(256) k_disc_klist_fill(int N, int B, const double *__restrict__ W, const double *__restrict__ A, const int *__restrict__ kptr,
                                                         int *__restrict__ klist) {
    typedef cub::BlockScan<int, 256> Scan;
    __shared__ typename Scan::TempStorage tmp;
    const int c = blockIdx.x;
    int next = kptr[c];
    for (int p0 = 0; p0 < N; p0 += 256) {
        const int p = p0 + threadIdx.x;
        int f = 0;
        if (p < N) {
            const int64_t e = p + (int64_t)N * c;
            f = (A ? A[e] * W[e] : W[e]) != 0.0;
        }
        int r, tot;
        Scan(tmp).ExclusiveSum(f, r, tot);
        if (f) for (int b = 0; b < B; b++) klist[next + r * B + b] = p * B + b;
        next += tot * B;
        __syncthreads();
    }
}

// Everything that follows from the context's lambda0, W, A, theta: the bump table (both layouts), the compact parent lists, the
// density of the effective weights and the sum of A.  One synchronisation: four scalars come back to the host.
int nhp_disc_tables_refresh(nhp_ctx *ctx) {
    cudaStream_t s = ctx->stream;
    const int64_t N = ctx->dN, B = ctx->dB, NN = N * N, NB = N * B;
    const double *A = ctx->d_has_A ? ctx->dd_A : nullptr;
    k_bump<<<(unsigned)((NB * N + 255) / 256), 256, 0, s>>>((int)N, (int)B, ctx->dd_W, A, ctx->dd_theta, ctx->ddt, ctx->dd_bump, ctx->dd_bump + NB * N);
    NHP_LAUNCHED(ctx);
    k_disc_klist_count<<<(unsigned)N, 256, 0, s>>>((int)N, ctx->dd_W, A, ctx->dd_kcnt, ctx->dd_ksum + 4);
    NHP_LAUNCHED(ctx);
    k_disc_klist_scan<<<1, 1024, 0, s>>>((int)N, (int)B, ctx->dd_kcnt, ctx->dd_ksum + 4, ctx->dd_kptr, ctx->dd_ksum);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaGetLastError());
    double h[4];
    DCUDA(ctx, cudaMemcpyAsync(h, ctx->dd_ksum, sizeof(h), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaStreamSynchronize(s));
    ctx->dd_density = h[2] / (double)NN;
    ctx->dd_a_sum = A ? h[3] : (double)NN;
    ctx->dd_lists = false;
    ctx->dd_maxNA = 0;
    if (h[2] > 0.0 && ctx->dd_density <= 0.5) {
        const size_t need = (size_t)h[0];
        if (need > ctx->dd_klist_cap) {
            cudaFree(ctx->dd_klist); cudaFree(ctx->dd_btc);
            ctx->dd_klist = nullptr; ctx->dd_btc = nullptr; ctx->dd_klist_cap = 0;
            DCUDA(ctx, cudaMalloc(&ctx->dd_klist, need * sizeof(int)));
            DCUDA(ctx, cudaMalloc(&ctx->dd_btc, need * sizeof(double)));
            ctx->dd_klist_cap = need;
        }
        k_disc_klist_fill<<<(unsigned)N, 256, 0, s>>>((int)N, (int)B, ctx->dd_W, A, ctx->dd_kptr, ctx->dd_klist);
        NHP_LAUNCHED(ctx);
        k_compact_bump<<<(unsigned)N, 256, 0, s>>>((int)NB, ctx->dd_bump + NB * N, ctx->dd_klist, ctx->dd_kptr, ctx->dd_btc);
        NHP_LAUNCHED(ctx);
        DCUDA(ctx, cudaGetLastError());
        ctx->dd_maxNA = (int64_t)h[1];
        ctx->dd_lists = true;
    }
    return NHP_OK;
}

extern "C" int nhp_disc_params_set(nhp_ctx *ctx, int64_t N, int64_t B, const double *lambda0, const double *W, const double *A, const double *theta, double dt) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, N >= 1 && B >= 1 && lambda0 && W && theta && dt > 0.0, NHP_ERR_INVALID, "nhp_disc_params_set: bad argument");
    for (int64_t n = 0; n < N; n++) NHP_CHECK(ctx, lambda0[n] >= 0.0, NHP_ERR_INVALID, "DiscreteHomogeneousProcess: intensity parameter must be non-negative (baselines.jl:367)");
    DCUDA(ctx, cudaSetDevice(ctx->device));
    cudaStream_t s = ctx->stream;
    const int64_t NN = N * N, NB = N * B;
    if (ctx->dN != N || ctx->dB != B) {
        DCUDA(ctx, cudaStreamSynchronize(s));
        cudaFree(ctx->dd_lambda0); cudaFree(ctx->dd_W); cudaFree(ctx->dd_A); cudaFree(ctx->dd_theta); cudaFree(ctx->dd_bump);
        cudaFree(ctx->dd_klist); cudaFree(ctx->dd_kptr); cudaFree(ctx->dd_btc); cudaFree(ctx->dd_kcnt); cudaFree(ctx->dd_ksum);
        ctx->dd_lambda0 = ctx->dd_W = ctx->dd_A = ctx->dd_theta = ctx->dd_bump = ctx->dd_btc = ctx->dd_ksum = nullptr;
        ctx->dd_klist = ctx->dd_kptr = ctx->dd_kcnt = nullptr;
        ctx->dd_klist_cap = 0; ctx->dd_lists = false;
        ctx->dN = ctx->dB = 0;
        DCUDA(ctx, cudaMalloc(&ctx->dd_lambda0, (size_t)N * sizeof(double)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_W, (size_t)NN * sizeof(double)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_A, (size_t)NN * sizeof(double)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_theta, (size_t)(NN * B) * sizeof(double)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_bump, (size_t)(2 * NB * N) * sizeof(double)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_kptr, (size_t)(N + 1) * sizeof(int)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_kcnt, (size_t)N * sizeof(int)));
        DCUDA(ctx, cudaMalloc(&ctx->dd_ksum, (size_t)(4 + N) * sizeof(double)));
        ctx->dN = N; ctx->dB = B;
    }
    ctx->disc_set = false;
    ctx->ddt = dt; ctx->d_has_A = A != nullptr;
    DCUDA(ctx, cudaMemcpyAsync(ctx->dd_lambda0, lambda0, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, s));
    DCUDA(ctx, cudaMemcpyAsync(ctx->dd_W, W, (size_t)NN * sizeof(double), cudaMemcpyHostToDevice, s));
    if (A) DCUDA(ctx, cudaMemcpyAsync(ctx->dd_A, A, (size_t)NN * sizeof(double), cudaMemcpyHostToDevice, s));
    DCUDA(ctx, cudaMemcpyAsync(ctx->dd_theta, theta, (size_t)(NN * B) * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_TRY(nhp_disc_tables_refresh(ctx));
    ctx->disc_set = true;
    return NHP_OK;
}

// Current parameters in the layouts of nhp_disc_params_set; any pointer may be NULL
extern "C" int nhp_disc_params_get(nhp_ctx *ctx, double *lambda0, double *W, double *A, double *theta) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, ctx->disc_set, NHP_ERR_STATE, "nhp_disc_params_get: discrete parameters not set");
    NHP_CHECK(ctx, !A || ctx->d_has_A, NHP_ERR_STATE, "nhp_disc_params_get: the process has no adjacency matrix");
    DCUDA(ctx, cudaSetDevice(ctx->device));
    const int64_t N = ctx->dN, NN = N * N;
    cudaStream_t s = ctx->stream;
    if (lambda0) DCUDA(ctx, cudaMemcpyAsync(lambda0, ctx->dd_lambda0, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (W) DCUDA(ctx, cudaMemcpyAsync(W, ctx->dd_W, (size_t)NN * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (A) DCUDA(ctx, cudaMemcpyAsync(A, ctx->dd_A, (size_t)NN * sizeof(double), cudaMemcpyDeviceToHost, s));
    if (theta) DCUDA(ctx, cudaMemcpyAsync(theta, ctx->dd_theta, (size_t)(NN * ctx->dB) * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// link probability of the discrete BernoulliNetworkModel (networks.jl:45-54), kept apart from the continuous model's
extern "C" int nhp_disc_network_set(nhp_ctx *ctx, double rho) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, rho >= 0.0 && rho <= 1.0, NHP_ERR_INVALID, "BernoulliNetworkModel: link probability must be in [0, 1]");
    ctx->dd_rho = rho;
    return NHP_OK;
}
extern "C" int nhp_disc_network_get(const nhp_ctx *ctx, double *rho) {
    if (!ctx || !rho) return NHP_ERR_INVALID;
    *rho = ctx->dd_rho;
    return NHP_OK;
}

const double *nhp_disc_rowsum(nhp_disc *dd) { return extra_of(dd)->rowsum; }

static int disc_ready(nhp_ctx *ctx, nhp_disc *dd, const char *who) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd != nullptr, NHP_ERR_INVALID, "%s: data handle is NULL", who);
    NHP_CHECK(ctx, ctx->disc_set, NHP_ERR_STATE, "%s: discrete parameters not set (call nhp_disc_params_set)", who);
    NHP_CHECK(ctx, dd->d_conv != nullptr, NHP_ERR_STATE, "%s: call nhp_disc_convolve first", who);
    NHP_CHECK(ctx, dd->N == ctx->dN && dd->B == ctx->dB, NHP_ERR_INVALID, "%s: data (N=%lld,B=%lld) and parameters (N=%lld,B=%lld) disagree", who,
              (long long)dd->N, (long long)dd->B, (long long)ctx->dN, (long long)ctx->dB);
    DCUDA(ctx, cudaSetDevice(ctx->device));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// intensity / log-likelihood: lambda[t,c] = lambda0_c dt + sum_k convT[t,k] bumpM[k,c]   (discrete.jl:115-129)
// FP64 tensor-core contraction with a fused Poisson epilogue: mma.sync.aligned.m8n8k4.f64 (SASS DMMA.8x8x4; tcgen05
// has no FP64 kind).  CTA tile 128 rows x 8*NT columns, warp tile 16 x 8*NT (2 x NT accumulator tiles),
// k staged 16 at a time through shared memory with pitches chosen so every fragment load is conflict-free.
// Measured DMMA peak on B200: 36.7 TFLOP/s (nhp_bench_fp64 which=3) vs 33.8 TFLOP/s for DFMA, at 1/8 of
// the instruction count.
// ---------------------------------------------------------------------------------------
constexpr int DBM = 128, DBK = 16, DLDA = 20;

__device__ __forceinline__ void dmma_8x8x4(double &c0, double &c1, double a, double b) {
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};" : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

template <int NT, bool LOGLIK>
__global__ void __launch_bounds__(256) k_disc_dmma(const double *__restrict__ convT, const double *__restrict__ bumpM, const double *__restrict__ lambda0,
                                                   double dt, int N, int NB, int64_t T, int64_t t_first, const int *__restrict__ data,
                                                   double *__restrict__ lam_out, double *__restrict__ partials) {
    constexpr int BN = 8 * NT, LDB = BN + 4;
    extern __shared__ double s_dm[];  // two stages: A tiles [2][DBM * DLDA] | B tiles [2][DBK * LDB]
    double *const As0 = s_dm, *const Bs0 = s_dm + 2 * DBM * DLDA;
    __shared__ double red[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int g = lane >> 2, q = lane & 3;
    const int c0 = blockIdx.x * BN;                       // column block fastest: CTAs sharing the A rows run together (L2 reuse)
    const int64_t t0 = t_first + (int64_t)blockIdx.y * DBM;
    double acc[2][NT][2];
#pragma unroll
    for (int m = 0; m < 2; m++)
#pragma unroll
        for (int n = 0; n < NT; n++) acc[m][n][0] = acc[m][n][1] = 0.0;
    // software pipeline: the next k-slab is fetched into registers while the tensor cores work on the current one
    constexpr int BPT = (DBK * BN + 255) / 256;  // B-tile elements per thread
    const int ar = threadIdx.x >> 1, ah = threadIdx.x & 1;
    const int64_t at = t0 + ar;
    const bool avec = (NB % 4 == 0);             // rows are 32 B aligned: 256-bit loads
    double va[8], vb[BPT];
    auto fetch = [&](int k0) {
        const int kb = k0 + ah * 8;
        if (at < T && avec && kb + 8 <= NB) {
            const double *src = convT + at * NB + kb;
            asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(va[0]), "=d"(va[1]), "=d"(va[2]), "=d"(va[3]) : "l"(src));
            asm("ld.global.nc.v4.f64 {%0,%1,%2,%3}, [%4];" : "=d"(va[4]), "=d"(va[5]), "=d"(va[6]), "=d"(va[7]) : "l"(src + 4));
        } else {
#pragma unroll
            for (int j = 0; j < 8; j++) va[j] = (at < T && kb + j < NB) ? __ldg(convT + at * NB + kb + j) : 0.0;
        }
#pragma unroll
        for (int u = 0; u < BPT; u++) {
            const int e = threadIdx.x + u * 256;
            const int kk = e / BN, cc = e - kk * BN;
            vb[u] = (e < DBK * BN && k0 + kk < NB && c0 + cc < N) ? __ldg(bumpM + (int64_t)(k0 + kk) * N + c0 + cc) : 0.0;
        }
    };
    auto stash = [&](int stage) {
        double *As = As0 + stage * (DBM * DLDA), *Bs = Bs0 + stage * (DBK * LDB);
#pragma unroll
        for (int j = 0; j < 8; j++) As[ar * DLDA + ah * 8 + j] = va[j];
#pragma unroll
        for (int u = 0; u < BPT; u++) {
            const int e = threadIdx.x + u * 256;
            if (e < DBK * BN) { const int kk = e / BN, cc = e - kk * BN; Bs[kk * LDB + cc] = vb[u]; }
        }
    };
    // two shared-memory stages, ONE barrier per k-slab: while the tensor cores work on stage s the next slab (already in registers)
    // goes to stage s ^ 1, which every warp finished reading before the previous barrier
    fetch(0);
    stash(0);
    __syncthreads();
    int stage = 0;
    for (int k0 = 0; k0 < NB; k0 += DBK, stage ^= 1) {
        const bool more = k0 + DBK < NB;
        if (more) fetch(k0 + DBK);
        const double *As = As0 + stage * (DBM * DLDA), *Bs = Bs0 + stage * (DBK * LDB);
#pragma unroll
        for (int ks = 0; ks < DBK / 4; ks++) {
            double a[2], b[NT];
#pragma unroll
            for (int m = 0; m < 2; m++) a[m] = As[(warp * 16 + m * 8 + g) * DLDA + ks * 4 + q];
#pragma unroll
            for (int n = 0; n < NT; n++) b[n] = Bs[(ks * 4 + q) * LDB + n * 8 + g];
#pragma unroll
            for (int m = 0; m < 2; m++)
#pragma unroll
                for (int n = 0; n < NT; n++) dmma_8x8x4(acc[m][n][0], acc[m][n][1], a[m], b[n]);
        }
        if (more) stash(stage ^ 1);
        __syncthreads();
    }
    double part = 0.0;
#pragma unroll
    for (int m = 0; m < 2; m++) {
        const int64_t t = t0 + warp * 16 + m * 8 + g;
#pragma unroll
        for (int n = 0; n < NT; n++)
#pragma unroll
            for (int j = 0; j < 2; j++) {
                const int c = c0 + n * 8 + q * 2 + j;
                if (t < T && c < N) {
                    const double lam = lambda0[c] * dt + acc[m][n][j];
                    if (LOGLIK) {
                        // log pdf(Poisson(lam), s) = xlogy(s, lam) - lam - loggamma(s + 1)   (discrete.jl:98); most bins are empty: the
                        // logarithm is taken for s > 0 only and loggamma (0 for s = 0, 1) for s > 1 only
                        const int sct = data[t * N + c];
                        double term = -lam;
                        if (sct > 0) {
                            term += (double)sct * log(lam);
                            if (sct > 1) term -= lgamma((double)sct + 1.0);
                        }
                        part += term;
                    } else lam_out[t + T * (int64_t)c] = lam;
                }
            }
    }
    if (LOGLIK) {
        part = warp_sum_d(part);
        if (lane == 0) red[warp] = part;
        __syncthreads();
        if (threadIdx.x == 0) {
            double s = 0.0;
            for (int w = 0; w < 8; w++) s += red[w];
            partials[(size_t)blockIdx.y * gridDim.x + blockIdx.x] = s;
        }
    }
}

// number of 8-column accumulator tiles per warp: the candidate in 4..6 that wastes the fewest columns
static int pick_nt(int64_t N) {
    int best = 4;
    int64_t best_cols = -1;
    for (int nt = 4; nt <= 6; nt++) {
        int64_t bn = 8 * nt, cols = (N + bn - 1) / bn * bn;
        if (best_cols < 0 || cols < best_cols || (cols == best_cols && nt > best)) { best = nt; best_cols = cols; }
    }
    return best;
}

// returns the grid: one CTA (and one log-likelihood partial) per DBM x 8 pick_nt(N) tile
template <bool LOGLIK>
static dim3 launch_dmma(nhp_ctx *ctx, nhp_disc *dd, int64_t t_first, int64_t rows, double *lam_out, double *partials) {
    const int64_t N = dd->N, NB = N * dd->B;
    const int nt = pick_nt(N);
    dim3 grid((unsigned)((N + 8 * nt - 1) / (8 * nt)), (unsigned)((rows + DBM - 1) / DBM));
#define NHP_DMMA_CASE(NTV) { constexpr size_t smem = (size_t)(2 * DBM * DLDA + 2 * DBK * (8 * NTV + 4)) * sizeof(double); \
        cudaFuncSetAttribute(k_disc_dmma<NTV, LOGLIK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem); \
        k_disc_dmma<NTV, LOGLIK><<<grid, 256, smem, ctx->stream>>>(dd->d_conv, ctx->dd_bump, ctx->dd_lambda0, ctx->ddt, (int)N, (int)NB, dd->T, t_first, dd->d_data, lam_out, partials); }
    switch (nt) { case 4: NHP_DMMA_CASE(4) break; case 5: NHP_DMMA_CASE(5) break; default: NHP_DMMA_CASE(6) break; }
#undef NHP_DMMA_CASE
    NHP_LAUNCHED(ctx);
    return grid;
}

__global__ void k_sum_partials(const double *__restrict__ partials, int64_t n, double *__restrict__ out) {
    __shared__ double sx[1024];
    double x = 0.0;
    for (int64_t i = threadIdx.x; i < n; i += blockDim.x) x += partials[i];
    sx[threadIdx.x] = x;
    __syncthreads();
    for (int s = blockDim.x / 2; s > 0; s >>= 1) { if ((int)threadIdx.x < s) sx[threadIdx.x] += sx[threadIdx.x + s]; __syncthreads(); }
    if (threadIdx.x == 0) out[0] = sx[0];
}

extern "C" int nhp_disc_intensity(nhp_ctx *ctx, nhp_disc *dd, double *lam) {
    NHP_TRY(disc_ready(ctx, dd, "nhp_disc_intensity"));
    NHP_CHECK(ctx, lam != nullptr, NHP_ERR_INVALID, "nhp_disc_intensity: lam is NULL");
    const int64_t N = dd->N, T = dd->T;
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)T * N * sizeof(double), &scratch));
    NHP_TRY(nhp_timer_begin(ctx));
    launch_dmma<false>(ctx, dd, 0, T, (double *)scratch, nullptr);
    DCUDA(ctx, cudaGetLastError());
    NHP_TRY(nhp_timer_end(ctx));
    DCUDA(ctx, cudaMemcpyAsync(lam, scratch, (size_t)T * N * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DCUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

extern "C" int nhp_disc_loglik(nhp_ctx *ctx, nhp_disc *dd, double *ll) {
    NHP_TRY(disc_ready(ctx, dd, "nhp_disc_loglik"));
    NHP_CHECK(ctx, ll != nullptr, NHP_ERR_INVALID, "nhp_disc_loglik: ll is NULL");
    const int64_t N = dd->N, T = dd->T, own = T - dd->t_halo;
    const int64_t bn = 8 * pick_nt(N);
    double *partials;  // [0]: the sum; [1..]: one per CTA of launch_dmma
    NHP_TRY(nhp_partials(ctx, (own + DBM - 1) / DBM * ((N + bn - 1) / bn) + 1, &partials));
    NHP_TRY(nhp_timer_begin(ctx));
    const dim3 grid = launch_dmma<true>(ctx, dd, dd->t_halo, own, nullptr, partials + 1);
    k_sum_partials<<<1, 1024, 0, ctx->stream>>>(partials + 1, (int64_t)grid.x * grid.y, partials);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaGetLastError());
    DCUDA(ctx, cudaMemcpyAsync(ll, partials, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_TRY(nhp_timer_end(ctx));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// Gibbs parent counts (parents.jl:82-134) and VB statistics (parents.jl:136-177 + the three update!
// reductions): one CTA per (child node, slab of its non-zero bins); threads own the k = (p,b) axis.
// ---------------------------------------------------------------------------------------
constexpr int KPT = 8;  // k entries per thread: N*B <= 256 * KPT * passes (looped)

__device__ __forceinline__ double block_sum_256(double v, double *red) {
    v = warp_sum_d(v);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = v;
    __syncthreads();
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < 8; w++) s += red[w];
    return s;
}

// counts[c + N*k'] with k' = 0 baseline, 1 + k.  mu_k = convT[t,k] * bumpT[c][k], baseline mu_0 = lambda0_c dt first in the cdf order.
__global__ void __launch_bounds__(256) k_disc_gibbs(const double *__restrict__ convT, const double *__restrict__ bumpT, const double *__restrict__ lambda0, double dt,
                                                    int N, int NB, const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int64_t *__restrict__ nz_off,
                                                    const int *__restrict__ child_ptr, int slabs, const double *__restrict__ u, uint64_t seed, uint64_t counter,
                                                    double *__restrict__ counts, int *__restrict__ flag) {
    extern __shared__ double s_cum[];  // [NB + 1] inclusive cumulative weights, index 0 = baseline
    __shared__ double red[8];
    __shared__ int s_pick;
    const int c = blockIdx.x / slabs, slab = blockIdx.x % slabs;
    const int e0 = child_ptr[c], e1 = child_ptr[c + 1];
    const int per = (e1 - e0 + slabs - 1) / slabs;
    const int b0 = e0 + slab * per, b1 = min(e1, b0 + per);
    const double *bt = bumpT + (int64_t)c * NB;
    const double mu0 = lambda0[c] * dt;
    for (int e = b0; e < b1; e++) {
        const int t = nz_t[e], s = nz_s[e];
        const double *row = convT + (int64_t)t * NB;
        // block-wide inclusive scan of [mu0, mu_1..mu_NB] in index order
        double carry = mu0;
        if (threadIdx.x == 0) s_cum[0] = mu0;
        for (int k0 = 0; k0 < NB; k0 += 256) {
            int k = k0 + threadIdx.x;
            double v = k < NB ? __ldg(row + k) * __ldg(bt + k) : 0.0;
            // warp scan
            double x = v;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) { double y = __shfl_up_sync(0xffffffffu, x, d); if ((threadIdx.x & 31) >= d) x += y; }
            __syncthreads();
            if ((threadIdx.x & 31) == 31) red[threadIdx.x >> 5] = x;
            __syncthreads();
            double base = carry;
            for (int w = 0; w < (int)(threadIdx.x >> 5); w++) base += red[w];
            if (k < NB) s_cum[k + 1] = base + x;
            double tot = 0.0;
            for (int w = 0; w < 8; w++) tot += red[w];
            carry += tot;
        }
        __syncthreads();
        const double S = s_cum[NB];
        if (threadIdx.x == 0 && !(S > 0.0 && S < 1.7e308)) atomicOr(flag, 8);
        for (int d = 0; d < s; d++) {
            const int64_t ui = nz_off[e] + d;
            const double uu = u ? u[ui] : philox_uniform(seed, (uint64_t)ui, counter);
            const double target = uu * S;
            // first index with cum > target (cp <= u keeps walking); last index if none
            if (threadIdx.x == 0) s_pick = NB;
            __syncthreads();
            for (int k = threadIdx.x; k <= NB; k += 256) {
                double ck = s_cum[k], prev = k > 0 ? s_cum[k - 1] : -1.0;
                if (ck > target && !(prev > target)) atomicMin(&s_pick, k);
            }
            __syncthreads();
            if (threadIdx.x == 0) atomicAdd(&counts[c + (int64_t)N * s_pick], 1.0);
            __syncthreads();
        }
    }
}

// first index in [lo, hi) of a child's time-sorted non-zero bins with nz_t >= t (hi if none)
__device__ __forceinline__ int nz_lower_bound(const int *__restrict__ nz_t, int lo, int hi, int t) {
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if (nz_t[mid] < t) lo = mid + 1; else hi = mid;
    }
    return lo;
}

// VB: Z = e0_c + sum_k convT[t,k] ET[c][k];  alpha_sum[c] += s e0_c / Z;  gamma[c][k] += s convT[t,k] ET[c][k] / Z over the bins
// t_lo <= t < t_hi, the child's share split into `slabs` equal slabs
__global__ void __launch_bounds__(256) k_disc_vb(const double *__restrict__ convT, const double *__restrict__ ET, const double *__restrict__ e0, int N, int NB,
                                                 const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int *__restrict__ child_ptr, int slabs,
                                                 int t_lo, int t_hi, double *__restrict__ alpha_sum, double *__restrict__ gammaT /* [c][k] */) {
    __shared__ double red[8];
    const int c = blockIdx.x / slabs, slab = blockIdx.x % slabs;
    const int e0i = nz_lower_bound(nz_t, child_ptr[c], child_ptr[c + 1], t_lo), e1 = nz_lower_bound(nz_t, e0i, child_ptr[c + 1], t_hi);
    const int per = (e1 - e0i + slabs - 1) / slabs;
    const int b0 = e0i + slab * per, b1 = min(e1, b0 + per);
    const double *et = ET + (int64_t)c * NB;
    const double base = e0[c];
    double asum = 0.0;
    for (int k0 = 0; k0 < NB; k0 += 256 * KPT) {
        double acc[KPT];
#pragma unroll
        for (int m = 0; m < KPT; m++) acc[m] = 0.0;
        for (int e = b0; e < b1; e++) {
            const double *row = convT + (int64_t)nz_t[e] * NB;
            // full Z needs every k: recompute the dot product over all k each pass (passes > 1 only when N*B > 2048)
            double part = 0.0;
            for (int k = threadIdx.x; k < NB; k += 256) part += __ldg(row + k) * __ldg(et + k);
            double Z = base + block_sum_256(part, red);
            double r = (double)nz_s[e] / Z;
            if (k0 == 0) asum += r * base;
#pragma unroll
            for (int m = 0; m < KPT; m++) {
                int k = k0 + m * 256 + threadIdx.x;
                if (k < NB) acc[m] += r * __ldg(row + k) * __ldg(et + k);
            }
        }
#pragma unroll
        for (int m = 0; m < KPT; m++) {
            int k = k0 + m * 256 + threadIdx.x;
            if (k < NB && acc[m] != 0.0) atomicAdd(&gammaT[(int64_t)c * NB + k], acc[m]);
        }
    }
    if (threadIdx.x == 0 && asum != 0.0) atomicAdd(&alpha_sum[c], asum);
}

// ---------------------------------------------------------------------------------------
// warp-per-bin variants (no block barriers in the bin loop): used whenever the per-warp buffers fit shared memory
// ---------------------------------------------------------------------------------------
// Work decomposition of the warp-per-bin kernels: CTA = (time block, child).  All children of a time block are resident
// together (blockIdx.x = block * N + child), so the block's conv rows are fetched from HBM once and served from L2 to
// the other children (the earlier (child, slab) split streamed every row once per child: 63 GB of DRAM reads at
// config 3 against 9.6 GB of rows).  A child's bins are time-sorted, so its share of a block is a binary search (nz_lower_bound).

// Gibbs: the warp stores the NB weights of a bin in its shared-memory buffer, every lane sums a contiguous chunk,
// a warp scan of the chunk sums gives the cdf at chunk granularity, and the lane owning the target walks its chunk.
__global__ void __launch_bounds__(256) k_disc_gibbs_warp(const double *__restrict__ convT, const double *__restrict__ bumpT, const double *__restrict__ lambda0, double dt,
                                                         int N, int NB, const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int64_t *__restrict__ nz_off,
                                                         const int *__restrict__ child_ptr, int tb, const double *__restrict__ u, uint64_t seed, uint64_t counter,
                                                         double *__restrict__ counts, int *__restrict__ flag, const int *__restrict__ klist,
                                                         const int *__restrict__ kptr, const double *__restrict__ btc, int maxNA) {
    // klist != NULL: sparse effective weights -- only the child's structurally non-zero (parent, basis) entries are
    // gathered from the conv row (compact list klist[kptr[c] .. kptr[c+1]) ascending, values btc); zero entries can never
    // be drawn and do not move the cumulative sum, so skipping them is exact.
    extern __shared__ double s_buf[];  // [8 warps][NBP]
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int c = blockIdx.x % N, blk = blockIdx.x / N;
    const int k0 = klist ? kptr[c] : 0;
    const int NA = klist ? kptr[c + 1] - k0 : NB;           // entries of this child
    const int L = (((klist ? maxNA : NB) + 31) / 32) | 1;   // odd chunk length: conflict-free strided reads
    const int NBP = 32 * L;
    double *w = s_buf + (size_t)warp * NBP;
    const int e0 = child_ptr[c], e1 = child_ptr[c + 1];
    const int b0 = nz_lower_bound(nz_t, e0, e1, blk * tb), b1 = nz_lower_bound(nz_t, b0, e1, (blk + 1) * tb);
    if (b0 == b1) return;
    const double *bt = bumpT + (int64_t)c * NB;
    const double mu0 = lambda0[c] * dt;
    for (int e = b0 + warp; e < b1; e += 8) {
        const int t = nz_t[e], s = nz_s[e];
        const double *row = convT + (int64_t)t * NB;
        if (klist) for (int k = lane; k < NBP; k += 32) w[k] = k < NA ? __ldg(row + __ldg(klist + k0 + k)) * __ldg(btc + k0 + k) : 0.0;
        else for (int k = lane; k < NBP; k += 32) w[k] = k < NB ? __ldg(row + k) * __ldg(bt + k) : 0.0;
        __syncwarp();
        double cs = 0.0;
        const double *mine = w + lane * L;
        for (int m = 0; m < L; m++) cs += mine[m];
        double incl = cs;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) { double y = __shfl_up_sync(0xffffffffu, incl, d); if (lane >= d) incl += y; }
        incl += mu0;  // cumulative weight up to the end of this lane's chunk, baseline first
        const double S = __shfl_sync(0xffffffffu, incl, 31);
        if (lane == 0 && !(S > 0.0 && S < 1.7e308)) atomicOr(flag, 8);
        for (int d = 0; d < s; d++) {
            const int64_t ui = nz_off[e] + d;
            const double uu = u ? u[ui] : philox_uniform(seed, (uint64_t)ui, counter);
            const double target = uu * S;
            int pick;
            if (mu0 > target) pick = 0;  // first index with cumulative weight > target (cp <= u keeps walking)
            else {
                const unsigned b = __ballot_sync(0xffffffffu, incl > target);
                if (b == 0u) pick = NB;  // rounding: target >= S -> last index, as the reference's `i < n` guard
                else {
                    const int owner = __ffs(b) - 1;
                    int found = NB;
                    if (lane == owner) {
                        double cum = incl - cs;
                        for (int m = 0; m < L; m++) {
                            cum += mine[m];
                            if (cum > target) { const int q = lane * L + m; found = q < NA ? 1 + (klist ? __ldg(klist + k0 + q) : q) : NB; break; }
                        }
                        if (found > NB) found = NB;
                    }
                    pick = __shfl_sync(0xffffffffu, found, owner);
                }
            }
            if (lane == 0) atomicAdd(&counts[c + (int64_t)N * pick], 1.0);
        }
        __syncwarp();
    }
}

// VB: Z and the gamma accumulators per warp; the child's exp-expectation row is shared by the CTA.  Time block blk covers the bins
// [t_lo + blk tb, t_lo + (blk + 1) tb) of the range [t_lo, t_hi).
__global__ void __launch_bounds__(256) k_disc_vb_warp(const double *__restrict__ convT, const double *__restrict__ ET, const double *__restrict__ e0, int N, int NB,
                                                      const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int *__restrict__ child_ptr, int tb,
                                                      int t_lo, int t_hi, double *__restrict__ alpha_sum, double *__restrict__ gammaT) {
    extern __shared__ double s_buf[];  // [NB] ET row | [8][NB] per-warp accumulators
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *et = s_buf, *acc = s_buf + NB + (size_t)warp * NB;
    const int c = blockIdx.x % N, blk = blockIdx.x / N;
    const int ei0 = child_ptr[c], e1 = child_ptr[c + 1], lo = t_lo + blk * tb;
    const int b0 = nz_lower_bound(nz_t, ei0, e1, lo), b1 = nz_lower_bound(nz_t, b0, e1, min(lo + tb, t_hi));
    if (b0 == b1) return;  // block-uniform
    for (int k = threadIdx.x; k < NB; k += 256) et[k] = ET[(int64_t)c * NB + k];
    for (int k = lane; k < NB; k += 32) acc[k] = 0.0;
    __syncthreads();
    const double base = e0[c];
    double asum = 0.0;
    for (int e = b0 + warp; e < b1; e += 8) {
        const double *row = convT + (int64_t)nz_t[e] * NB;
        double part = 0.0;
        for (int k = lane; k < NB; k += 32) part += __ldg(row + k) * et[k];
        const double Z = base + warp_sum_d(part);
        const double r = (double)nz_s[e] / Z;
        asum += r * base;
        for (int k = lane; k < NB; k += 32) acc[k] += r * __ldg(row + k) * et[k];
    }
    __syncthreads();
    for (int k = threadIdx.x; k < NB; k += 256) {
        double g = 0.0;
#pragma unroll
        for (int wv = 0; wv < 8; wv++) g += s_buf[NB + (size_t)wv * NB + k];
        if (g != 0.0) atomicAdd(&gammaT[(int64_t)c * NB + k], g);
    }
    if (lane == 0 && asum != 0.0) atomicAdd(&alpha_sum[c], asum);
}

// bins per time block for the (time block, child) kernels: the rows of the ~(resident CTAs / N) blocks in flight should fit in
// about half of L2, and an item should carry enough non-zero bins to amortise its set-up
static int pick_time_block(nhp_ctx *ctx, const nhp_disc *dd, int64_t nnz) {
    const int64_t N = dd->N, NB = N * dd->B, own = dd->T - dd->t_halo;
    const double inflight = std::max(1.0, (double)ctx->sm_count * 8.0 / (double)N);
    double tb = 64e6 / ((double)NB * 8.0 * inflight);
    const double per_bin = (double)nnz / (double)std::max<int64_t>(N * own, 1);  // non-zero fraction
    tb = std::max(tb, 128.0 / std::max(per_bin, 1e-9));
    const char *env = getenv("NHP_DISC_TB");
    if (env && atoi(env) > 0) tb = atoi(env);
    return (int)std::min<double>(std::max(tb, 32.0), (double)std::max<int64_t>(dd->T, 32));
}

static int pick_slabs(nhp_ctx *ctx, int64_t N, int64_t nnz) {
    int64_t want = (int64_t)ctx->sm_count * 8;
    int64_t slabs = std::max<int64_t>(1, want / std::max<int64_t>(N, 1));
    slabs = std::min<int64_t>(slabs, std::max<int64_t>(1, nnz / std::max<int64_t>(N, 1) / 4));
    return (int)std::max<int64_t>(1, slabs);
}

extern "C" int nhp_disc_gibbs_counts(nhp_ctx *ctx, nhp_disc *dd, uint64_t seed, uint64_t counter, const double *u, int64_t nu, double *counts) {
    NHP_TRY(disc_ready(ctx, dd, "nhp_disc_gibbs_counts"));
    NHP_CHECK(ctx, !u || nu >= dd->total_events, NHP_ERR_INVALID, "nhp_disc_gibbs_counts: need %lld uniforms, got %lld", (long long)dd->total_events, (long long)nu);
    DiscExtra *ex = extra_of(dd);
    const int64_t N = dd->N, NB = N * dd->B, NK = 1 + NB;
    cudaStream_t s = ctx->stream;
    void *scratch;
    size_t bytes_c = (size_t)(N * NK) * sizeof(double), bytes_u = u ? (size_t)dd->total_events * sizeof(double) : 0;
    NHP_TRY(nhp_scratch(ctx, bytes_c + bytes_u + 16, &scratch));
    double *d_counts = (double *)scratch, *d_u = u ? d_counts + N * NK : nullptr;
    DCUDA(ctx, cudaMemsetAsync(d_counts, 0, bytes_c, s));
    DCUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
    if (u && dd->total_events > 0) DCUDA(ctx, cudaMemcpyAsync(d_u, u, bytes_u, cudaMemcpyHostToDevice, s));
    NHP_TRY(nhp_timer_begin(ctx));
    if (ex->nnz > 0) {
        int slabs = pick_slabs(ctx, N, ex->nnz);
        const char *envs = getenv("NHP_DISC_SPARSE");
        const bool sparse = ctx->dd_lists && ctx->dd_density <= 0.5 && !(envs && atoi(envs) == 0);
        const int64_t wid = sparse ? ctx->dd_maxNA : NB;
        const size_t wsmem = (size_t)8 * 32 * (((wid + 31) / 32) | 1) * sizeof(double);
        const char *envw = getenv("NHP_DISC_WARP");
        if (wsmem <= (size_t)ctx->smem_optin - 4096 && !(envw && atoi(envw) == 0)) {
            DCUDA(ctx, cudaFuncSetAttribute(k_disc_gibbs_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
            const int tb = pick_time_block(ctx, dd, ex->nnz);
            const int64_t nblk = (dd->T + tb - 1) / tb;
            k_disc_gibbs_warp<<<(unsigned)(N * nblk), 256, wsmem, s>>>(dd->d_conv, ctx->dd_bump + NB * N, ctx->dd_lambda0, ctx->ddt, (int)N, (int)NB, ex->nz_t, ex->nz_s,
                                                                        ex->nz_off, ex->child_ptr, tb, d_u, seed, counter, d_counts, ctx->d_flag,
                                                                        sparse ? ctx->dd_klist : nullptr, ctx->dd_kptr, ctx->dd_btc, (int)ctx->dd_maxNA);
        } else {
        size_t smem = (size_t)(NB + 1) * sizeof(double);
        DCUDA(ctx, cudaFuncSetAttribute(k_disc_gibbs, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k_disc_gibbs<<<(unsigned)(N * slabs), 256, smem, s>>>(dd->d_conv, ctx->dd_bump + NB * N, ctx->dd_lambda0, ctx->ddt, (int)N, (int)NB, ex->nz_t, ex->nz_s, ex->nz_off,
                                                               ex->child_ptr, slabs, d_u, seed, counter, d_counts, ctx->d_flag);
        }
        NHP_LAUNCHED(ctx);
        DCUDA(ctx, cudaGetLastError());
    }
    int flag = 0;
    DCUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    NHP_TRY(nhp_timer_end(ctx));
    NHP_CHECK(ctx, !(flag & 8), NHP_ERR_NUMERIC, "resample_parents (discrete): invalid Multinomial probability vector (parents.jl:116)");
    // the counts stay on the device for nhp_disc_resample_params (device-side conjugate draws); the host copy is optional
    if (ctx->dd_counts_cap < (size_t)(N * NK)) {
        DCUDA(ctx, cudaStreamSynchronize(s));
        cudaFree(ctx->dd_counts); ctx->dd_counts = nullptr; ctx->dd_counts_cap = 0;
        DCUDA(ctx, cudaMalloc(&ctx->dd_counts, bytes_c));
        ctx->dd_counts_cap = (size_t)(N * NK);
    }
    DCUDA(ctx, cudaMemcpyAsync(ctx->dd_counts, d_counts, bytes_c, cudaMemcpyDeviceToDevice, s));
    ctx->dd_counts_N = N; ctx->dd_counts_B = dd->B;
    if (counts) DCUDA(ctx, cudaMemcpyAsync(counts, d_counts, bytes_c, cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// ET[c][k] = E[p + N*(c + N*b)]
__global__ void k_transpose_E(const double *__restrict__ E, int N, int B, double *__restrict__ ET) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t NB = (int64_t)N * B;
    if (e >= NB * N) return;
    int c = (int)(e / NB), k = (int)(e % NB), p = k / B, b = k - p * B;
    ET[e] = E[p + (int64_t)N * (c + (int64_t)N * b)];
}
// kappa_sum[p,c] = sum_b gamma[p,c,b]; gamma_sum[p + N*(c + N*b)] = gammaT[c][p*B+b]; nu_sum[p,c] = rowsum[p]
__global__ void k_vb_finish(const double *__restrict__ gammaT, const double *__restrict__ rowsum, int N, int B, double *__restrict__ kappa, double *__restrict__ nu,
                            double *__restrict__ gamma) {
    int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= (int64_t)N * N) return;
    int c = (int)(e / N), p = (int)(e % N);
    double ks = 0.0;
    for (int b = 0; b < B; b++) {
        double g = gammaT[(int64_t)c * N * B + p * B + b];
        ks += g;
        gamma[p + (int64_t)N * (c + (int64_t)N * b)] = g;
    }
    kappa[p + (int64_t)N * c] = ks;
    nu[p + (int64_t)N * c] = rowsum[p];
}

// responsibilities + reductions of one VB step over the bins t_lo <= t < t_hi into zeroed alpha_sum[N] and gammaT[c][p*B+b] (the
// sums accumulate, so a range split in two is two calls): the warp-per-bin kernel when its buffers fit shared memory (and
// NHP_DISC_WARP is not 0), the block kernel otherwise; nothing to do without non-zero bins.  A range shorter than the series takes
// time blocks short enough that its CTAs fill the SMs once, and the slabs of the share of non-zero bins it expects, so the cost of
// a window scales with the window.
int nhp_disc_vb_reduce(nhp_ctx *ctx, nhp_disc *dd, int64_t t_lo, int64_t t_hi, const double *e0, const double *ET, double *alpha_sum, double *gammaT) {
    DiscExtra *ex = extra_of(dd);
    const int64_t n = t_hi - t_lo;
    if (ex->nnz == 0 || n <= 0) return NHP_OK;
    const int64_t N = dd->N, NB = N * dd->B;
    const bool window = n < dd->T;
    cudaStream_t s = ctx->stream;
    const size_t wsmem = (size_t)9 * NB * sizeof(double);
    const char *envw = getenv("NHP_DISC_WARP");
    if (wsmem <= (size_t)ctx->smem_optin - 4096 && !(envw && atoi(envw) == 0)) {
        DCUDA(ctx, cudaFuncSetAttribute(k_disc_vb_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        int tb = pick_time_block(ctx, dd, ex->nnz);
        if (window) {
            int per_sm = 1;
            DCUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_disc_vb_warp, 256, wsmem));
            const int64_t want = ((int64_t)ctx->sm_count * std::max(per_sm, 1) + N - 1) / N;  // time blocks of one full wave
            tb = (int)std::min<int64_t>(tb, std::max<int64_t>(32, (n + want - 1) / want));
        }
        const int64_t nblk = (n + tb - 1) / tb;
        k_disc_vb_warp<<<(unsigned)(N * nblk), 256, wsmem, s>>>(dd->d_conv, ET, e0, (int)N, (int)NB, ex->nz_t, ex->nz_s, ex->child_ptr, tb, (int)t_lo, (int)t_hi,
                                                                 alpha_sum, gammaT);
    } else {
        const int slabs = pick_slabs(ctx, N, window ? ex->nnz * n / dd->T : ex->nnz);
        k_disc_vb<<<(unsigned)(N * slabs), 256, 0, s>>>(dd->d_conv, ET, e0, (int)N, (int)NB, ex->nz_t, ex->nz_s, ex->child_ptr, slabs, (int)t_lo, (int)t_hi,
                                                        alpha_sum, gammaT);
    }
    NHP_LAUNCHED(ctx);
    return NHP_OK;
}

// events[p] += sum of data[p, t] over t_lo <= t < t_hi: one warp per node, a binary search into its time-sorted non-zero bins and a sum
// of their counts
__global__ void __launch_bounds__(256) k_disc_range_events(const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int *__restrict__ child_ptr, int N,
                                                           int t_lo, int t_hi, double *__restrict__ events) {
    const int p = (int)(((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
    if (p >= N) return;  // warp-uniform
    const int b0 = nz_lower_bound(nz_t, child_ptr[p], child_ptr[p + 1], t_lo), b1 = nz_lower_bound(nz_t, b0, child_ptr[p + 1], t_hi);
    long long sum = 0;
    for (int e = b0 + lane; e < b1; e += 32) sum += nz_s[e];
#pragma unroll
    for (int d = 16; d >= 1; d >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, d);
    if (lane == 0) events[p] += (double)sum;
}

int nhp_disc_range_events(nhp_ctx *ctx, nhp_disc *dd, int64_t t_lo, int64_t t_hi, double *events) {
    DiscExtra *ex = extra_of(dd);
    if (ex->nnz == 0 || t_hi <= t_lo) return NHP_OK;
    k_disc_range_events<<<(unsigned)((dd->N + 7) / 8), 256, 0, ctx->stream>>>(ex->nz_t, ex->nz_s, ex->child_ptr, (int)dd->N, (int)t_lo, (int)t_hi, events);
    NHP_LAUNCHED(ctx);
    return NHP_OK;
}

extern "C" int nhp_disc_vb_stats(nhp_ctx *ctx, nhp_disc *dd, const double *e0, const double *E, double *alpha_sum, double *kappa_sum, double *nu_sum,
                                 double *gamma_sum) {
    NHP_CHECK(ctx, ctx != nullptr, NHP_ERR_INVALID, "ctx is NULL");
    NHP_CHECK(ctx, dd && dd->d_conv, NHP_ERR_STATE, "nhp_disc_vb_stats: call nhp_disc_convolve first");
    NHP_CHECK(ctx, e0 && E && alpha_sum && kappa_sum && nu_sum && gamma_sum, NHP_ERR_INVALID, "nhp_disc_vb_stats: NULL argument");
    DCUDA(ctx, cudaSetDevice(ctx->device));
    DiscExtra *ex = extra_of(dd);
    const int64_t N = dd->N, B = dd->B, NB = N * B;
    cudaStream_t s = ctx->stream;
    void *scratch;
    // layout: e0[N] | E[N*N*B] | ET[N*NB] | gammaT[N*NB] | alpha[N] | kappa[N*N] | nu[N*N] | gamma[N*N*B]
    size_t tot = (size_t)(N + NB * N * 4 + N + 2 * N * N) * sizeof(double);
    NHP_TRY(nhp_scratch(ctx, tot, &scratch));
    double *d_e0 = (double *)scratch, *d_E = d_e0 + N, *d_ET = d_E + NB * N, *d_gT = d_ET + NB * N, *d_alpha = d_gT + NB * N, *d_kappa = d_alpha + N,
           *d_nu = d_kappa + N * N, *d_gamma = d_nu + N * N;
    DCUDA(ctx, cudaMemcpyAsync(d_e0, e0, (size_t)N * sizeof(double), cudaMemcpyHostToDevice, s));
    DCUDA(ctx, cudaMemcpyAsync(d_E, E, (size_t)(NB * N) * sizeof(double), cudaMemcpyHostToDevice, s));
    DCUDA(ctx, cudaMemsetAsync(d_gT, 0, (size_t)(NB * N + N) * sizeof(double), s));
    unsigned eb = (unsigned)((NB * N + 255) / 256);
    k_transpose_E<<<eb, 256, 0, s>>>(d_E, (int)N, (int)B, d_ET);
    NHP_LAUNCHED(ctx);
    NHP_TRY(nhp_timer_begin(ctx));
    NHP_TRY(nhp_disc_vb_reduce(ctx, dd, 0, dd->T, d_e0, d_ET, d_alpha, d_gT));
    k_vb_finish<<<(unsigned)((N * N + 255) / 256), 256, 0, s>>>(d_gT, ex->rowsum, (int)N, (int)B, d_kappa, d_nu, d_gamma);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaGetLastError());
    NHP_TRY(nhp_timer_end(ctx));
    DCUDA(ctx, cudaMemcpyAsync(alpha_sum, d_alpha, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaMemcpyAsync(kappa_sum, d_kappa, (size_t)(N * N) * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaMemcpyAsync(nu_sum, d_nu, (size_t)(N * N) * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaMemcpyAsync(gamma_sum, d_gamma, (size_t)(NB * N) * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// Analytic gradient of the discrete log-likelihood for `mle!` (discrete.jl:211-296; the reference hands Optim a gradient-free
// objective, its comments at :220-231 sketch the gradient form).  With r[t,c] = s[t,c] / lambda[t,c] - 1:
//   d ll / d lambda0[c]   = dt sum_t r[t,c]
//   d ll / d bump[k,c]    = sum_t conv[t,k] r[t,c] = Gs[k,c] - csum[k],   Gs[k,c] = sum over the NON-ZERO bins of conv[t,k] s / lambda
//   d ll / d W[p,c]       = [A] dt sum_b theta[p,c,b] (Gs - csum)[(p,b),c];    d ll / d theta[p,c,b] = [A] W[p,c] dt (Gs - csum)[(p,b),c]
// so the T x N x (N B) contraction collapses to the non-zero bins (4 % of the cells at config 3) plus the conv column sums that the
// convolution already left behind: the same (time block, child) warp-per-bin pass as the VB statistics.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_disc_grad_warp(const double *__restrict__ convT, const double *__restrict__ bumpT, const double *__restrict__ lambda0, double dt,
                                                        int N, int NB, const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int *__restrict__ child_ptr, int tb,
                                                        double *__restrict__ rsum, double *__restrict__ GsT) {
    extern __shared__ double s_buf[];  // [NB] bump column of the child | [8][NB] per-warp accumulators
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double *bt = s_buf, *acc = s_buf + NB + (size_t)warp * NB;
    const int c = blockIdx.x % N, blk = blockIdx.x / N;
    const int ei0 = child_ptr[c], e1 = child_ptr[c + 1];
    const int b0 = nz_lower_bound(nz_t, ei0, e1, blk * tb), b1 = nz_lower_bound(nz_t, b0, e1, (blk + 1) * tb);
    if (b0 == b1) return;  // block-uniform
    for (int k = threadIdx.x; k < NB; k += 256) bt[k] = bumpT[(int64_t)c * NB + k];
    for (int k = lane; k < NB; k += 32) acc[k] = 0.0;
    __syncthreads();
    const double base = lambda0[c] * dt;
    double asum = 0.0;
    for (int e = b0 + warp; e < b1; e += 8) {
        const double *row = convT + (int64_t)nz_t[e] * NB;
        double part = 0.0;
        for (int k = lane; k < NB; k += 32) part += __ldg(row + k) * bt[k];
        const double r = (double)nz_s[e] / (base + warp_sum_d(part));  // s / lambda[t,c]
        asum += r;
        for (int k = lane; k < NB; k += 32) acc[k] += r * __ldg(row + k);
    }
    __syncthreads();
    for (int k = threadIdx.x; k < NB; k += 256) {
        double g = 0.0;
#pragma unroll
        for (int wv = 0; wv < 8; wv++) g += s_buf[NB + (size_t)wv * NB + k];
        if (g != 0.0) atomicAdd(&GsT[(int64_t)c * NB + k], g);
    }
    if (lane == 0 && asum != 0.0) atomicAdd(&rsum[c], asum);
}
// one thread per (p, c): chain rule from the bump gradient to W and theta; thread c < N also finishes d/d lambda0
__global__ void k_disc_grad_finish(const double *__restrict__ GsT, const double *__restrict__ csum, const double *__restrict__ rsum, const double *__restrict__ W,
                                   const double *__restrict__ A, const double *__restrict__ theta, double dt, double own_bins, int N, int B,
                                   double *__restrict__ dl0, double *__restrict__ dW, double *__restrict__ dth) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x, NN = (int64_t)N * N;
    if (e < N) dl0[e] = dt * (rsum[e] - own_bins);
    if (e >= NN) return;
    const int p = (int)(e % N), c = (int)(e / N);  // e = p + N c
    const double a = A ? A[e] : 1.0, w = W[e];
    double s = 0.0;
    for (int b = 0; b < B; b++) {
        const double g = GsT[(int64_t)c * N * B + p * B + b] - csum[p * B + b];
        s += theta[e + NN * b] * g;
        dth[e + NN * b] = a * w * dt * g;
    }
    dW[e] = a * dt * s;
}

extern "C" int nhp_disc_loglik_grad(nhp_ctx *ctx, nhp_disc *dd, double *ll, double *dlambda0, double *dW, double *dtheta) {
    NHP_TRY(disc_ready(ctx, dd, "nhp_disc_loglik_grad"));
    NHP_CHECK(ctx, dlambda0 && dW && dtheta, NHP_ERR_INVALID, "nhp_disc_loglik_grad: NULL output");
    if (ll) NHP_TRY(nhp_disc_loglik(ctx, dd, ll));
    const double ms_ll = ll ? ctx->last_ms : 0.0;
    DiscExtra *ex = extra_of(dd);
    const int64_t N = dd->N, B = dd->B, NB = N * B, NN = N * N;
    cudaStream_t s = ctx->stream;
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)(NB * N + N + N + NN + NN * B) * sizeof(double), &scratch));
    double *d_Gs = (double *)scratch, *d_rs = d_Gs + NB * N, *d_l0 = d_rs + N, *d_dW = d_l0 + N, *d_dth = d_dW + NN;
    DCUDA(ctx, cudaMemsetAsync(d_Gs, 0, (size_t)(NB * N + N) * sizeof(double), s));
    NHP_TRY(nhp_timer_begin(ctx));
    if (ex->nnz > 0) {
        const size_t wsmem = (size_t)9 * NB * sizeof(double);
        NHP_CHECK(ctx, wsmem <= (size_t)ctx->smem_optin - 4096, NHP_ERR_UNSUPPORTED, "nhp_disc_loglik_grad: N B = %lld exceeds the shared-memory accumulators", (long long)NB);
        DCUDA(ctx, cudaFuncSetAttribute(k_disc_grad_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)wsmem));
        const int tb = pick_time_block(ctx, dd, ex->nnz);
        const int64_t nblk = (dd->T + tb - 1) / tb;
        k_disc_grad_warp<<<(unsigned)(N * nblk), 256, wsmem, s>>>(dd->d_conv, ctx->dd_bump + NB * N, ctx->dd_lambda0, ctx->ddt, (int)N, (int)NB, ex->nz_t, ex->nz_s, ex->child_ptr,
                                                                  tb, d_rs, d_Gs);
        NHP_LAUNCHED(ctx);
    }
    k_disc_grad_finish<<<(unsigned)((NN + 255) / 256), 256, 0, s>>>(d_Gs, ex->csum, d_rs, ctx->dd_W, ctx->d_has_A ? ctx->dd_A : nullptr, ctx->dd_theta, ctx->ddt,
                                                                    (double)(dd->T - dd->t_halo), (int)N, (int)B, d_l0, d_dW, d_dth);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaGetLastError());
    NHP_TRY(nhp_timer_end(ctx));
    ctx->last_ms += ms_ll;
    DCUDA(ctx, cudaMemcpyAsync(dlambda0, d_l0, (size_t)N * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaMemcpyAsync(dW, d_dW, (size_t)NN * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaMemcpyAsync(dtheta, d_dth, (size_t)(NN * B) * sizeof(double), cudaMemcpyDeviceToHost, s));
    DCUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// ---------------------------------------------------------------------------------------
// discrete adjacency Gibbs (discrete.jl:426-480): per column c, p sequential.
//   ll1 - ll0 = sum_{t: s>0} s [log(lam^{-p} + G_p) - log(lam^{-p})] - sum_t G_p[t] + log rho - log(1-rho),
//   G_p[t] = sum_b convT[t,(p,b)] W[p,c] theta[p,c,b] dt.   One CTA per column; the rank-1 update of the
//   column's intensities touches only its non-zero bins; sum_t G_p[t] comes from the conv column sums.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_disc_adjacency(const double *__restrict__ convT, const double *__restrict__ csum, const double *__restrict__ lambda0,
                                                        const double *__restrict__ W, const double *__restrict__ theta, double dt, double *__restrict__ A,
                                                        const double *__restrict__ rho, double rho_s, const double *__restrict__ u, uint64_t seed, uint64_t counter,
                                                        int N, int B, const int *__restrict__ nz_t, const int *__restrict__ nz_s, const int *__restrict__ child_ptr,
                                                        double *__restrict__ lam_scratch, int *__restrict__ flag) {
    __shared__ double red[8];
    __shared__ double s_anew;
    const int c = blockIdx.x;
    const int NB = N * B;
    const int e0 = child_ptr[c], e1 = child_ptr[c + 1];
    double *lam = lam_scratch + e0;
    // current intensities at the column's non-zero bins
    for (int e = e0 + threadIdx.x; e < e1; e += 256) {
        const double *row = convT + (int64_t)nz_t[e] * NB;
        double v = lambda0[c] * dt;
        for (int p = 0; p < N; p++) {
            double a = A[p + (int64_t)N * c], w = W[p + (int64_t)N * c];
            if (a != 0.0)
                for (int b = 0; b < B; b++) v += row[p * B + b] * a * w * theta[p + (int64_t)N * (c + (int64_t)N * b)] * dt;
        }
        lam[e - e0] = v;
    }
    __syncthreads();
    for (int p = 0; p < N; p++) {
        const int64_t kk = p + (int64_t)N * c;
        const double a_old = A[kk], w = W[kk];
        double gsum = 0.0;  // sum over all own bins of G_p
        for (int b = 0; b < B; b++) gsum += csum[p * B + b] * w * theta[kk + (int64_t)N * N * b] * dt;
        double part = 0.0;
        for (int e = e0 + threadIdx.x; e < e1; e += 256) {
            const double *row = convT + (int64_t)nz_t[e] * NB + p * B;
            double g = 0.0;
            for (int b = 0; b < B; b++) g += row[b] * w * theta[kk + (int64_t)N * N * b] * dt;
            if (g != 0.0) {
                double l = lam[e - e0];
                double base = a_old != 0.0 ? l - g : l;
                part += (double)nz_s[e] * log((base + g) / base);
            }
        }
        double sum = block_sum_256(part, red);
        if (threadIdx.x == 0) {
            double r = rho ? rho[kk] : rho_s;
            double delta = sum - gsum + (log(r) - log(1.0 - r));
            double p1 = delta >= 0.0 ? 1.0 / (1.0 + exp(-delta)) : exp(delta) / (1.0 + exp(delta));
            if (delta != delta) { atomicOr(flag, 64); p1 = 0.0; }
            double uu = u ? u[kk] : philox_uniform(seed, (uint64_t)kk, counter);
            double an = uu <= p1 ? 1.0 : 0.0;
            A[kk] = an;
            s_anew = an;
        }
        __syncthreads();
        const double an = s_anew;
        if (an != a_old) {
            for (int e = e0 + threadIdx.x; e < e1; e += 256) {
                const double *row = convT + (int64_t)nz_t[e] * NB + p * B;
                double g = 0.0;
                for (int b = 0; b < B; b++) g += row[b] * w * theta[kk + (int64_t)N * N * b] * dt;
                lam[e - e0] += an != 0.0 ? g : -g;
            }
        }
        __syncthreads();
    }
}

// Streaming variant (default when the scratch fits): the candidate contributions G_p[e] = sum_b conv[t_e,(p,b)] W theta dt do not
// depend on the decisions, so they are computed for ALL (bin, parent) pairs first, by the whole GPU:
//   phase A (k_disc_adj_gather): CTA = 32 consecutive non-zero bins of a child; a warp takes a bin and its lanes take consecutive
//     parents, so the warp reads the bin's conv row as one contiguous stream (full DRAM bursts); the 32 x N tile is transposed
//     through shared memory and written parent-major (G[p][e], 256-byte runs); the bins' current intensities fall out of the same pass.
//   phase B (k_disc_adj_steps): one CTA per column runs the N sequential Bernoulli steps on coalesced reads of one G row each.
// HBM traffic per sweep: rows once (nnz * N * B * 8 B) + G written and read once (nnz * N * 8 B each), against one scattered
// 32-byte sector per (bin, parent) per pass in k_disc_adjacency (ncu at config 3: 290 GB, 17 % of the warps active).
constexpr int ADJ_TE = 32;  // bins per phase-A tile

__global__ void __launch_bounds__(256) k_disc_adj_gather(const double *__restrict__ convT, const double *__restrict__ lambda0, const double *__restrict__ W,
                                                         const double *__restrict__ theta, double dt, const double *__restrict__ A, int N, int B,
                                                         const int *__restrict__ nz_t, const int *__restrict__ child_ptr, double *__restrict__ lam_scratch,
                                                         double *__restrict__ g_scratch) {
    extern __shared__ double s_dynd[];  // [N*B] coefficients | [N][ADJ_TE + 1] tile
    // children vary fastest over the grid: the CTAs that are resident together work on the same stretch of time for different
    // children, so a conv row comes from HBM once and from L2 for the other children with a count in that bin (with the children on
    // the slow axis every non-zero (bin, child) re-read its 8 N B-byte row from DRAM: 75 GB for 9.6 GB of rows at config 3)
    const int c = blockIdx.x;
    const int NB = N * B;
    const int e0 = child_ptr[c], ne = child_ptr[c + 1] - e0;
    const int t0 = blockIdx.y * ADJ_TE;
    if (t0 >= ne) return;
    double *s_coef = s_dynd, *tile = s_dynd + NB;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int k = threadIdx.x; k < NB; k += 256) {
        const int p = k / B, b = k % B;
        s_coef[k] = W[p + (int64_t)N * c] * theta[p + (int64_t)N * (c + (int64_t)N * b)] * dt;
    }
    __syncthreads();
    const int nt = min(ADJ_TE, ne - t0);
    for (int el = warp; el < nt; el += 8) {
        const double *row = convT + (int64_t)nz_t[e0 + t0 + el] * NB;
        double v = 0.0;
        for (int p = lane; p < N; p += 32) {
            double g = 0.0;
            for (int b = 0; b < B; b++) g += __ldg(row + p * B + b) * s_coef[p * B + b];
            tile[p * (ADJ_TE + 1) + el] = g;
            if (A[p + (int64_t)N * c] != 0.0) v += g;
        }
        v = warp_sum_d(v);
        if (lane == 0) lam_scratch[e0 + t0 + el] = lambda0[c] * dt + v;
    }
    __syncthreads();
    double *G = g_scratch + (int64_t)e0 * N;  // [N][ne]
    for (int k = threadIdx.x; k < N * ADJ_TE; k += 256) {
        const int p = k / ADJ_TE, el = k % ADJ_TE;
        if (el < nt) G[(int64_t)p * ne + t0 + el] = tile[p * (ADJ_TE + 1) + el];
    }
}

__global__ void __launch_bounds__(1024) k_disc_adj_steps(const double *__restrict__ csum, const double *__restrict__ W, const double *__restrict__ theta, double dt,
                                                         double *__restrict__ A, const double *__restrict__ rho, double rho_s, const double *__restrict__ u,
                                                         uint64_t seed, uint64_t counter, int N, int B, const int *__restrict__ nz_s, const int *__restrict__ child_ptr,
                                                         double *__restrict__ lam_scratch, const double *__restrict__ g_scratch, int *__restrict__ flag) {
    __shared__ double red[32];
    __shared__ double s_anew;
    const int c = blockIdx.x;
    const int e0 = child_ptr[c], e1 = child_ptr[c + 1], ne = e1 - e0;
    double *lam = lam_scratch + e0;
    const double *G = g_scratch + (int64_t)e0 * N;
    for (int p = 0; p < N; p++) {
        const int64_t kk = p + (int64_t)N * c;
        const double a_old = A[kk], w = W[kk];
        double gsum = 0.0;  // sum over all own bins of G_p
        for (int b = 0; b < B; b++) gsum += csum[p * B + b] * (w * theta[kk + (int64_t)N * N * b] * dt);
        const double *Gp = G + (int64_t)p * ne;
        double part = 0.0;
        for (int e = threadIdx.x; e < ne; e += blockDim.x) {
            const double g = Gp[e];
            if (g != 0.0) {
                const double l = lam[e];
                const double base = a_old != 0.0 ? l - g : l;
                part += (double)nz_s[e0 + e] * log((base + g) / base);
            }
        }
        part = warp_sum_d(part);
        if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = part;
        __syncthreads();
        if (threadIdx.x == 0) {
            double sum = 0.0;
            for (int wv = 0; wv < (int)(blockDim.x >> 5); wv++) sum += red[wv];
            const double r = rho ? rho[kk] : rho_s;
            const double delta = sum - gsum + (log(r) - log(1.0 - r));
            double p1 = delta >= 0.0 ? 1.0 / (1.0 + exp(-delta)) : exp(delta) / (1.0 + exp(delta));
            if (delta != delta) { atomicOr(flag, 64); p1 = 0.0; }
            const double uu = u ? u[kk] : philox_uniform(seed, (uint64_t)kk, counter);
            const double an = uu <= p1 ? 1.0 : 0.0;
            A[kk] = an;
            s_anew = an;
        }
        __syncthreads();
        const double an = s_anew;
        if (an != a_old) {
            for (int e = threadIdx.x; e < ne; e += blockDim.x) lam[e] += an != 0.0 ? Gp[e] : -Gp[e];
        }
        __syncthreads();
    }
}

// The sweep over every column of the device matrix A (in place).  rho: per-entry link probabilities [N*N], or NULL for the scalar
// rho_s; u: uniforms [N*N] or NULL for Philox (seed, p + N c, counter).  The streaming form needs G[p][e] for every (parent, non-zero
// bin) next to the bins' intensities in the work buffer: adj_work_doubles tells the caller how much to reserve.
static bool adj_streaming(nhp_ctx *ctx, const nhp_disc *dd, size_t *work_doubles) {
    const int64_t N = dd->N, B = dd->B, nnz1 = std::max<int64_t>(extra_of(const_cast<nhp_disc *>(dd))->nnz, 1);
    const size_t g_bytes = (size_t)nnz1 * (size_t)N * sizeof(double), coef_smem = (size_t)(N * B + N * (ADJ_TE + 1)) * sizeof(double);
    size_t free_b = 0, total_b = 0;
    cudaMemGetInfo(&free_b, &total_b);
    const char *envt = getenv("NHP_DISC_ADJ_STREAM");
    const bool stream_variant = !(envt && atoi(envt) == 0) && coef_smem <= (size_t)ctx->smem_optin - 4096 && g_bytes <= free_b / 2 + ctx->scratch_cap;
    *work_doubles = (size_t)nnz1 + (stream_variant ? (size_t)nnz1 * (size_t)N : 0);
    return stream_variant;
}
static int adj_sweep(nhp_ctx *ctx, nhp_disc *dd, bool stream_variant, double *d_A, const double *d_rho, double rho_s, const double *d_u, uint64_t seed,
                     uint64_t counter, double *work) {
    DiscExtra *ex = extra_of(dd);
    const int64_t N = dd->N, B = dd->B, nnz1 = std::max<int64_t>(ex->nnz, 1);
    cudaStream_t s = ctx->stream;
    double *d_lam = work, *d_G = work + nnz1;
    DCUDA(ctx, cudaMemsetAsync(ctx->d_flag, 0, sizeof(int), s));
    NHP_TRY(nhp_timer_begin(ctx));
    if (stream_variant) {
        if (ex->max_ne > 0) {
            const size_t coef_smem = (size_t)(N * B + N * (ADJ_TE + 1)) * sizeof(double);
            DCUDA(ctx, cudaFuncSetAttribute(k_disc_adj_gather, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)coef_smem));
            dim3 gg((unsigned)N, (unsigned)((ex->max_ne + ADJ_TE - 1) / ADJ_TE));
            k_disc_adj_gather<<<gg, 256, coef_smem, s>>>(dd->d_conv, ctx->dd_lambda0, ctx->dd_W, ctx->dd_theta, ctx->ddt, d_A, (int)N, (int)B, ex->nz_t, ex->child_ptr, d_lam, d_G);
            NHP_LAUNCHED(ctx);
        }
        k_disc_adj_steps<<<(unsigned)N, 1024, 0, s>>>(ex->csum, ctx->dd_W, ctx->dd_theta, ctx->ddt, d_A, d_rho, rho_s, d_u, seed, counter, (int)N, (int)B, ex->nz_s,
                                                       ex->child_ptr, d_lam, d_G, ctx->d_flag);
    } else
    k_disc_adjacency<<<(unsigned)N, 256, 0, s>>>(dd->d_conv, ex->csum, ctx->dd_lambda0, ctx->dd_W, ctx->dd_theta, ctx->ddt, d_A, d_rho, rho_s, d_u, seed, counter,
                                                 (int)N, (int)B, ex->nz_t, ex->nz_s, ex->child_ptr, d_lam, ctx->d_flag);
    NHP_LAUNCHED(ctx);
    DCUDA(ctx, cudaGetLastError());
    int flag = 0;
    DCUDA(ctx, cudaMemcpyAsync(&flag, ctx->d_flag, sizeof(int), cudaMemcpyDeviceToHost, s));
    NHP_TRY(nhp_timer_end(ctx));
    NHP_CHECK(ctx, !(flag & 64), NHP_ERR_NUMERIC, "discrete adjacency sampler: NaN log-likelihood difference");
    return NHP_OK;
}

extern "C" int nhp_disc_resample_adjacency(nhp_ctx *ctx, nhp_disc *dd, const double *rho, uint64_t seed, uint64_t counter, const double *u, double *A_inout) {
    NHP_TRY(disc_ready(ctx, dd, "nhp_disc_resample_adjacency"));
    NHP_CHECK(ctx, rho && A_inout, NHP_ERR_INVALID, "nhp_disc_resample_adjacency: NULL rho/A");
    NHP_CHECK(ctx, dd->t_halo == 0, NHP_ERR_UNSUPPORTED, "nhp_disc_resample_adjacency works on unsharded data");
    const int64_t NN = dd->N * dd->N;
    cudaStream_t s = ctx->stream;
    size_t work = 0;
    const bool stream_variant = adj_streaming(ctx, dd, &work);
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, (size_t)(3 * NN) * sizeof(double) + work * sizeof(double), &scratch));
    double *d_A = (double *)scratch, *d_rho = d_A + NN, *d_u = d_rho + NN, *d_work = d_u + NN;
    DCUDA(ctx, cudaMemcpyAsync(d_A, A_inout, (size_t)NN * sizeof(double), cudaMemcpyHostToDevice, s));
    DCUDA(ctx, cudaMemcpyAsync(d_rho, rho, (size_t)NN * sizeof(double), cudaMemcpyHostToDevice, s));
    if (u) DCUDA(ctx, cudaMemcpyAsync(d_u, u, (size_t)NN * sizeof(double), cudaMemcpyHostToDevice, s));
    NHP_TRY(adj_sweep(ctx, dd, stream_variant, d_A, d_rho, 0.0, u ? d_u : nullptr, seed, counter, d_work));
    DCUDA(ctx, cudaMemcpyAsync(A_inout, d_A, (size_t)NN * sizeof(double), cudaMemcpyDeviceToHost, s));
    // the new adjacency becomes the context's A, and the derived tables (bump, compact parent lists) follow it
    if (ctx->d_has_A) {
        DCUDA(ctx, cudaMemcpyAsync(ctx->dd_A, d_A, (size_t)NN * sizeof(double), cudaMemcpyDeviceToDevice, s));
        NHP_TRY(nhp_disc_tables_refresh(ctx));
    }
    DCUDA(ctx, cudaStreamSynchronize(s));
    return NHP_OK;
}

// resample_adjacency_matrix! (discrete.jl:426-460) in place on the context's adjacency matrix, with a scalar link probability
extern "C" int nhp_disc_resample_adjacency_dev(nhp_ctx *ctx, nhp_disc *dd, double rho, uint64_t seed, uint64_t counter) {
    NHP_TRY(disc_ready(ctx, dd, "nhp_disc_resample_adjacency_dev"));
    NHP_CHECK(ctx, dd->t_halo == 0, NHP_ERR_UNSUPPORTED, "nhp_disc_resample_adjacency_dev works on unsharded data");
    NHP_CHECK(ctx, ctx->d_has_A, NHP_ERR_STATE, "nhp_disc_resample_adjacency_dev: the process has no adjacency matrix");
    if (rho < 0.0) {
        NHP_CHECK(ctx, ctx->dd_rho >= 0.0, NHP_ERR_STATE, "nhp_disc_resample_adjacency_dev: no link probability kept with the context (nhp_disc_network_set)");
        rho = ctx->dd_rho;
    }
    NHP_CHECK(ctx, rho <= 1.0, NHP_ERR_INVALID, "BernoulliNetworkModel: link probability must be in [0, 1]");
    size_t work = 0;
    const bool stream_variant = adj_streaming(ctx, dd, &work);
    void *scratch;
    NHP_TRY(nhp_scratch(ctx, work * sizeof(double), &scratch));
    const int rc = adj_sweep(ctx, dd, stream_variant, ctx->dd_A, nullptr, rho, nullptr, seed, counter, (double *)scratch);
    const double ms = ctx->last_ms;
    NHP_TRY(nhp_disc_tables_refresh(ctx));  // also after a refused decision: the tables follow whatever A now holds
    ctx->last_ms = ms;
    return rc;
}
