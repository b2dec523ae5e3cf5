// cont_child.cu -- child-major dense sweeps for large K (parameter table K^2 * 16|32 B beyond what L2 serves well:
// 400 MB at K = 5000, config 5).  The time-tiled sweep gathers one random table entry per pair; once the table
// no longer fits L2 that gather is an HBM sector per pair (173 GB for 2e7 events at K = 5000).  Here one CTA owns a
// child node c at a time: the table column of c (K entries, 80-160 KB) is staged in shared memory once, and the
// CTA walks the child events of c (by-node order built once per data set with a stable radix sort); each warp
// takes one event and strides its window with coalesced reads of the time-sorted stream.  HBM traffic becomes
// the window reads (12 B per pair, sequential) and the parameter lookups are shared-memory reads.
// Same arithmetic and the same per-event order as the reference loops (continuous.jl:286-300, parents.jl:25-46).
#include "cont_sweep.cuh"
#include <cub/cub.cuh>
#include <algorithm>

constexpr int CH_EVENTS = 256;  // child events per work item
constexpr int CR = 8;           // cached window rows (32 entries each) per warp in the parent sweep

struct ChildArgs {
    SweepArgs s;
    const int *order;       // [n_own] local event indices grouped by node, time order inside a node
    const int *node_ptr;    // [K+1]
    const int *item_node;   // [nitems]
    const int *item_e0;     // [nitems] first position in `order`
    int64_t nitems;
    int mode;               // 0 loglik, 1 intensity, 2 parents
    const unsigned short *wlen;  // [n_own] cached window length per own event (65535 = saturated)
};

__global__ void k_child_iota(int *v, int64_t n, int first) {
    int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) v[i] = first + (int)i;
}

template <int KIND> __global__ void __launch_bounds__(1024) k_child_sweep(const ChildArgs ca) {
    typedef typename EntryOf<KIND>::type E;
    const SweepArgs &a = ca.s;
    extern __shared__ __align__(128) unsigned char smem[];
    __shared__ FastTables s_ft;
    __shared__ double red[64];
    const int BS = blockDim.x;  // 256 .. 1024: as many warps per column as the column's shared-memory footprint leaves room for
    E *col = reinterpret_cast<E *>(smem);                                        // [K] table column of the current child
    double *s_v = reinterpret_cast<double *>(smem + (size_t)a.K * sizeof(E));   // [CR * BS] parent-sweep weight cache
    fast_tables_load(&s_ft);
    const FastTables *ft = &s_ft;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const StatsLayout sl{a.K};
    const int64_t ipc = (ca.nitems + gridDim.x - 1) / gridDim.x;
    const int64_t it0 = blockIdx.x * ipc, it1 = min(ca.nitems, it0 + ipc);
    double sum_log = 0.0, sum_row = 0.0;
    int cur = -1;
    double *my_v = s_v + threadIdx.x;
    for (int64_t item = it0; item < it1; item++) {
        const int c = ca.item_node[item];
        if (c != cur) {
            __syncthreads();
            const E *src = reinterpret_cast<const E *>(a.table) + (size_t)c * a.K;
            for (int k = threadIdx.x; k < a.K; k += BS) col[k] = load_entry(src + k);
            cur = c;
            __syncthreads();
        }
        const int e0 = ca.item_e0[item], e1 = min(e0 + CH_EVENTS, ca.node_ptr[c + 1]);
        const double lam0_node = __ldg(a.lambda0 + c);
        int m0 = 0;
        for (int e = e0 + warp; e < e1; e += BS / 32) {
            const int i = ca.order[e];
            const double lam0 = a.lam0ev ? __ldg(a.lam0ev + i) : lam0_node;
            const double ti = __ldg(a.t + i);
            const double thr = ti - a.horizon;
            const int jlo = (int)a.jmin;
            // pass 1: window weights, most recent first, lanes striding the window (coalesced stream reads)
            double acc = 0.0;
            int nr = 0;
            const int wraw = (int)__ldg(ca.wlen + (i - a.first));
            if (wraw < 65535) {
                // window length known up front: no data-dependent exit, so the loads of several trips are in flight together
                // (child events of one node are ~K events apart in the stream: every window is a cold DRAM read)
                const int w = min(wraw, i - jlo);
#pragma unroll 4
                for (int k = lane; k < w; k += 32, nr++) {
                    const int j = i - 1 - k;
                    const double v = pair_value(col[__ldg(a.c + j)], ti - __ldg(a.t + j), a.D, ft);
                    acc += v;
                    if (ca.mode == 2 && nr < CR) my_v[nr * BS] = v;
                }
            } else {
                for (int j = i - 1 - lane; j >= jlo; j -= 32, nr++) {
                    const double tj = __ldg(a.t + j);
                    if (!(tj > thr)) break;
                    const double v = pair_value(col[__ldg(a.c + j)], ti - tj, a.D, ft);
                    acc += v;
                    if (ca.mode == 2 && nr < CR) my_v[nr * BS] = v;
                }
            }
            const double S = warp_sum(acc) + lam0;
            if (ca.mode == 0) { if (lane == 0) { sum_log += log(S); sum_row += __ldg(a.rowsum + c); } }
            else if (ca.mode == 1) { if (lane == 0) a.lam_out[i - a.first] = S; }
            else {
                const int64_t gi = a.index_base + i;
                const double u = a.u ? __ldg(a.u + (i - a.first)) : philox_uniform(a.seed, (uint64_t)gi, a.counter);
                const double target = u * S;
                const int nrows = (gi == 0) ? 0 : __shfl_sync(0xffffffffu, nr, 0);
                int chosen = 0;
                double carry = 0.0;
                for (int r = 0; r < nrows; r++) {
                    double v = 0.0;
                    if (r < nr) {
                        if (r < CR) v = my_v[r * BS];
                        else {
                            const int jj = i - 1 - lane - r * 32;
                            v = pair_value(col[__ldg(a.c + jj)], ti - __ldg(a.t + jj), a.D, ft);
                        }
                    }
                    const double x = group_incl_scan<32>(v, 0xffffffffu, lane);
                    const unsigned b = __ballot_sync(0xffffffffu, carry + x > target);
                    if (b) { chosen = r * 32 + (__ffs(b) - 1) + 1; break; }
                    carry += __shfl_sync(0xffffffffu, x, 31);
                }
                if (lane == 0) {
                    if (!(S > 0.0) || S > 1.7976931348623157e308) atomicOr(a.flag, 8);
                    if (a.want_ll) { sum_log += log(S); sum_row += __ldg(a.rowsum + c); }
                    a.poff[i] = chosen;
                    if (chosen == 0) m0++;
                    else {
                        const int jp = i - chosen;
                        const int cj = __ldg(a.c + jp);
                        const double dt = ti - __ldg(a.t + jp);
                        const int64_t k = cj + (int64_t)a.K * c;
                        red_add_f64(a.stats + sl.off_Mnm() + k, 1.0);
                        red_add_f64(a.stats + sl.off_S1() + k, KIND == NHP_LOGITNORMAL ? log_duration_dev(dt, a.D) : dt);
                    }
                }
            }
        }
        if (ca.mode == 2 && lane == 0 && m0) red_add_f64(a.stats + sl.off_M0() + c, (double)m0);
    }
    if (ca.mode == 0 || ca.mode == 2) {
        block_sum2_any(sum_log, sum_row, red);
        if (threadIdx.x == 0) { a.partials[2 * (size_t)blockIdx.x] = sum_log; a.partials[2 * (size_t)blockIdx.x + 1] = sum_row; }
    }
}

// by-node order of the own events + work items; cached in the events handle (data dependent only)
int nhp_events_build_node_index(nhp_ctx *ctx, nhp_events *ev) {
    if (ev->d_order) return NHP_OK;
    const int64_t own = ev->n - ev->n_halo, K = ev->K;
    cudaStream_t s = ctx->stream;
    int *d_vals = nullptr, *d_keys = nullptr;
    void *d_tmp = nullptr;
    // every failure path releases the temporaries and leaves the handle without a (partial) index
    auto fail = [&](cudaError_t e, const char *what) {
        cudaFreeAsync(d_vals, s); cudaFreeAsync(d_keys, s); cudaFreeAsync(d_tmp, s);
        cudaFreeAsync(ev->d_order, s); cudaFreeAsync(ev->d_node_ptr, s); cudaFreeAsync(ev->d_item_node, s); cudaFreeAsync(ev->d_item_e0, s);
        ev->d_order = ev->d_node_ptr = ev->d_item_node = ev->d_item_e0 = nullptr;
        return nhp_fail(ctx, NHP_ERR_CUDA, "node index: %s failed: %s", what, cudaGetErrorString(e));
    };
#define NI_CUDA(call) do { cudaError_t e__ = (call); if (e__ != cudaSuccess) return fail(e__, #call); } while (0)
    NI_CUDA(cudaMallocAsync(&ev->d_order, (size_t)std::max<int64_t>(own, 1) * sizeof(int), s));
    NI_CUDA(cudaMallocAsync(&d_vals, (size_t)std::max<int64_t>(own, 1) * sizeof(int), s));
    NI_CUDA(cudaMallocAsync(&d_keys, (size_t)std::max<int64_t>(own, 1) * sizeof(int), s));
    if (own > 0) {
        k_child_iota<<<(unsigned)((own + 255) / 256), 256, 0, s>>>(d_vals, own, (int)ev->n_halo);
        NHP_LAUNCHED(ctx);
        int bits = 1;
        while ((1 << bits) < K) bits++;
        size_t tb = 0;
        cub::DeviceRadixSort::SortPairs(nullptr, tb, ev->d_c + ev->n_halo, d_keys, d_vals, ev->d_order, (int)own, 0, bits, s);
        NI_CUDA(cudaMallocAsync(&d_tmp, tb, s));
        NI_CUDA(cub::DeviceRadixSort::SortPairs(d_tmp, tb, ev->d_c + ev->n_halo, d_keys, d_vals, ev->d_order, (int)own, 0, bits, s));  // stable
        NHP_LAUNCHED(ctx);
    }
    std::vector<double> mn(K);
    NI_CUDA(cudaMemcpyAsync(mn.data(), ev->d_Mn, (size_t)K * sizeof(double), cudaMemcpyDeviceToHost, s));
    NI_CUDA(cudaStreamSynchronize(s));
    cudaFreeAsync(d_vals, s); cudaFreeAsync(d_keys, s); cudaFreeAsync(d_tmp, s);  // stream-ordered pool: no device synchronisation
    d_vals = d_keys = nullptr; d_tmp = nullptr;
    std::vector<int> ptr(K + 1), inode, ie0;
    int run = 0;
    for (int64_t k = 0; k < K; k++) {
        ptr[k] = run;
        int nk = (int)mn[k];
        for (int off = 0; off < nk; off += CH_EVENTS) { inode.push_back((int)k); ie0.push_back(run + off); }
        run += nk;
    }
    ptr[K] = run;
    ev->n_items = (int64_t)inode.size();
    NI_CUDA(cudaMallocAsync(&ev->d_node_ptr, (size_t)(K + 1) * sizeof(int), s));
    NI_CUDA(cudaMallocAsync(&ev->d_item_node, std::max<size_t>(inode.size(), 1) * sizeof(int), s));
    NI_CUDA(cudaMallocAsync(&ev->d_item_e0, std::max<size_t>(inode.size(), 1) * sizeof(int), s));
    NI_CUDA(cudaMemcpyAsync(ev->d_node_ptr, ptr.data(), (size_t)(K + 1) * sizeof(int), cudaMemcpyHostToDevice, s));
    if (!inode.empty()) {
        NI_CUDA(cudaMemcpyAsync(ev->d_item_node, inode.data(), inode.size() * sizeof(int), cudaMemcpyHostToDevice, s));
        NI_CUDA(cudaMemcpyAsync(ev->d_item_e0, ie0.data(), ie0.size() * sizeof(int), cudaMemcpyHostToDevice, s));
    }
    NI_CUDA(cudaStreamSynchronize(s));  // the host vectors go out of scope
#undef NI_CUDA
    return NHP_OK;
}

// mode: 0 loglik, 1 intensity, 2 parents.  Returns NHP_OK after launching (grid in *grid_out), 1 if not applicable.
int nhp_cont_try_child(nhp_ctx *ctx, nhp_events *ev, SweepArgs &a, int mode, int *grid_out) {
    const char *env = getenv("NHP_CHILD");
    if (env && atoi(env) == 0) return 1;
    const bool force = env && atoi(env) == 1;
    const int64_t K = ctx->K, own = ev->n - ev->n_halo;
    const size_t esz = ctx->kind == NHP_LOGITNORMAL ? sizeof(EntryLN) : sizeof(EntryEX);
    // threads per CTA: the column (K entries) is the CTA's fixed shared-memory cost, so large columns leave room for few CTAs
    // per SM; give those CTAs more warps (the per-event window reads are cold DRAM: latency is hidden by warps in flight)
    const size_t col_bytes = (size_t)K * esz;
    const int fit = (int)std::max<size_t>(1, ((size_t)ctx->smem_optin - 8192) / std::max<size_t>(col_bytes, 1));
    const int block = fit >= 8 ? 256 : (fit >= 4 ? 512 : 1024);
    const size_t smem = col_bytes + (mode == 2 ? (size_t)CR * block * sizeof(double) : 0);
    if (smem > (size_t)ctx->smem_optin - 8192 || own == 0) return 1;
    // worthwhile when the table no longer sits comfortably in L2 and every column is amortised over enough pairs
    const bool big_table = (double)K * K * esz > 96e6;  // beyond L2 (126 MB): measured crossover (K = 1000 LN, 32 MB: time-tiled 5.1 ms vs child-major 7.7 ms per 1e7 events; K = 5000 Exp, 400 MB: 140 ms vs 61 ms per 2e7)
    const bool amortised = (double)own / K * std::max(ev->mean_win, 1.0) > 8.0 * K;
    if (!force && !(big_table && amortised)) return 1;
    NHP_TRY(nhp_events_build_node_index(ctx, ev));
    if (ev->n_items == 0) return 1;
    NHP_CUDA(ctx, fast_tables_upload(ctx->stream));
    ChildArgs ca;
    ca.s = a; ca.order = ev->d_order; ca.node_ptr = ev->d_node_ptr; ca.item_node = ev->d_item_node; ca.item_e0 = ev->d_item_e0;
    ca.nitems = ev->n_items; ca.mode = mode; ca.wlen = ev->d_wlen;
    auto launch = [&](auto kernel) -> int {
        NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)std::max<size_t>(smem, 1024)));  // always: static + dynamic may exceed the 48 KB default even when the dynamic part is small
        NHP_CUDA(ctx, cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
        int per_sm = 1;
        NHP_CUDA(ctx, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kernel, block, smem));
        int grid = (int)std::min<int64_t>(ev->n_items, (int64_t)ctx->sm_count * std::max(per_sm, 1));
        *grid_out = grid;
        kernel<<<grid, block, smem, ctx->stream>>>(ca);
        NHP_LAUNCHED(ctx);
        NHP_CUDA(ctx, cudaGetLastError());
        return NHP_OK;
    };
    if (ctx->kind == NHP_LOGITNORMAL) return launch(k_child_sweep<NHP_LOGITNORMAL>);
    return launch(k_child_sweep<NHP_EXPONENTIAL>);
}
