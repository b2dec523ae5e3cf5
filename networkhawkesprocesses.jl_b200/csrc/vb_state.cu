// vb_state.cu -- the mean-field VB state kept with the context (VbState, nhp_internal.cuh), shared by the discrete (disc_vb.cu) and
// the continuous (cont_vb.cu) steps: the checks of q's entries and its upload, the read-back, and the trace of the steps' states.  The
// model-specific checks (hyper-parameters, dimensions) stay with the models.
#include "nhp_internal.cuh"
#include <cmath>

int nhp_vb_state_set(nhp_ctx *ctx, VbState &st, const char *fn, const double *q, size_t doubles, size_t alloc, size_t fin_lo, size_t fin_hi,
                     size_t p_lo, size_t p_hi, int64_t n, int64_t b, bool network) {
    for (size_t i = 0; i < doubles; i++) {
        if (i >= fin_lo && i < fin_hi)
            NHP_CHECK(ctx, std::isfinite(q[i]), NHP_ERR_INVALID, "%s: q[%zu] = %g is not finite", fn, i, q[i]);
        else if (i >= p_lo && i < p_hi)
            NHP_CHECK(ctx, q[i] >= 0.0 && q[i] <= 1.0, NHP_ERR_INVALID, "%s: q[%zu] = %g is a link probability outside [0, 1]", fn, i, q[i]);
        else
            NHP_CHECK(ctx, q[i] > 0.0 && std::isfinite(q[i]), NHP_ERR_INVALID, "%s: q[%zu] = %g is not positive and finite", fn, i, q[i]);
    }
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    if (st.cap < alloc) {
        NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        cudaFree(st.q); st.q = nullptr; st.cap = 0; st.set = false;
        NHP_CUDA(ctx, cudaMalloc(&st.q, alloc * sizeof(double)));
        st.cap = alloc;
    }
    NHP_CUDA(ctx, cudaMemcpyAsync(st.q, q, doubles * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));  // the caller may reuse q after return
    st.n = n; st.b = b; st.network = network; st.doubles = doubles;
    st.set = true;
    return NHP_OK;
}

int nhp_vb_state_get(nhp_ctx *ctx, const VbState &st, const char *fn, const char *set_fn, double *q) {
    NHP_CHECK(ctx, st.set, NHP_ERR_STATE, "%s: no VB state (call %s)", fn, set_fn);
    NHP_CHECK(ctx, q != nullptr, NHP_ERR_INVALID, "%s: NULL argument", fn);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_CUDA(ctx, cudaMemcpyAsync(q, st.q, st.doubles * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}

void nhp_vb_state_free(nhp_ctx *ctx, VbState &st) {
    nhp_trace_free(ctx, st.trace);
    cudaFree(st.q);
    st = VbState();
}

int nhp_vb_trace_begin(nhp_ctx *ctx, VbState &st, const char *fn, const char *set_fn, int64_t capacity) {
    NHP_CHECK(ctx, st.set, NHP_ERR_STATE, "%s: no VB state (the slot size follows it; call %s)", fn, set_fn);
    return nhp_trace_begin(ctx, st.trace, fn, capacity, st.doubles, 0, 0, TraceShape{st.n, st.b, st.network, 0});
}

int nhp_vb_trace_push(nhp_ctx *ctx, VbState &st) {
    if (double *slot = st.trace.next()) {
        NHP_CUDA(ctx, cudaMemcpyAsync(slot, st.q, st.trace.doubles * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        st.trace.len++;
    }
    return NHP_OK;
}

int nhp_vb_trace_read(nhp_ctx *ctx, const VbState &st, const char *fn, int64_t first, int64_t count, double *q_out) {
    NHP_TRY(nhp_trace_check_range(ctx, st.trace, fn, first, count));
    if (count == 0) return NHP_OK;
    NHP_CHECK(ctx, q_out != nullptr, NHP_ERR_INVALID, "%s: NULL argument", fn);
    NHP_CUDA(ctx, cudaSetDevice(ctx->device));
    NHP_TRY(nhp_trace_read_field(ctx, st.trace, first, count, 0, st.trace.doubles, q_out));
    NHP_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return NHP_OK;
}
