"""ctypes binding of libnhp.so (include/nhp.h).  The library is the product; this module only
loads it and declares the prototypes.  There is no CPU fallback: if the shared library is
missing, or no sm_100 GPU is present, the calls raise."""
import ctypes
import os
from ctypes import POINTER, c_char_p, c_double, c_int, c_int64, c_uint64, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("NHP_LIB_PATH") or os.path.join(os.path.dirname(_HERE), "lib", "libnhp.so")  # override: A/B builds

NHP_OK = 0
NHP_ERR_INVALID, NHP_ERR_CUDA, NHP_ERR_NO_DEVICE, NHP_ERR_STATE, NHP_ERR_NUMERIC, NHP_ERR_UNSUPPORTED = -1, -2, -3, -4, -5, -6
NHP_EXPONENTIAL, NHP_LOGITNORMAL = 0, 1
NHP_OPT_SWEEP_LOGLIK = 1

c_double_p = POINTER(c_double)
c_int64_p = POINTER(c_int64)

# name -> (restype, argtypes); mirrors include/nhp.h (the boundary) and include/nhp_devel.h (measurement / test hooks) one to one
PROTOTYPES = {
    "nhp_create": (c_int, [c_int, POINTER(c_void_p)]),
    "nhp_destroy": (c_int, [c_void_p]),
    "nhp_last_error": (c_char_p, [c_void_p]),
    "nhp_version": (c_int, []),
    "nhp_launch_count": (c_int64, [c_void_p]),
    "nhp_last_kernel_ms": (c_double, [c_void_p]),
    "nhp_set_option": (c_int, [c_void_p, c_int, c_int64]),
    "nhp_set_stream": (c_int, [c_void_p, c_void_p]),
    "nhp_bench_fp64": (c_int, [c_void_p, c_int, c_double_p]),
    "nhp_test_fastmath": (c_int, [c_void_p, c_int, c_void_p, c_int64, c_void_p]),
    "nhp_events_upload": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_double, c_int64, c_int64, c_int64, c_int, POINTER(c_void_p)]),
    "nhp_events_free": (c_int, [c_void_p, c_void_p]),
    "nhp_events_count": (c_int64, [c_void_p]),
    "nhp_cont_rand": (c_int, [c_void_p, c_double, c_uint64, c_int64, POINTER(c_void_p)]),
    "nhp_events_download": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_double_p]),
    "nhp_cont_params_set": (c_int, [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_double]),
    "nhp_cont_horizon": (c_int, [c_void_p, c_int64, c_int, c_double_p]),
    "nhp_cont_loglik": (c_int, [c_void_p, c_void_p, c_int, c_double_p]),
    "nhp_cont_loglik_grad": (c_int, [c_void_p, c_void_p, c_int, c_double_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_loglik_grad_dev": (c_int, [c_void_p, c_void_p, c_int]),
    "nhp_cont_loglik_grad_read": (c_int, [c_void_p, c_void_p, c_double_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_event_intensity": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nhp_cont_intensity": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_void_p]),
    "nhp_cont_resample_parents": (c_int, [c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_sweep_loglik": (c_int, [c_void_p, c_void_p, c_double_p]),
    "nhp_cont_parents_set": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nhp_cont_suffstats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_resample_adjacency": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p]),
    "nhp_cont_resample_adjacency_cols": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p, c_int64, c_int64]),
    "nhp_cont_resample_adjacency_dev": (c_int, [c_void_p, c_void_p, c_double, c_uint64, c_uint64, c_int64, c_int64, c_int]),
    "nhp_cont_adjacency_commit": (c_int, [c_void_p]),
    "nhp_cont_network_get": (c_int, [c_void_p, c_double_p]),
    "nhp_cont_parents_get": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_disc_conv_export": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nhp_cont_network_set": (c_int, [c_void_p, c_double]),
    "nhp_cont_resample_network": (c_int, [c_void_p, c_uint64, c_uint64, c_double, c_double, c_double_p]),
    "nhp_cont_adjacency_info": (c_int, [c_void_p, c_double_p]),
    "nhp_cont_sweep_info": (c_int, [c_void_p, c_double_p]),
    "nhp_cont_params_save": (c_int, [c_void_p]),
    "nhp_cont_params_restore": (c_int, [c_void_p]),
    "nhp_comm_unique_id": (c_int, [c_void_p]),
    "nhp_comm_init": (c_int, [c_void_p, c_void_p, c_int, c_int]),
    "nhp_comm_destroy": (c_int, [c_void_p]),
    "nhp_comm_rank": (c_int, [c_void_p, POINTER(c_int), POINTER(c_int)]),
    "nhp_comm_allreduce_stats": (c_int, [c_void_p, c_int]),
    "nhp_comm_allreduce_host": (c_int, [c_void_p, c_void_p, c_int64]),
    "nhp_disc_loglik_grad": (c_int, [c_void_p, c_void_p, POINTER(c_double), c_void_p, c_void_p, c_void_p]),
    "nhp_disc_resample_params": (c_int, [c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_loglik_dist": (c_int, [c_void_p, c_void_p, c_void_p, c_int, POINTER(c_double)]),
    "nhp_cont_baseline_grid": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "nhp_cont_baseline_loglik": (c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_baseline_prior": (c_int, [c_void_p, c_int64, c_void_p, c_double]),
    "nhp_cont_resample_baseline": (c_int, [c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_baseline_get": (c_int, [c_void_p, c_void_p]),
    "nhp_cont_slice_info": (c_int, [c_void_p, c_double_p]),
    "nhp_cont_trace_begin": (c_int, [c_void_p, c_int64]),
    "nhp_cont_trace_push": (c_int, [c_void_p]),
    "nhp_cont_trace_count": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "nhp_cont_trace_read": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_trace_free": (c_int, [c_void_p]),
    "nhp_cont_trace_read_curves": (c_int, [c_void_p, c_int64, c_int64, c_void_p]),
    "nhp_comm_allgather_adjacency": (c_int, [c_void_p]),
    "nhp_comm_allgather_events": (c_int, [c_void_p, c_void_p, ctypes.POINTER(c_void_p)]),
    "nhp_cont_gibbs_sweep": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint64, c_double, c_void_p, c_int, c_double, c_double]),
    "nhp_cont_stats_dev": (c_int, [c_void_p, c_int, POINTER(c_void_p), c_int64_p]),
    "nhp_cont_suffstats_second_pass": (c_int, [c_void_p, c_void_p]),
    "nhp_cont_suffstats_read": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_resample_params": (c_int, [c_void_p, c_void_p, c_uint64, c_uint64, c_double, c_void_p, c_int, c_int]),
    "nhp_cont_params_get": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_loglik_dev": (c_int, [c_void_p, c_void_p, c_int]),
    "nhp_cont_vb_set": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "nhp_cont_vb_get": (c_int, [c_void_p, c_void_p]),
    "nhp_cont_vb_network_set": (c_int, [c_void_p, c_void_p, c_int, c_void_p]),
    "nhp_cont_vb_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_cont_vb_step": (c_int, [c_void_p, c_void_p, c_double_p]),
    "nhp_cont_vb_trace_begin": (c_int, [c_void_p, c_int64]),
    "nhp_cont_vb_trace_count": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "nhp_cont_vb_trace_read": (c_int, [c_void_p, c_int64, c_int64, c_void_p]),
    "nhp_cont_vb_trace_free": (c_int, [c_void_p]),
    "nhp_disc_upload": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_int64, POINTER(c_void_p)]),
    "nhp_disc_free": (c_int, [c_void_p, c_void_p]),
    "nhp_disc_rand": (c_int, [c_void_p, c_int64, c_int64, c_uint64, c_int64, POINTER(c_void_p)]),
    "nhp_disc_download": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nhp_disc_events_count": (c_int64, [c_void_p]),
    "nhp_disc_basis": (c_int, [c_int64, c_int64, c_double, c_void_p]),
    "nhp_disc_convolve": (c_int, [c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_void_p]),
    "nhp_disc_params_set": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_double]),
    "nhp_disc_intensity": (c_int, [c_void_p, c_void_p, c_void_p]),
    "nhp_disc_loglik": (c_int, [c_void_p, c_void_p, c_double_p]),
    "nhp_disc_gibbs_counts": (c_int, [c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_int64, c_void_p]),
    "nhp_disc_vb_stats": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_disc_resample_adjacency": (c_int, [c_void_p, c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_void_p]),
    "nhp_disc_params_get": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_disc_resample_adjacency_dev": (c_int, [c_void_p, c_void_p, c_double, c_uint64, c_uint64]),
    "nhp_disc_network_set": (c_int, [c_void_p, c_double]),
    "nhp_disc_network_get": (c_int, [c_void_p, c_double_p]),
    "nhp_disc_trace_begin": (c_int, [c_void_p, c_int64]),
    "nhp_disc_trace_push": (c_int, [c_void_p]),
    "nhp_disc_trace_count": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "nhp_disc_trace_read": (c_int, [c_void_p, c_int64, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "nhp_disc_trace_free": (c_int, [c_void_p]),
    "nhp_disc_gibbs_sweep": (c_int, [c_void_p, c_void_p, c_uint64, c_uint64, c_void_p, c_int, c_double, c_double]),
    "nhp_disc_vb_set": (c_int, [c_void_p, c_int64, c_int64, c_double, c_void_p, c_int, c_void_p]),
    "nhp_disc_vb_get": (c_int, [c_void_p, c_void_p]),
    "nhp_disc_vb_network_set": (c_int, [c_void_p, c_int64, c_int64, c_double, c_void_p, c_int, c_void_p]),
    "nhp_disc_vb_step": (c_int, [c_void_p, c_void_p, c_double_p]),
    "nhp_disc_svi_step": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_double, c_double_p]),
    "nhp_disc_vb_trace_begin": (c_int, [c_void_p, c_int64]),
    "nhp_disc_vb_trace_count": (c_int, [c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "nhp_disc_vb_trace_read": (c_int, [c_void_p, c_int64, c_int64, c_void_p]),
    "nhp_disc_vb_trace_free": (c_int, [c_void_p]),
}

_lib = None


class NHPError(RuntimeError):
    def __init__(self, code, message):
        super().__init__(f"libnhp error {code}: {message}")
        self.code = code


def load():
    """Load libnhp.so; raises if it has not been built (python __graft_entry__.py / make -C csrc)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: build it with `make -C networkhawkesprocesses.jl_b200/csrc` "
                          "(there is no CPU fallback for the hot path)")
    lib = ctypes.CDLL(LIB_PATH)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(ctx, rc):
    if rc != NHP_OK:
        msg = load().nhp_last_error(ctx)
        raise NHPError(rc, msg.decode() if msg else "")
