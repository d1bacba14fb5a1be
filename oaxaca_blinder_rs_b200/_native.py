"""ctypes binding of libobboot (include/obboot.h).  No fallback: if the CUDA library is missing or
no B200 is visible, every entry point raises."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "_lib", "libobboot.so")
CSRC = os.path.join(_HERE, "csrc")

_DP = C.POINTER(C.c_double)
_IP = C.POINTER(C.c_int32)
_U32P = C.POINTER(C.c_uint32)

STATUS_NAMES = {0: "Ok", 1: "PolarsError", 2: "ColumnNotFound", 3: "InvalidGroupVariable", 4: "NalgebraError",
                5: "DiagnosticError", 6: "InsufficientData", 7: "InvalidArgument", 8: "CudaError", 9: "NcclError",
                10: "NoDevice", 11: "Unsupported"}

# every symbol include/obboot.h declares (checked by tests/test_abi.py against the header)
SYMBOLS = ["ob_abi_version", "ob_device_count", "ob_ctx_create", "ob_ctx_destroy", "ob_last_error",
           "ob_design_pack", "ob_design_from_dense", "ob_design_destroy", "ob_design_shape", "ob_design_download",
           "ob_design_apply_rif", "ob_num_stats", "ob_bootstrap_run", "ob_reduce_stats", "ob_debug_counts",
           "ob_comm_unique_id", "ob_comm_init_nccl", "ob_local_group_create", "ob_local_group_destroy",
           "ob_comm_init_local", "ob_comm_destroy", "ob_row_shard_plan", "ob_design_set_row_shard",
           "ob_design_pack_timings", "ob_design_allgather_rows", "ob_design_update_outcome",
           "ob_ingest_begin", "ob_ingest_rows_kept", "ob_ingest_presence", "ob_ingest_finish", "ob_ingest_destroy",
           "ob_debug_gram_schedule", "ob_debug_counts_from_indices", "ob_host_alloc", "ob_host_free",
           "ob_host_register", "ob_host_unregister", "ob_replicate_shard", "ob_design_pack_async", "ob_design_wait",
           "ob_design_redistribute_rows", "ob_design_row_shard", "ob_design_apply_rif_multi", "ob_design_num_outcomes",
           "ob_design_pack_row_shard_async", "ob_design_attach_selection", "ob_design_selection_cols", "ob_num_stats_heckman",
           "ob_mm_run", "ob_debug_gram_columns", "ob_gram_cache_create", "ob_gram_cache_destroy", "ob_gram_cache_last_use",
           "ob_bootstrap_run_cached", "ob_debug_gram_outcome_columns", "ob_design_attach_clusters", "ob_design_clusters",
           "ob_bootstrap_run_bayes", "ob_debug_bayes_weights",
           "ob_debug_gram_cache_read"]


class FrameView(C.Structure):
    _fields_ = [("n", C.c_int64), ("n_cont", C.c_int32), ("cont", C.POINTER(_DP)), ("n_cat", C.c_int32),
                ("cat_codes", C.POINTER(_IP)), ("cat_levels", _IP), ("outcome", _DP), ("weights", _DP),
                ("group", C.POINTER(C.c_uint8))]


class RawF64(C.Structure):
    _fields_ = [("data", _DP), ("valid", C.POINTER(C.c_uint8))]


class RawDict(C.Structure):
    _fields_ = [("codes", _IP), ("dict_size", C.c_int32)]


class RawFrame(C.Structure):
    _fields_ = [("n", C.c_int64), ("n_cont", C.c_int32), ("cont", C.POINTER(RawF64)), ("n_cat", C.c_int32),
                ("cat", C.POINTER(RawDict)), ("outcome", RawF64), ("weights", RawF64), ("group", RawDict),
                ("nan_is_null", C.c_int32)]


class SelectionView(C.Structure):
    _fields_ = [("n_pred", C.c_int32), ("pred", C.POINTER(_DP)), ("outcome", _DP)]


class BayesOpts(C.Structure):
    _fields_ = [("wt_a", C.POINTER(C.c_float)), ("wt_b", C.POINTER(C.c_float))]


class BootOpts(C.Structure):
    _fields_ = [("ref_kind", C.c_int32), ("n_norm", C.c_int32), ("norm_m", _IP), ("norm_off", _IP),
                ("norm_idx", _IP), ("norm_has_base", _IP), ("reps", C.c_int64), ("seed", C.c_uint64),
                ("idx_a", _U32P), ("idx_b", _U32P), ("rep_begin", C.c_int64), ("rep_end", C.c_int64),
                ("skip_reduce", C.c_int32), ("count_bits", C.c_int32), ("max_workspace_bytes", C.c_int64),
                ("shard_replicates", C.c_int32)]


class Result(C.Structure):
    _fields_ = [("total_gap", C.c_double), ("point_stats", _DP), ("xa_mean", _DP), ("xb_mean", _DP),
                ("beta_star", _DP), ("beta_a", _DP), ("beta_b", _DP), ("residuals_b", _DP),
                ("n_ok", C.c_int64), ("std_err", _DP), ("p_value", _DP), ("ci_lower", _DP), ("ci_upper", _DP),
                ("t_stat", _DP), ("rep_stats", _DP), ("rep_status", _IP), ("rep_beta_a", _DP), ("rep_beta_b", _DP),
                ("ms_counts", C.c_double), ("ms_gram", C.c_double), ("ms_solve", C.c_double),
                ("ms_reduce", C.c_double), ("ms_total", C.c_double), ("ms_gram_kernel", C.c_double),
                ("gpu_launches", C.c_int32), ("ms_comm", C.c_double), ("total_gap_multi", _DP), ("sel_gamma_a", _DP), ("sel_gamma_b", _DP)]


class MmOpts(C.Structure):
    _fields_ = [("simulations", C.c_int32), ("n_quantiles", C.c_int32), ("quantiles", _DP), ("reps", C.c_int64),
                ("seed", C.c_uint64), ("idx_a", _U32P), ("idx_b", _U32P), ("taus", _DP), ("draw_a", _U32P), ("draw_b", _U32P),
                ("rep_begin", C.c_int64), ("rep_end", C.c_int64), ("skip_reduce", C.c_int32), ("count_bits", C.c_int32),
                ("max_workspace_bytes", C.c_int64), ("shard_replicates", C.c_int32)]


class MmResult(C.Structure):
    _fields_ = [("point_stats", _DP), ("n_ok", C.c_int64), ("std_err", _DP), ("p_value", _DP), ("ci_lower", _DP),
                ("ci_upper", _DP), ("t_stat", _DP), ("rep_stats", _DP), ("rep_status", _IP), ("point_betas_a", _DP),
                ("point_betas_b", _DP), ("point_qr_info_a", _IP), ("point_qr_info_b", _IP), ("qr_total", C.c_int64),
                ("qr_vertex", C.c_int64), ("qr_approx", C.c_int64), ("qr_failed", C.c_int64), ("qr_iterations", C.c_int64),
                ("ms_counts", C.c_double), ("ms_qr", C.c_double), ("ms_effects", C.c_double), ("ms_reduce", C.c_double),
                ("ms_total", C.c_double), ("gpu_launches", C.c_int32)]


def build(force: bool = False) -> str:
    """Compile libobboot.so for sm_100a in-tree (nvcc cross-compiles without a GPU)."""
    srcs = [os.path.join(dp, f) for dp, _, fs in os.walk(CSRC) for f in fs]
    srcs += [os.path.join(_HERE, "..", "include", h) for h in ("obboot.h", "obboot_builder.h")]
    newest = max(os.path.getmtime(s) for s in srcs)
    if force or not os.path.exists(LIB_PATH) or os.path.getmtime(LIB_PATH) < newest:
        subprocess.check_call(["make", "-C", CSRC, "-j8", "-s"])
    return LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(f"libobboot.so not built ({LIB_PATH}); run `python -c 'import __graft_entry__ as g; "
                               f"g.build()'` -- there is no CPU fallback")
        L = C.CDLL(LIB_PATH)
        L.ob_abi_version.restype = C.c_uint32
        L.ob_last_error.restype = C.c_char_p
        L.ob_last_error.argtypes = [C.c_void_p]
        L.ob_ctx_create.argtypes = [C.c_int32, C.POINTER(C.c_void_p)]
        L.ob_ctx_destroy.argtypes = [C.c_void_p]
        L.ob_ctx_destroy.restype = None
        L.ob_design_destroy.argtypes = [C.c_void_p]
        L.ob_design_destroy.restype = None
        L.ob_design_pack.argtypes = [C.c_void_p, C.POINTER(FrameView), C.POINTER(C.c_void_p)]
        L.ob_design_from_dense.argtypes = [C.c_void_p, C.c_int32, C.c_int32, _DP, _DP, _DP, C.c_int64,
                                           _DP, _DP, _DP, C.c_int64, C.POINTER(C.c_void_p)]
        L.ob_design_shape.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _IP, _IP]
        L.ob_design_download.argtypes = [C.c_void_p, C.c_void_p, _DP, _DP, _DP, _DP, _DP, _DP]
        L.ob_design_apply_rif.argtypes = [C.c_void_p, C.c_void_p, C.c_double]
        L.ob_num_stats.argtypes = [C.c_int32, C.c_int32, _IP]
        L.ob_num_stats.restype = C.c_int32
        L.ob_bootstrap_run.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(BootOpts), C.POINTER(Result)]
        L.ob_gram_cache_create.argtypes = [C.c_void_p, C.POINTER(C.c_void_p)]
        L.ob_gram_cache_destroy.argtypes = [C.c_void_p]
        L.ob_gram_cache_destroy.restype = None
        L.ob_gram_cache_last_use.argtypes = [C.c_void_p, _IP, C.POINTER(C.c_int64)]
        L.ob_bootstrap_run_cached.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(BootOpts), C.c_void_p, C.POINTER(Result)]
        L.ob_bootstrap_run_bayes.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(BootOpts), C.POINTER(BayesOpts), C.c_void_p,
                                             C.POINTER(Result)]
        L.ob_debug_bayes_weights.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_int32, C.POINTER(C.c_float)]
        L.ob_debug_gram_cache_read.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), _DP, _DP, C.POINTER(C.c_int64)]
        L.ob_debug_gram_outcome_columns.argtypes = [C.c_int32, C.c_int32, C.POINTER(C.c_uint16), _IP, C.c_int64, _IP]
        L.ob_debug_gram_outcome_columns.restype = C.c_int64
        L.ob_reduce_stats.argtypes = [C.c_void_p, _DP, _IP, C.c_int64, C.c_int32, _DP, C.POINTER(C.c_int64),
                                      _DP, _DP, _DP, _DP, _DP]
        L.ob_debug_counts.argtypes = [C.c_void_p, C.c_void_p, C.c_uint64, C.c_int64, C.c_int32,
                                      C.POINTER(C.c_uint16)]
        _U8P = C.POINTER(C.c_uint8)
        L.ob_comm_unique_id.argtypes = [_U8P]
        L.ob_comm_init_nccl.argtypes = [C.c_void_p, _U8P, C.c_int32, C.c_int32]
        L.ob_local_group_create.argtypes = [C.c_int32, C.POINTER(C.c_void_p)]
        L.ob_local_group_destroy.argtypes = [C.c_void_p]
        L.ob_local_group_destroy.restype = None
        L.ob_comm_init_local.argtypes = [C.c_void_p, C.c_void_p, C.c_int32]
        L.ob_comm_destroy.argtypes = [C.c_void_p]
        L.ob_comm_destroy.restype = None
        L.ob_row_shard_plan.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.ob_design_set_row_shard.argtypes = [C.c_void_p, C.c_int64, C.c_int64, C.c_int32, C.c_int32]
        L.ob_design_pack_timings.argtypes = [C.c_void_p, _DP, _DP]
        L.ob_design_allgather_rows.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.ob_design_update_outcome.argtypes = [C.c_void_p, C.c_void_p, _DP, C.c_int64]
        L.ob_ingest_begin.argtypes = [C.c_void_p, C.POINTER(RawFrame), C.POINTER(C.c_void_p)]
        L.ob_ingest_rows_kept.argtypes = [C.c_void_p, C.POINTER(C.c_int64)]
        L.ob_ingest_presence.argtypes = [C.c_void_p, C.c_int32, _U8P]
        L.ob_ingest_finish.argtypes = [C.c_void_p, C.c_void_p, _IP, C.POINTER(_IP), _IP, C.POINTER(C.c_void_p)]
        L.ob_ingest_destroy.argtypes = [C.c_void_p]
        L.ob_ingest_destroy.restype = None
        L.ob_debug_gram_schedule.argtypes = [C.c_int32, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int32,
                                             C.POINTER(C.c_int64), C.c_int64]
        L.ob_debug_gram_schedule.restype = C.c_int64
        L.ob_debug_counts_from_indices.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, _U32P, C.c_int64, C.c_int32,
                                                   C.POINTER(C.c_uint16), _IP]
        L.ob_design_pack_async.argtypes = [C.c_void_p, C.POINTER(FrameView), C.POINTER(C.c_void_p)]
        L.ob_design_wait.argtypes = [C.c_void_p, C.c_void_p]
        L.ob_design_pack_row_shard_async.argtypes = [C.c_void_p, C.POINTER(FrameView), C.POINTER(C.c_void_p)]
        L.ob_design_apply_rif_multi.argtypes = [C.c_void_p, C.c_void_p, _DP, C.c_int32]
        L.ob_design_num_outcomes.argtypes = [C.c_void_p, _IP]
        L.ob_design_attach_selection.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(SelectionView), C.c_int64]
        L.ob_design_selection_cols.argtypes = [C.c_void_p, _IP]
        L.ob_design_attach_clusters.argtypes = [C.c_void_p, C.c_void_p, _IP, C.c_int64, C.c_int32, C.c_int32]
        L.ob_design_clusters.argtypes = [C.c_void_p, _IP, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        L.ob_num_stats_heckman.argtypes = [C.c_int32, C.c_int32]
        L.ob_num_stats_heckman.restype = C.c_int32
        L.ob_design_row_shard.argtypes = [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64), _IP, _IP]
        L.ob_design_redistribute_rows.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(C.c_void_p)]
        L.ob_host_alloc.argtypes = [C.c_size_t, C.POINTER(C.c_void_p)]
        L.ob_host_free.argtypes = [C.c_void_p]
        L.ob_host_free.restype = None
        L.ob_host_register.argtypes = [C.c_void_p, C.c_size_t]
        L.ob_host_unregister.argtypes = [C.c_void_p]
        L.ob_mm_run.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(MmOpts), C.POINTER(MmResult)]
        L.ob_replicate_shard.argtypes = [C.c_int64, C.c_int32, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]
        _lib = L
    return _lib
