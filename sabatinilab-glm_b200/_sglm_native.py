"""
ctypes binding of libsglm_b200.so (the C ABI declared in include/sglm_b200.h).

There is no CPU fallback: if the shared library is missing, or no CUDA device is
present when a compute entry point is called, this module raises.  PyTorch is used
only for device memory, streams and host<->device copies.
"""
import ctypes
import os
import threading

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libsglm_b200.so")

c_i32, c_i64, c_u64, c_f64 = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint64, ctypes.c_double
c_vp, c_sz = ctypes.c_void_p, ctypes.c_size_t

_PROTOTYPES = {
    "sglm_version": (c_i32, []),
    "sglm_last_error": (ctypes.c_char_p, []),
    "sglm_timeshift_f64": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_i32, c_u64, c_vp, c_i64, c_vp]),
    "sglm_timeshift_f64_ranged": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_i32, c_i32, c_i32,
                                          c_u64, c_vp, c_i64, c_vp]),
    "sglm_lag_valid_rows": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_i32, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "sglm_index_mask_u8": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_vp, c_vp]),
    "sglm_rows_or_bit_u64": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, c_vp]),
    "sglm_cells_from_signatures": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_vp]),
    "sglm_match_compact_rows": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_sz, c_vp]),
    "sglm_roll_f64": (c_i32, [c_vp, c_i64, c_i64, c_vp, c_vp]),
    "sglm_mask_compact_workspace_bytes": (c_sz, [c_i64]),
    "sglm_mask_compact_rows": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "sglm_timeshift_rows_f64": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_vp, c_i32, c_u64, c_vp, c_i64, c_vp,
                                        c_i64, c_vp]),
    "sglm_crop_rows_f64": (c_i32, [c_vp, c_i64, c_i64, c_i64, c_i32, c_vp, c_i64, c_vp]),
    "sglm_suffstats_workspace_bytes": (c_sz, [c_i64, c_i32, c_i32, c_i32, c_vp]),
    "sglm_suffstats_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_i64, c_i32,
                                   c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "sglm_gram_tc_analyze_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp]),
    "sglm_gram_tc_workspace_bytes": (c_sz, [c_i32, c_vp, c_i32, c_vp]),
    "sglm_gram_tc_plan_info": (c_i32, [c_i32, c_vp, c_i32, c_vp, c_vp]),
    "sglm_gram_tc_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp,
                                 c_vp, c_vp, c_i64, c_vp, c_sz, c_i32, c_vp]),
    "sglm_gram_tc_analyze_scaled_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_i32, c_vp, c_vp,
                                                c_vp, c_vp, c_vp]),
    "sglm_gram_tc_scaled_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_i32,
                                        c_vp, c_vp, c_vp, c_i64, c_vp, c_sz, c_vp]),
    "sglm_xt_vec_workspace_bytes": (c_sz, [c_i32]),
    "sglm_xt_vec_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_vp, c_vp, c_sz, c_vp]),
    "sglm_gram_tc_cells_workspace_bytes": (c_sz, [c_i32, c_vp, c_i32, c_vp, c_i32]),
    "sglm_gram_tc_cells_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp,
                                       c_vp, c_i32, c_vp, c_vp, c_i64, c_vp, c_sz, c_i32, c_vp]),
    "sglm_quadform_gemm_f64": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "sglm_gram_tc_lag_workspace_bytes": (c_sz, [c_i32, c_vp, c_i32, c_vp, c_i32, c_i32, c_vp, c_i64]),
    "sglm_gram_tc_lag_cells_f64": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp, c_vp, c_i32,
                                           c_vp, c_vp, c_i64, c_vp, c_sz, c_i32, c_vp]),
    "sglm_gram_tc_colstats_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp]),
    "sglm_gram_tc_exponents": (c_i32, [c_vp, c_i32, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "sglm_gram_tc_cells_sgout": (c_i32, [c_i32, c_vp, c_i32, c_vp, c_i32, c_vp, c_vp]),
    "sglm_gram_tc_cells_partial_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_i32,
                                               c_vp, c_vp, c_i32, c_vp, c_vp, c_sz, c_vp]),
    "sglm_gram_tc_colstats_scaled_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp]),
    "sglm_gram_tc_scaled_partial_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_i32, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp,
                                                c_i32, c_vp, c_vp, c_i32, c_vp, c_vp, c_sz, c_vp]),
    "sglm_reduce_parts_f64": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp]),
    "sglm_gram_tc_cells_combine_f64": (c_i32, [c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp, c_i32, c_vp, c_i64, c_vp,
                                               c_sz, c_vp]),
    "sglm_index_counts_f64": (c_i32, [c_vp, c_i64, c_vp, c_i64, c_vp]),
    "sglm_center_stats_f64": (c_i32, [c_vp, c_vp, c_i64, c_i32, c_i32, c_i32, c_i32, c_vp, c_i64,
                                      c_vp, c_vp, c_vp, c_vp, c_vp]),
    "sglm_enet_cd_gram_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp,
                                      c_i32, c_i32, c_i32, c_vp, c_i64, c_vp, c_vp]),
    "sglm_enet_cd_cluster_supported": (c_i32, [c_i32, c_i32]),
    "sglm_enet_cd_cluster_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp, c_vp, c_vp, c_vp,
                                         c_i32, c_i32, c_i32, c_i32, c_i32, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp]),
    "sglm_enet_cd_cluster_tmap_bytes": (c_sz, []),
    "sglm_enet_cd_cluster_smem_bytes": (c_sz, [c_i32, c_i32, c_i32]),
    "sglm_enet_cd_cluster_encode_tmaps": (c_i32, [c_vp, c_i32, c_i32, c_i64, c_vp]),
    "sglm_ridge_workspace_bytes": (c_sz, [c_i32, c_i64, c_i32]),
    "sglm_ridge_solve_f64": (c_i32, [c_vp, c_i64, c_vp, c_i32, c_vp, c_i32, c_vp, c_i64, c_vp, c_vp,
                                     c_sz, c_vp]),
    "sglm_ols_minnorm_workspace_bytes": (c_sz, [c_i32]),
    "sglm_ols_minnorm_f64": (c_i32, [c_vp, c_i64, c_vp, c_i32, c_f64, c_f64, c_i32, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sglm_chol_solve_f64": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp]),
    "sglm_finalize_models_f64": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp, c_vp, c_i32, c_vp,
                                         c_vp, c_i64, c_vp]),
    "sglm_quadform_f64": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_vp, c_vp]),
    "sglm_quadform_split_f64": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "sglm_predict_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp]),
    "sglm_score_workspace_bytes": (c_sz, []),
    "sglm_score_f64": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_i32, c_vp, c_vp,
                               c_vp, c_vp]),
    "sglm_chol_solve_batched_f64": (c_i32, [c_vp, c_i64, c_i32, c_vp, c_vp, c_i64, c_vp, c_i32, c_vp]),
    "sglm_pb_gemm_tn_workspace_bytes": (c_sz, [c_i64, c_i32, c_i64]),
    "sglm_pb_eta_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp]),
    "sglm_pb_xt_r_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_vp, c_i64, c_vp, c_vp, c_sz, c_vp]),
    "sglm_pb_epilogue_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "sglm_pb_epilogue_f64": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                     c_i32, c_vp, c_vp, c_sz, c_vp]),
    "sglm_pb_state_words": (c_i32, []),
    "sglm_pb_step_f64": (c_i32, [c_vp, c_vp, c_vp]),
    "sglm_pb_enet_workspace_bytes": (c_sz, [c_i32, c_i64, c_i32]),
    "sglm_pb_step_enet_f64": (c_i32, [c_vp, c_vp, c_vp, c_vp, c_i32, c_vp, c_sz, c_vp, c_vp]),
    "sglm_col_moments_workspace_bytes": (c_sz, [c_i64, c_i32]),
    "sglm_col_moments_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_i32, c_i32, c_vp, c_vp, c_vp, c_sz, c_vp]),
    "sglm_zscore_apply_f64": (c_i32, [c_vp, c_i64, c_i64, c_i32, c_vp, c_vp, c_vp, c_i64, c_vp]),
    "sglm_diff1_f64": (c_i32, [c_vp, c_i64, c_i64, c_vp, c_i32, c_vp, c_i64, c_vp]),
    "sglm_rolling_minmax_f64": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i32, c_vp, c_vp]),
    "sglm_probe_mma_i8": (c_i32, [c_i32, c_vp, c_vp]),
    "sglm_probe_read_f64": (c_i32, [c_vp, c_i64, c_i32, c_i32, c_vp, c_vp]),
    "sglm_poisson_irls_prepare_f64": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_vp,
                                              c_vp, c_vp, c_vp, c_vp]),
    "sglm_score_glm_f64": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_f64, c_vp, c_vp,
                                   c_vp, c_vp]),
    "sglm_glm_irls_prepare_f64": (c_i32, [c_vp, c_i64, c_vp, c_vp, c_i64, c_i32, c_vp, c_vp, c_f64, c_vp,
                                          c_vp, c_vp, c_vp, c_vp]),
    "sglm_glm_epilogue_f64": (c_i32, [c_vp, c_i64, c_i32, c_i64, c_vp, c_i64, c_vp, c_vp, c_i64, c_vp, c_vp, c_vp, c_vp,
                                      c_f64, c_i32, c_vp, c_vp, c_sz, c_vp]),
}

_lib = None
_lock = threading.Lock()
_launches = 0          # number of kernel-launching ABI calls made through this binding (bench.py reads it)


class SglmNativeError(RuntimeError):
    pass


def lib():
    """Load libsglm_b200.so (once).  Raises if it has not been built."""
    global _lib
    with _lock:
        if _lib is None:
            if not os.path.exists(LIB_PATH):
                raise SglmNativeError(
                    f"{LIB_PATH} is missing: build it with `python __graft_entry__.py` "
                    "(nvcc, sm_100a).  There is no CPU fallback.")
            handle = ctypes.CDLL(LIB_PATH)
            for name, (res, args) in _PROTOTYPES.items():
                fn = getattr(handle, name)
                fn.restype = res
                fn.argtypes = args
            _lib = handle
    return _lib


def exported_symbols():
    return sorted(_PROTOTYPES)


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise SglmNativeError("sglm_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
    return torch


def stream_ptr():
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def ptr(t):
    """Device pointer of a torch tensor (or None)."""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr())


# kernels launched per ABI call (for the launch count bench.py reports)
_KERNELS_PER_CALL = {"sglm_suffstats_f64": 3, "sglm_gram_tc_analyze_f64": 2, "sglm_gram_tc_f64": 4, "sglm_gram_tc_cells_f64": 5,
                     "sglm_gram_tc_lag_cells_f64": 7, "sglm_gram_tc_cells_partial_f64": 4, "sglm_gram_tc_scaled_partial_f64": 4, "sglm_gram_tc_scaled_f64": 4,
                     "sglm_gram_tc_analyze_scaled_f64": 2, "sglm_quadform_gemm_f64": 3, "sglm_xt_vec_f64": 2, "sglm_score_f64": 2,
                     "sglm_poisson_irls_prepare_f64": 2, "sglm_timeshift_f64": 2, "sglm_pb_xt_r_f64": 2, "sglm_pb_epilogue_f64": 2,
                     "sglm_glm_epilogue_f64": 2, "sglm_score_glm_f64": 2, "sglm_glm_irls_prepare_f64": 2,
                     "sglm_pb_step_f64": 3, "sglm_pb_step_enet_f64": 6, "sglm_lag_valid_rows": 3, "sglm_col_moments_f64": 4, "sglm_mask_compact_rows": 3}
_timing = None         # when enabled: list of (name, start_event, end_event) on the current stream


def enable_timing(on=True):
    """Bracket every ABI call with CUDA events on the launching stream (bench.py only)."""
    global _timing
    _timing = [] if on else None


def collect_timing():
    """-> {entry point: (calls, total ms)}; synchronises.  Clears the record."""
    import torch
    global _timing
    global last_intervals
    out = {}
    if _timing:
        torch.cuda.synchronize()
        ref = _timing[0][1]
        global _first_event
        _first_event = ref
        last_intervals = []
        for name, e0, e1 in _timing:
            c, t = out.get(name, (0, 0.0))
            out[name] = (c + 1, t + e0.elapsed_time(e1))
            a = ref.elapsed_time(e0)
            last_intervals.append((name, a, a + e0.elapsed_time(e1)))
        _timing = []
    return out


_first_event = None
last_intervals = []     # (entry point, start ms, end ms) of the calls of the last collect_timing(), relative to its first call


def union_ms(names):
    """Total time covered by the calls of `names` in the last collected record (calls on different
    streams overlap: the coordinate-descent parts of one grid run concurrently)."""
    iv = sorted((a, b) for n, a, b in last_intervals if n in names)
    total, cur_a, cur_b = 0.0, None, None
    for a, b in iv:
        if cur_b is None or a > cur_b:
            if cur_b is not None:
                total += cur_b - cur_a
            cur_a, cur_b = a, b
        else:
            cur_b = max(cur_b, b)
    if cur_b is not None:
        total += cur_b - cur_a
    return total


last_tc_plan = None     # {S, n_pos, tiles, segs} of the most recent tensor-core Gram (bench.py reads it)


def call(name, *args):
    """Invoke an int-returning entry point; raise with sglm_last_error() on failure."""
    global _launches
    if _timing is not None:
        import torch
        e0 = torch.cuda.Event(enable_timing=True)
        e1 = torch.cuda.Event(enable_timing=True)
        e0.record()
    rc = getattr(lib(), name)(*args)
    if rc != 0:
        msg = lib().sglm_last_error()
        raise SglmNativeError(f"{name} failed (code {rc}): {msg.decode() if msg else ''}")
    if _timing is not None:
        e1.record()
        _timing.append((name, e0, e1))
    _launches += _KERNELS_PER_CALL.get(name, 1)
    return rc


def launches():
    return _launches


class LagDesignStruct(ctypes.Structure):
    """sglm_lag_design of include/sglm_b200.h."""
    _fields_ = [("base", ctypes.c_void_p), ("ldb", ctypes.c_int64), ("n_u", ctypes.c_int64), ("P", ctypes.c_int32),
                ("src_host", ctypes.c_void_p), ("off_host", ctypes.c_void_p), ("baseE", ctypes.c_void_p),
                ("baseS", ctypes.c_void_p), ("baseS_host", ctypes.c_void_p)]


NAN_BITS = int(np.array([np.nan], dtype=np.float64).view(np.uint64)[0])


def f64_bits(value):
    return int(np.array([value], dtype=np.float64).view(np.uint64)[0])
