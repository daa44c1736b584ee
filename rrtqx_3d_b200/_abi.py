"""ctypes binding of librrtqx_b200.so (include/rrtqx_b200.h).

This is the Python twin of julia/RRTQXGpu.jl's `ccall` layer: one thin function
per C entry point, numpy arrays (or raw device pointers) in, numpy arrays out.
There is no fallback: if the shared library is missing this module raises at
import of the first symbol, and if no B200 is present `Context()` raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# RRTQX_B200_LIB: alternative build of the same CUDA library (kernel experiments); never a non-CUDA fallback
LIB_PATH = os.environ.get("RRTQX_B200_LIB") or os.path.join(_HERE, "librrtqx_b200.so")

OK = 0
ERR_INVALID, ERR_CUDA, ERR_NOMEM, ERR_EMPTY_TREE, ERR_UNSUPPORTED, ERR_STATE = 1, 2, 3, 4, 5, 6
RANGE_WANT_DIST, RANGE_COUNT_ONLY = 1, 2
CHECK_FMA_DOT, CHECK_IGNORE_ACTIVE, CHECK_QUICK_PASS = 1, 2, 4
SWEEP_REMOVED_INACTIVE = 16
SWEEP_STATS = 32
EXTEND_SATURATE = 8

vp = C.c_void_p
i32, i64, u32, f64 = C.c_int32, C.c_int64, C.c_uint32, C.c_double

# name -> (restype, argtypes); must list every RRTQX_API symbol of the header
SIGNATURES = {
    "rrtqx_version": (C.c_char_p, []),
    "rrtqx_ctx_create": (i32, [i32, vp, C.POINTER(vp)]),
    "rrtqx_ctx_destroy": (i32, [vp]),
    "rrtqx_last_error": (C.c_char_p, [vp]),
    "rrtqx_ctx_reload_tuning": (i32, [vp]),
    "rrtqx_host_alloc": (i32, [vp, i64, C.POINTER(vp)]),
    "rrtqx_host_free": (i32, [vp, vp]),
    "rrtqx_ctx_sync": (i32, [vp]),
    "rrtqx_ctx_kernel_launches": (i32, [vp, C.POINTER(i64)]),
    "rrtqx_ctx_last_phase_ms": (i32, [vp, C.c_char_p, C.POINTER(C.c_float)]),
    "rrtqx_ctx_measure_fp64_peak": (i32, [vp, C.POINTER(f64)]),
    "rrtqx_tree_create": (i32, [vp, i32, i32, vp, vp, C.POINTER(vp)]),
    "rrtqx_tree_destroy": (i32, [vp]),
    "rrtqx_tree_insert_batch": (i32, [vp, vp, i64, C.POINTER(i32)]),
    "rrtqx_tree_insert": (i32, [vp, vp, C.POINTER(i32)]),
    "rrtqx_tree_size": (i32, [vp, C.POINTER(i64)]),
    "rrtqx_tree_kd_fields": (i32, [vp, i64, i64, vp, vp, vp, vp]),
    "rrtqx_tree_positions": (i32, [vp, i64, i64, vp]),
    "rrtqx_tree_preorder": (i32, [vp, vp]),
    "rrtqx_tree_set_cell_occupancy": (i32, [vp, f64]),
    "rrtqx_tree_reindex": (i32, [vp]),
    "rrtqx_range_query_batch": (i32, [vp, vp, i64, f64, vp, u32, C.POINTER(vp), C.POINTER(i64)]),
    "rrtqx_range_result_destroy": (i32, [vp]),
    "rrtqx_range_result_sizes": (i32, [vp, C.POINTER(i64), C.POINTER(i64)]),
    "rrtqx_range_result_layout": (i32, [vp, vp, vp]),
    "rrtqx_range_result_fetch": (i32, [vp, vp, vp]),
    "rrtqx_range_result_device": (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
    "rrtqx_nearest_batch": (i32, [vp, vp, i64, vp, vp]),
    "rrtqx_extend_query": (i32, [vp, vp, vp, f64, f64, u32, i32, C.POINTER(i32), C.POINTER(f64), C.POINTER(C.c_uint8),
                                 C.POINTER(f64), C.POINTER(i32), vp, vp, vp, vp]),
    "rrtqx_extend_query_dubins": (i32, [vp, vp, vp, f64, f64, f64, f64, u32, i32, C.POINTER(i32), C.POINTER(f64),
                                        C.POINTER(i32), vp, vp, vp, vp, vp, C.POINTER(vp)]),
    "rrtqx_spheres_create": (i32, [vp, C.POINTER(vp)]),
    "rrtqx_spheres_destroy": (i32, [vp]),
    "rrtqx_spheres_upload": (i32, [vp, vp, vp, vp, i64]),
    "rrtqx_spheres_update": (i32, [vp, i64, i64, vp, vp]),
    "rrtqx_spheres_size": (i32, [vp, C.POINTER(i64)]),
    "rrtqx_edge_check_batch": (i32, [vp, vp, vp, vp, i64, f64, u32, vp]),
    "rrtqx_segment_check_batch": (i32, [vp, vp, vp, vp, i64, f64, u32, vp]),
    "rrtqx_node_check_batch": (i32, [vp, vp, vp, i64, f64, u32, vp, vp]),
    "rrtqx_edges_create": (i32, [vp, C.POINTER(vp)]),
    "rrtqx_edges_destroy": (i32, [vp]),
    "rrtqx_edges_upload": (i32, [vp, vp, vp, i64, vp, i64]),
    "rrtqx_edges_size": (i32, [vp, C.POINTER(i64)]),
    "rrtqx_edges_check_batch": (i32, [vp, vp, f64, u32, vp]),
    "rrtqx_edges_append": (i32, [vp, vp, vp, i64]),
    "rrtqx_edges_set_parents": (i32, [vp, vp, vp, i64]),
    "rrtqx_obstacle_add_sweep": (i32, [vp, vp, vp, i64, f64, f64, u32, C.POINTER(vp)]),
    "rrtqx_obstacle_remove_sweep": (i32, [vp, vp, i32, vp, i64, vp, f64, f64, u32, C.POINTER(vp)]),
    "rrtqx_comm_init_local": (i32, [vp, i32, C.POINTER(vp)]),
    "rrtqx_comm_unique_id": (i32, [vp]),
    "rrtqx_comm_init_rank": (i32, [vp, vp, i32, i32, C.POINTER(vp)]),
    "rrtqx_comm_destroy": (i32, [vp]),
    "rrtqx_comm_info": (i32, [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]),
    "rrtqx_comm_allgather": (i32, [vp, vp, vp, i64, i32]),
    "rrtqx_comm_join": (i32, [vp]),
    "rrtqx_comm_packed_words": (i32, [vp, i64, C.POINTER(i64), C.POINTER(i64)]),
    "rrtqx_edge_check_batch_sharded": (i32, [vp, vp, vp, vp, vp, i64, f64, u32, vp]),
    "rrtqx_edges_set_trajectories": (i32, [vp, vp, vp]),
    "rrtqx_edges_solve_trajectories": (i32, [vp, f64, C.POINTER(i64)]),
    "rrtqx_edges_trajectories_device": (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(i64), C.POINTER(i64)]),
    "rrtqx_edges_trajectories_fetch": (i32, [vp, vp, vp]),
    "rrtqx_obstacle_add_sweep_2d": (i32, [vp, vp, vp, i64, f64, f64, f64, u32, C.POINTER(vp)]),
    "rrtqx_obstacle_remove_sweep_2d": (i32, [vp, vp, i32, vp, i64, vp, f64, f64, f64, u32, C.POINTER(vp)]),
    "rrtqx_sweep_result_destroy": (i32, [vp]),
    "rrtqx_sweep_result_sizes": (i32, [vp, C.POINTER(i64), C.POINTER(i64), C.POINTER(i64), C.POINTER(i64)]),
    "rrtqx_sweep_result_fetch": (i32, [vp, vp, vp]),
    "rrtqx_sweep_result_flags": (i32, [vp, vp, vp]),
    "rrtqx_polygons_create": (i32, [vp, C.POINTER(vp)]),
    "rrtqx_polygons_destroy": (i32, [vp]),
    "rrtqx_polygons_upload": (i32, [vp, vp, vp, vp, vp, vp, vp, i64]),
    "rrtqx_segment_check_2d_batch": (i32, [vp, vp, vp, i64, f64, u32, vp]),
    "rrtqx_dubins_edge_check_batch": (i32, [vp, vp, vp, vp, vp, i64, f64, f64, u32, vp]),
    "rrtqx_dubins_trajectory_batch": (i32, [vp, vp, vp, i64, f64, C.POINTER(vp)]),
    "rrtqx_dubins_result_destroy": (i32, [vp]),
    "rrtqx_dubins_result_sizes": (i32, [vp, C.POINTER(i64), C.POINTER(i64)]),
    "rrtqx_dubins_result_fetch": (i32, [vp, vp, vp, vp, vp]),
    "rrtqx_dubins_result_device": (i32, [vp, C.POINTER(vp), C.POINTER(vp), C.POINTER(vp), C.POINTER(vp)]),
    "rrtqx_dubins_saturate_batch": (i32, [vp, vp, vp, i64, f64]),
}

_lib = None


class RRTQXError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"rrtqx status {status}: {message}")
        self.status = status


def lib() -> C.CDLL:
    """Load the CUDA library; fail loudly when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(nvcc, sm_100a). There is no CPU fallback.")
        L = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def ptr(a) -> int | None:
    """Address of a numpy array / raw integer device pointer / None."""
    if a is None:
        return None
    if isinstance(a, (int, np.integer)):
        return int(a)
    if isinstance(a, np.ndarray):
        assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous"
        return a.ctypes.data
    if hasattr(a, "data_ptr"):  # torch tensor (device or host)
        assert a.is_contiguous()
        return int(a.data_ptr())
    raise TypeError(type(a))


def check(status: int, ctx_handle=None):
    if status != OK:
        msg = lib().rrtqx_last_error(ctx_handle)
        raise RRTQXError(status, (msg or b"").decode("utf-8", "replace"))


def as_f64(a, cols=None) -> np.ndarray:
    a = np.ascontiguousarray(a, dtype=np.float64)
    if cols is not None:
        a = a.reshape(-1, cols)
    return a


def as_i32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.int32)


def as_u8(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.uint8)
