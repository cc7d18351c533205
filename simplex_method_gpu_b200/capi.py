"""ctypes binding of include/b200lp.h — the same stub a maintainer of the reference
would add to call the engine instead of its solve() (src/v4_cub_reduction.cu:219).
Fails loudly when the native library is missing: there is no Python/CPU fallback."""
from __future__ import annotations

import ctypes as C
import os

from ._build import LIB_PATH

STATUS_MAX_ITER, STATUS_OPTIMUM, STATUS_UNBOUNDED, STATUS_THETA_OVERFLOW = 0, 1, 2, 3
STATUS_INFEASIBLE, STATUS_NOT_DUAL_FEASIBLE = 4, 5      # dual simplex (options.algorithm = 1) only
OK, ERR_ARG, ERR_CUDA, ERR_NO_GPU, ERR_STATE = 0, -1, -2, -3, -4
F32, F64 = 0, 1

EXPORTS = [
    "b200lp_default_options", "b200lp_solve_f64", "b200lp_solve_f32", "b200lp_create", "b200lp_destroy",
    "b200lp_set_memory_cache",
    "b200lp_upload", "b200lp_generate_dense", "b200lp_reset", "b200lp_run", "b200lp_run_async", "b200lp_wait",
    "b200lp_download", "b200lp_download_binv", "b200lp_download_trace", "b200lp_phase_price",
    "b200lp_phase_update_ftran", "b200lp_phase_ratio", "b200lp_phase_pivot_update", "b200lp_download_vector",
    "b200lp_stream", "b200lp_grid_ctas", "b200lp_dense_columns", "b200lp_bytes_per_pivot",
    "b200lp_last_error", "b200lp_version",
    "b200lp_create_sharded", "b200lp_ipc_handle_bytes", "b200lp_ipc_export", "b200lp_ipc_import", "b200lp_shard_rows",
    "b200lp_shard_columns", "b200lp_upload_columns", "b200lp_lpgen_dense_host",
    "b200lp_profile_stamps", "b200lp_profile_names", "b200lp_download_profile", "b200lp_check_basis",
    "b200lp_solve_f64_multi", "b200lp_solve_f32_multi", "b200lp_create_multi", "b200lp_abort",
    "b200lp_refactor", "b200lp_run_guarded", "b200lp_sizeof_options", "b200lp_sizeof_result",
    "b200lp_solve_batch_f64", "b200lp_solve_batch_f32", "b200lp_phase_info",
    # include/b200lp_io.h
    "b200lp_read_lp", "b200lp_write_lp_text", "b200lp_write_lp_binary", "b200lp_free_problem",
]


class Options(C.Structure):
    _fields_ = [("eps", C.c_double), ("max_iter", C.c_int64), ("device", C.c_int32), ("grid_ctas", C.c_int32),
                ("tile_shape", C.c_int32), ("check_slack", C.c_int32), ("mode", C.c_int32), ("profile", C.c_int32),
                ("price_cols", C.c_int32), ("l2_persist_mb", C.c_int32),
                ("price_mode", C.c_int32), ("ratio_group_rows", C.c_int32), ("pivot_tol", C.c_double),
                ("price_tail", C.c_int32), ("fuse_book2", C.c_int32), ("fuse_ratio", C.c_int32),
                ("pricing_rule", C.c_int32), ("ratio_mode", C.c_int32), ("resident", C.c_int32),
                ("harris_delta", C.c_double), ("algorithm", C.c_int32),
                ("cost_shift", C.c_int32), ("shift_delta", C.c_double)]


class Result(C.Structure):
    _fields_ = [("status", C.c_int32), ("aborted", C.c_int32), ("iterations", C.c_int64), ("pivots", C.c_int64),
                ("z", C.c_double), ("min_reduced_cost", C.c_double), ("ms_upload", C.c_double),
                ("ms_solve", C.c_double), ("ms_download", C.c_double), ("kernel_launches", C.c_int64)]


class Problem(C.Structure):
    """b200lp_problem (include/b200lp_io.h)."""
    _fields_ = [("dtype", C.c_int32), ("reserved", C.c_int32), ("m", C.c_int64), ("n", C.c_int64),
                ("A", C.c_void_p), ("b", C.c_void_p), ("c", C.c_void_p)]


class B200LPError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"b200lp error {code}: {msg}")
        self.code = code


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the engine has no CPU fallback)")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32, dbl = C.c_void_p, C.c_int64, C.c_int32, C.c_double
    PO, PR = C.POINTER(Options), C.POINTER(Result)
    sig = {
        "b200lp_default_options": (None, [PO]),
        "b200lp_solve_f64": (C.c_int, [vp, vp, vp, i64, i64, PO, vp, vp, vp, i64, PR]),
        "b200lp_solve_f32": (C.c_int, [vp, vp, vp, i64, i64, PO, vp, vp, vp, i64, PR]),
        "b200lp_solve_f64_multi": (C.c_int, [vp, vp, vp, i64, i64, PO, C.POINTER(i32), i32, vp, vp, vp, i64, PR]),
        "b200lp_solve_f32_multi": (C.c_int, [vp, vp, vp, i64, i64, PO, C.POINTER(i32), i32, vp, vp, vp, i64, PR]),
        "b200lp_solve_batch_f64": (C.c_int, [vp, vp, vp, i64, i64, i64, PO, vp, vp, vp, vp, i64, vp]),
        "b200lp_solve_batch_f32": (C.c_int, [vp, vp, vp, i64, i64, i64, PO, vp, vp, vp, vp, i64, vp]),
        "b200lp_create_multi": (C.c_int, [i32, i64, i64, C.POINTER(i32), i32, PO, C.POINTER(vp)]),
        "b200lp_abort": (C.c_int, [vp]),
        "b200lp_refactor": (C.c_int, [vp, dbl, C.POINTER(i64)]),
        "b200lp_run_guarded": (C.c_int, [vp, i64, i64, dbl, PR, C.POINTER(i64)]),
        "b200lp_set_memory_cache": (C.c_int, [i32]),
        "b200lp_create": (C.c_int, [i32, i64, i64, PO, C.POINTER(vp)]),
        "b200lp_destroy": (C.c_int, [vp]),
        "b200lp_upload": (C.c_int, [vp, vp, vp, vp]),
        "b200lp_generate_dense": (C.c_int, [vp, C.c_uint64]),
        "b200lp_reset": (C.c_int, [vp]),
        "b200lp_run": (C.c_int, [vp, i64, PR]),
        "b200lp_run_async": (C.c_int, [vp, i64]),
        "b200lp_wait": (C.c_int, [vp, PR]),
        "b200lp_phase_info": (C.c_int, [vp, C.POINTER(i32), C.POINTER(i64), C.POINTER(i64)]),
        "b200lp_download": (C.c_int, [vp, vp, vp, vp]),
        "b200lp_download_binv": (C.c_int, [vp, vp]),
        "b200lp_download_trace": (C.c_int, [vp, vp, i64, C.POINTER(i64)]),
        "b200lp_phase_price": (C.c_int, [vp, C.POINTER(i64), C.POINTER(dbl)]),
        "b200lp_phase_update_ftran": (C.c_int, [vp, i64]),
        "b200lp_phase_ratio": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64)]),
        "b200lp_phase_pivot_update": (C.c_int, [vp, i64, i64]),
        "b200lp_download_vector": (C.c_int, [vp, i32, vp]),
        "b200lp_stream": (vp, [vp]),
        "b200lp_grid_ctas": (C.c_int, [vp]),
        "b200lp_dense_columns": (C.c_int, [vp]),
        "b200lp_bytes_per_pivot": (i64, [vp]),
        "b200lp_create_sharded": (C.c_int, [i32, i64, i64, i32, i32, PO, C.POINTER(vp)]),
        "b200lp_ipc_handle_bytes": (C.c_int, []),
        "b200lp_ipc_export": (C.c_int, [vp, vp]),
        "b200lp_ipc_import": (C.c_int, [vp, vp, i32]),
        "b200lp_shard_rows": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64)]),
        "b200lp_shard_columns": (C.c_int, [vp, C.POINTER(i64), C.POINTER(i64)]),
        "b200lp_upload_columns": (C.c_int, [vp, vp, i64, i64, vp, vp]),
        "b200lp_lpgen_dense_host": (C.c_int, [i32, vp, vp, vp, i64, i64, i64, i64, C.c_uint64]),
        "b200lp_check_basis": (C.c_int, [vp, C.POINTER(dbl), C.POINTER(dbl)]),
        "b200lp_profile_stamps": (C.c_int, []),
        "b200lp_profile_names": (C.c_char_p, []),
        "b200lp_download_profile": (C.c_int, [vp, vp, i64, C.POINTER(i64)]),
        "b200lp_read_lp": (C.c_int, [C.c_char_p, i32, i32, C.POINTER(Problem)]),
        "b200lp_write_lp_text": (C.c_int, [C.c_char_p, C.POINTER(Problem)]),
        "b200lp_write_lp_binary": (C.c_int, [C.c_char_p, C.POINTER(Problem)]),
        "b200lp_free_problem": (None, [C.POINTER(Problem)]),
        "b200lp_last_error": (C.c_char_p, []),
        "b200lp_version": (C.c_char_p, []),
        "b200lp_sizeof_options": (C.c_int, []),
        "b200lp_sizeof_result": (C.c_int, []),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    if L.b200lp_sizeof_options() != C.sizeof(Options) or L.b200lp_sizeof_result() != C.sizeof(Result):
        raise ImportError("capi.Options / capi.Result do not mirror include/b200lp.h of the library that was loaded "
                          f"({C.sizeof(Options)} / {C.sizeof(Result)} bytes here, "
                          f"{L.b200lp_sizeof_options()} / {L.b200lp_sizeof_result()} in {LIB_PATH}): rebuild")
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != OK:
        raise B200LPError(rc, lib().b200lp_last_error().decode())


def default_options(**kw) -> Options:
    o = Options()
    lib().b200lp_default_options(C.byref(o))
    for k, v in kw.items():
        if not hasattr(o, k):
            raise TypeError(f"unknown option {k}")
        setattr(o, k, v)
    return o
