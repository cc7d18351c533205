"""B200-native dense revised simplex: the hot path of Girjoaba/simplex_method_gpu
(the per-pivot loop of src/v4_cub_reduction.cu:286-359) as hand-written sm_100a
kernels behind a C ABI (include/b200lp.h)."""
from . import capi  # noqa: F401
from .solver import (EPS, MAX_ITER, REAL, BatchSolution, Engine, Solution, SolveStatus, format_result, read_lp,  # noqa: F401
                     set_memory_cache, solve, solve_batch, write_lp)

__all__ = ["solve", "solve_batch", "BatchSolution", "Engine", "Solution", "SolveStatus", "read_lp", "write_lp", "format_result", "set_memory_cache", "EPS", "MAX_ITER", "REAL"]
