"""Host-side mirror of the reference's solver interface for the hot path.

Reference contract (src/v4_cub_reduction.cu):
  * ``solve(A, b, c, x_b, b_ixs, m, n, t) -> (z, SolveStatus)``           v4:219
  * LP text format ``m n`` / A (m rows x n) / b / c, slack block last     v4:401-420, input/sample.txt
  * result printing                                                        v4:426-445
Everything numeric happens in libb200lp.so (hand-written sm_100a kernels); this
module only marshals numpy arrays across the C ABI.
"""
from __future__ import annotations

import ctypes as C
import enum
import io
from dataclasses import dataclass

import numpy as np

from . import capi


class SolveStatus(enum.IntEnum):
    """`enum class SolveStatus` (v4:49-54), plus the two outcomes only the dual simplex (algorithm=1) reports."""
    MaxIter = 0
    OptimumFound = 1
    Unbounded = 2
    ThetaOverflow = 3
    Infeasible = 4           # the constraints have no solution (row r of B^-1 is a Farkas certificate)
    NotDualFeasible = 5      # some reduced cost < -eps: the dual method cannot run from this basis


# reference compile-time constants (v4:12, 18-19)
REAL = np.float32
EPS = 1e-4
MAX_ITER = 5


@dataclass
class Solution:
    z: float
    status: SolveStatus
    x_b: np.ndarray          # basis-ordered values (v4:366)
    b_ixs: np.ndarray        # basis-ordered column indices (v4:367)
    iterations: int          # "# Iteration k" lines the reference prints (v4:287)
    pivots: int
    trace: np.ndarray        # (pivots, 2) int32: entering column p, leaving row q
    ms_upload: float = 0.0
    ms_solve: float = 0.0
    ms_download: float = 0.0
    kernel_launches: int = 0
    min_reduced_cost: float = 0.0

    def x(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=self.x_b.dtype)
        out[self.b_ixs] = self.x_b
        return out


def _dtype_code(dt) -> int:
    dt = np.dtype(dt)
    if dt == np.float32:
        return capi.F32
    if dt == np.float64:
        return capi.F64
    raise TypeError(f"real must be float32 or float64, got {dt}")


def _vp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _prep(A, b, c, dtype):
    dt = np.dtype(dtype if dtype is not None else A.dtype)
    _dtype_code(dt)
    A = np.asfortranarray(A, dtype=dt)      # column-major like the reference (v4:59-60, 98)
    if A.ndim != 2:
        raise ValueError("A must be a matrix")
    m, n = A.shape
    b = np.ascontiguousarray(b, dtype=dt).reshape(-1)
    c = np.ascontiguousarray(c, dtype=dt).reshape(-1)
    if b.size != m or c.size != n:
        raise ValueError(f"shape mismatch: A is {m}x{n}, b has {b.size}, c has {c.size}")
    if m > n:
        raise ValueError("Either failed to read m and n, or m > n.")   # v4:403
    return A, b, c, m, n, dt


def solve(A, b, c, eps: float = EPS, max_iter: int = MAX_ITER, dtype=None, device: int = 0,
          trace_cap: int | None = None, devices=None, **opts) -> Solution:
    """Drop-in for the reference's ``solve()`` (v4:219): host arrays in, host arrays out.
    ``devices``: list of CUDA ordinals -> b200lp_solve_*_multi (B^-1 row-sharded, A column-sharded over them).
    ``opts``: any field of b200lp_options, e.g. ``algorithm=1`` for the dual simplex (LPs with negative b and a
    dual feasible slack basis, such as c <= 0), ``algorithm=1, cost_shift=1`` for the composite method (LPs with
    negative b and positive c: the dual loop on shifted costs, then the primal loop)."""
    A, b, c, m, n, dt = _prep(A, b, c, dtype)
    L = capi.lib()
    o = capi.default_options(eps=eps, max_iter=int(max_iter), device=device, **opts)
    cap = int(trace_cap if trace_cap is not None else min(int(max_iter), 1 << 22))
    x_b = np.zeros(m, dt)
    b_ixs = np.zeros(m, np.int32)
    trace = np.full((max(cap, 1), 2), -1, np.int32)
    res = capi.Result()
    if devices is not None:
        devs = (C.c_int32 * len(devices))(*[int(x) for x in devices])
        fn = L.b200lp_solve_f64_multi if dt == np.float64 else L.b200lp_solve_f32_multi
        capi.check(fn(_vp(A), _vp(b), _vp(c), m, n, C.byref(o), devs, len(devices), _vp(x_b), _vp(b_ixs), _vp(trace), cap,
                      C.byref(res)))
    else:
        fn = L.b200lp_solve_f64 if dt == np.float64 else L.b200lp_solve_f32
        capi.check(fn(_vp(A), _vp(b), _vp(c), m, n, C.byref(o), _vp(x_b), _vp(b_ixs), _vp(trace), cap, C.byref(res)))
    k = min(res.pivots, cap)
    return Solution(res.z, SolveStatus(res.status), x_b, b_ixs, res.iterations, res.pivots, trace[:k].copy(),
                    res.ms_upload, res.ms_solve, res.ms_download, res.kernel_launches, res.min_reduced_cost)


@dataclass
class BatchSolution:
    """Outcome of solve_batch: arrays indexed by LP, the call's timings once."""
    z: np.ndarray                 # (batch,)
    status: np.ndarray            # (batch,) int32, SolveStatus values
    iterations: np.ndarray        # (batch,) int64
    pivots: np.ndarray            # (batch,) int64
    min_reduced_cost: np.ndarray  # (batch,)
    x_b: np.ndarray               # (batch, m) basis-ordered values
    b_ixs: np.ndarray             # (batch, m) basis-ordered column indices
    y: np.ndarray | None          # (batch, m) duals, None unless want_y
    trace: np.ndarray             # (batch, trace_cap, 2) int32 (p, q), -1 past an LP's pivots
    ms_upload: float = 0.0
    ms_solve: float = 0.0
    ms_download: float = 0.0
    kernel_launches: int = 0

    def __len__(self) -> int:
        return len(self.z)

    def solution(self, k: int) -> Solution:
        """LP k as the Solution of a single solve() (format_result works on it)."""
        k = int(k)
        piv = int(self.pivots[k])
        return Solution(float(self.z[k]), SolveStatus(int(self.status[k])), self.x_b[k].copy(), self.b_ixs[k].copy(),
                        int(self.iterations[k]), piv, self.trace[k, :min(piv, self.trace.shape[1])].copy(),
                        self.ms_upload, self.ms_solve, self.ms_download, self.kernel_launches,
                        float(self.min_reduced_cost[k]))


def solve_batch(A, b, c, eps: float = EPS, max_iter: int = MAX_ITER, dtype=None, device: int = 0, trace_cap: int = 0,
                want_y: bool = True, **opts) -> BatchSolution:
    """Many LPs of one shape in one call (b200lp_solve_batch_*): A is (batch, m, n), b (batch, m), c (batch, n).
    LP k's results are bit-identical to ``solve(A[k], b[k], c[k], ...)`` with the same options."""
    A = np.asarray(A)
    dt = np.dtype(dtype if dtype is not None else A.dtype)
    _dtype_code(dt)
    if A.ndim != 3:
        raise ValueError("A must be a stack of matrices (batch, m, n)")
    batch, m, n = A.shape
    At = np.ascontiguousarray(A.transpose(0, 2, 1), dtype=dt)     # every LP column-major (v4:59-60)
    b = np.ascontiguousarray(b, dtype=dt)
    c = np.ascontiguousarray(c, dtype=dt)
    if b.shape != (batch, m) or c.shape != (batch, n):
        raise ValueError(f"shape mismatch: A is {batch}x{m}x{n}, b is {'x'.join(map(str, b.shape))}, "
                         f"c is {'x'.join(map(str, c.shape))}")
    if m > n:
        raise ValueError("Either failed to read m and n, or m > n.")   # v4:403
    if batch == 0:
        raise ValueError("the batch is empty")
    cap = int(trace_cap)
    if cap < 0:
        raise ValueError("trace_cap must not be negative")
    L = capi.lib()
    o = capi.default_options(eps=eps, max_iter=int(max_iter), device=device, **opts)
    x_b = np.zeros((batch, m), dt)
    b_ixs = np.zeros((batch, m), np.int32)
    y = np.zeros((batch, m), dt) if want_y else None
    trace = np.full((batch, cap, 2), -1, np.int32)
    res = (capi.Result * batch)()
    fn = L.b200lp_solve_batch_f64 if dt == np.float64 else L.b200lp_solve_batch_f32
    capi.check(fn(_vp(At), _vp(b), _vp(c), batch, m, n, C.byref(o), _vp(x_b), _vp(b_ixs), _vp(y),
                  _vp(trace) if cap > 0 else None, cap, res))
    r0 = res[0]
    return BatchSolution(z=np.array([r.z for r in res]), status=np.array([r.status for r in res], np.int32),
                         iterations=np.array([r.iterations for r in res], np.int64),
                         pivots=np.array([r.pivots for r in res], np.int64),
                         min_reduced_cost=np.array([r.min_reduced_cost for r in res]),
                         x_b=x_b, b_ixs=b_ixs, y=y, trace=trace, ms_upload=r0.ms_upload, ms_solve=r0.ms_solve,
                         ms_download=r0.ms_download, kernel_launches=r0.kernel_launches)


def set_memory_cache(on: bool) -> bool:
    """Keep the device buffers of the last solve() for the next call of the same shape (b200lp_set_memory_cache)."""
    return bool(capi.lib().b200lp_set_memory_cache(1 if on else 0))


class Engine:
    """Handle API: device state survives between calls (benchmark windows, phase tests)."""

    def __init__(self, m: int, n: int, dtype=np.float64, eps: float = EPS, max_iter: int = MAX_ITER,
                 device: int = 0, devices=None, binv_sparse: int = 0, **opts):
        """``devices``: list of CUDA ordinals -> one handle over several GPUs of this process (b200lp_create_multi).
        ``binv_sparse``: touched-column passes over B^-1 (b200lp_set_binv_sparse): 0 auto, -1 off, > 0 the largest
        touched-column count they run at."""
        self.m, self.n, self.dtype = int(m), int(n), np.dtype(dtype)
        self._L = capi.lib()
        self._o = capi.default_options(eps=eps, max_iter=int(max_iter), device=device, **opts)
        self._h = C.c_void_p()
        if devices is not None:
            devs = (C.c_int32 * len(devices))(*[int(x) for x in devices])
            capi.check(self._L.b200lp_create_multi(_dtype_code(self.dtype), self.m, self.n, devs, len(devices),
                                                   C.byref(self._o), C.byref(self._h)))
        else:
            capi.check(self._L.b200lp_create(_dtype_code(self.dtype), self.m, self.n, C.byref(self._o), C.byref(self._h)))
        if binv_sparse != 0:
            self.set_binv_sparse(binv_sparse)

    def set_binv_sparse(self, k: int):
        """Touched-column passes over B^-1 from the next run on: 0 auto, -1 off, > 0 while at most k columns are touched."""
        capi.check(self._L.b200lp_set_binv_sparse(self._h, int(k)))

    def binv_info(self) -> dict:
        """Touched columns of B^-1 since the last reset / refactor and the update passes that streamed only them."""
        k, n = C.c_int64(0), C.c_int64(0)
        capi.check(self._L.b200lp_binv_info(self._h, C.byref(k), C.byref(n)))
        return {"touched": k.value, "sparse_passes": n.value}

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.b200lp_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- data
    def upload(self, A, b, c):
        A, b, c, m, n, dt = _prep(A, b, c, self.dtype)
        if (m, n) != (self.m, self.n):
            raise ValueError("problem size differs from the engine's")
        capi.check(self._L.b200lp_upload(self._h, _vp(A), _vp(b), _vp(c)))

    def upload_raw(self, A_ptr: int, b_ptr: int, c_ptr: int):
        """Host pointers of the engine's dtype (e.g. pinned torch tensors), no copies made here."""
        capi.check(self._L.b200lp_upload(self._h, C.c_void_p(A_ptr), C.c_void_p(b_ptr), C.c_void_p(c_ptr)))

    def generate_dense(self, seed: int = 1):
        capi.check(self._L.b200lp_generate_dense(self._h, seed))

    def reset(self):
        capi.check(self._L.b200lp_reset(self._h))

    # -- loop
    def _result(self, res) -> dict:
        return {"status": SolveStatus(res.status), "aborted": bool(res.aborted), "iterations": res.iterations,
                "pivots": res.pivots, "z": res.z,
                "min_reduced_cost": res.min_reduced_cost, "ms_solve": res.ms_solve, "ms_upload": res.ms_upload,
                "kernel_launches": res.kernel_launches}

    def run(self, iterations: int) -> dict:
        res = capi.Result()
        capi.check(self._L.b200lp_run(self._h, int(iterations), C.byref(res)))
        return self._result(res)

    def run_async(self, iterations: int):
        capi.check(self._L.b200lp_run_async(self._h, int(iterations)))

    def wait(self) -> dict:
        res = capi.Result()
        capi.check(self._L.b200lp_wait(self._h, C.byref(res)))
        return self._result(res)

    def phase_info(self) -> dict:
        """Composite method (cost_shift=1): phase 0 (not started), 1 (dual loop on the shifted costs) or 2 (primal loop
        on the original costs), the number of shifted columns and the pivots of phase 1 (b200lp_phase_info)."""
        ph, k, p1 = C.c_int32(0), C.c_int64(0), C.c_int64(0)
        capi.check(self._L.b200lp_phase_info(self._h, C.byref(ph), C.byref(k), C.byref(p1)))
        return {"phase": ph.value, "shifted_columns": k.value, "phase1_pivots": p1.value}

    def refactor(self, rel_pivot_tol: float = 0.0) -> int:
        """Rebuild B^-1, x_b and y from the current basis (b200lp_refactor); returns the number of replayed pivots."""
        k = C.c_int64(0)
        capi.check(self._L.b200lp_refactor(self._h, float(rel_pivot_tol), C.byref(k)))
        return k.value

    def run_guarded(self, iterations: int, window: int, drift_tol: float):
        """run() in windows with a drift check and a refactorisation when needed -> (result, refactorisations)."""
        res, k = capi.Result(), C.c_int64(0)
        capi.check(self._L.b200lp_run_guarded(self._h, int(iterations), int(window), float(drift_tol), C.byref(res), C.byref(k)))
        return self._result(res), k.value

    def abort(self):
        """Ask a running loop to stop at its next iteration boundary (b200lp_abort); pair with wait()."""
        capi.check(self._L.b200lp_abort(self._h))

    # -- results
    def download(self):
        x_b = np.zeros(self.m, self.dtype)
        y = np.zeros(self.m, self.dtype)
        b_ixs = np.zeros(self.m, np.int32)
        capi.check(self._L.b200lp_download(self._h, _vp(x_b), _vp(b_ixs), _vp(y)))
        return x_b, b_ixs, y

    def download_binv(self) -> np.ndarray:
        B = np.zeros((self.m, self.m), self.dtype, order="F")
        capi.check(self._L.b200lp_download_binv(self._h, _vp(B)))
        return B

    def trace(self, cap: int = 1 << 22) -> np.ndarray:
        buf = np.full((cap, 2), -1, np.int32)
        k = C.c_int64(0)
        capi.check(self._L.b200lp_download_trace(self._h, _vp(buf), cap, C.byref(k)))
        return buf[:k.value].copy()

    def vector(self, name: str) -> np.ndarray:
        which = {"alpha": 0, "E_q": 1, "row_q": 2, "x_b": 3, "y": 4, "c_b": 5, "vbt": 6, "gamma": 7}[name]
        out = np.zeros(self.n if name == "gamma" else self.m, self.dtype)
        capi.check(self._L.b200lp_download_vector(self._h, which, _vp(out)))
        return out

    def check_basis(self):
        """(max |B^-1 b - x_b|, max |x_b|): drift between the product-form inverse and the linearly updated x_b."""
        err, scale = C.c_double(0), C.c_double(0)
        capi.check(self._L.b200lp_check_basis(self._h, C.byref(err), C.byref(scale)))
        return err.value, scale.value

    def profile(self, cap: int = 1 << 16) -> np.ndarray:
        """Phase time stamps (ns) of the last persistent launch, shape (iterations, stamps); needs profile=N."""
        ns = self._L.b200lp_profile_stamps()
        buf = np.zeros((cap, ns), np.uint64)
        k = C.c_int64(0)
        capi.check(self._L.b200lp_download_profile(self._h, _vp(buf), cap, C.byref(k)))
        return buf[:k.value].copy()

    # -- single phases
    def phase_price(self):
        p, mn = C.c_int64(0), C.c_double(0)
        capi.check(self._L.b200lp_phase_price(self._h, C.byref(p), C.byref(mn)))
        return p.value, mn.value

    def phase_update_ftran(self, p: int):
        capi.check(self._L.b200lp_phase_update_ftran(self._h, int(p)))

    def phase_ratio(self):
        q, el = C.c_int64(0), C.c_int64(0)
        capi.check(self._L.b200lp_phase_ratio(self._h, C.byref(q), C.byref(el)))
        return q.value, el.value

    def phase_pivot_update(self, p: int, q: int):
        capi.check(self._L.b200lp_phase_pivot_update(self._h, int(p), int(q)))

    # -- introspection
    @property
    def stream(self) -> int:
        return int(self._L.b200lp_stream(self._h) or 0)

    @property
    def grid_ctas(self) -> int:
        return self._L.b200lp_grid_ctas(self._h)

    @property
    def dense_columns(self) -> int:
        return self._L.b200lp_dense_columns(self._h)

    @property
    def bytes_per_pivot(self) -> int:
        return self._L.b200lp_bytes_per_pivot(self._h)


def lpgen_dense_into(A_ptr, b_ptr, c_ptr, m, n, col0, ncols, seed, dtype=np.float64):
    """Fill caller-owned host memory (e.g. pinned) with columns [col0, col0+ncols) of the synthetic dense LP."""
    vp = lambda p: C.c_void_p(int(p)) if p else None
    capi.check(capi.lib().b200lp_lpgen_dense_host(_dtype_code(dtype), vp(A_ptr), vp(b_ptr), vp(c_ptr), m, n, col0, ncols, seed))


def lpgen_dense(m, n, seed=1, dtype=np.float64):
    """Synthetic dense LP of the benchmark configurations (full [A_s, I] matrix, column-major)."""
    dt = np.dtype(dtype)
    A = np.empty((m, n), dt, order="F")
    b = np.empty(m, dt)
    c = np.empty(n, dt)
    lpgen_dense_into(A.ctypes.data, b.ctypes.data, c.ctypes.data, m, n, 0, n, seed, dt)
    return A, b, c


# ---------------------------------------------------------------- text format + printing

def _round_once_f32(tok: str, x: float) -> np.float32:
    """Decimal token -> float32 rounded ONCE, like the reference's ``operator>>(float)`` (v4:94-104).  ``x`` is the
    correctly rounded double of the token; casting it is wrong only when it sits exactly on the midpoint of two
    neighbouring floats while the decimal itself does not — decided with exact rational arithmetic."""
    f = np.float32(x)
    if not np.isfinite(f) or float(f) == x:
        return f
    other = np.nextafter(f, np.float32(np.inf) if x > float(f) else np.float32(-np.inf))
    if not np.isfinite(other) or (float(f) + float(other)) / 2 != x:
        return f
    try:
        from fractions import Fraction
        exact, mid = Fraction(tok), Fraction(x)
    except (ValueError, ZeroDivisionError):
        return f
    if exact == mid:
        return f                                    # a true tie: round-half-even already applied by the cast
    return f if (exact < mid) == (float(f) < float(other)) else other


def read_lp(path_or_file, dtype=REAL):
    """Parse the reference's LP text format (v4:401-420, input/sample.txt): ``m n``,
    A as m rows of n numbers, b (m), c (n); anything after that is ignored."""
    if hasattr(path_or_file, "read"):
        text = path_or_file.read()
    else:
        with open(path_or_file, "r") as f:
            text = f.read()
    toks = text.split()
    try:
        m, n = int(toks[0]), int(toks[1])
    except (IndexError, ValueError):
        raise ValueError("Either failed to read m and n, or m > n.")      # v4:403
    if m > n:
        raise ValueError("Either failed to read m and n, or m > n.")
    need = m * n + m + n
    vals = []
    for k, t in enumerate(toks[2:2 + need]):
        try:
            vals.append(float(t))
        except ValueError:
            break
    if len(vals) < need:
        k = len(vals)
        if k < m * n:
            raise ValueError(f"Failed to read ({k // n},{k % n}) for A")   # v4:99
        if k < m * n + m:
            raise ValueError(f"Failed to read ({k - m * n},0) for b")
        raise ValueError(f"Failed to read (0,{k - m * n - m}) for c")
    if np.dtype(dtype) == np.float32:
        v = np.array([_round_once_f32(t, x) for t, x in zip(toks[2:2 + need], vals)], dtype=np.float32)
    else:
        v = np.asarray(vals, dtype=np.float64)
    A = np.asfortranarray(v[:m * n].reshape(m, n), dtype=dtype)              # row-major text -> col-major
    b = v[m * n:m * n + m].astype(dtype)
    c = v[m * n + m:].astype(dtype)
    return A, b, c


def read_lp_native(path, dtype=REAL):
    """Same contract as read_lp, through the library's parallel reader (include/b200lp_io.h); also reads
    the binary twin of the format.  Raises ValueError with the reference's messages (v4:397-404, 99)."""
    dt = np.dtype(dtype)
    L = capi.lib()
    prob = capi.Problem()
    rc = L.b200lp_read_lp(str(path).encode(), _dtype_code(dt), 0, C.byref(prob))
    if rc != capi.OK:
        raise ValueError(L.b200lp_last_error().decode())
    try:
        m, n = prob.m, prob.n
        ct = C.c_double if dt == np.float64 else C.c_float
        A = np.ctypeslib.as_array(C.cast(prob.A, C.POINTER(ct)), shape=(n, m)).T.copy(order="F")
        b = np.ctypeslib.as_array(C.cast(prob.b, C.POINTER(ct)), shape=(m,)).copy()
        c = np.ctypeslib.as_array(C.cast(prob.c, C.POINTER(ct)), shape=(n,)).copy()
    finally:
        L.b200lp_free_problem(C.byref(prob))
    return A, b, c


def write_lp_native(path, A, b, c, binary=False):
    """Write the text format (shortest round-trip decimals) or the binary twin through the library."""
    A, b, c, m, n, dt = _prep(A, b, c, None)
    prob = capi.Problem(_dtype_code(dt), 0, m, n, A.ctypes.data, b.ctypes.data, c.ctypes.data)
    L = capi.lib()
    fn = L.b200lp_write_lp_binary if binary else L.b200lp_write_lp_text
    if fn(str(path).encode(), C.byref(prob)) != capi.OK:
        raise OSError(L.b200lp_last_error().decode())


def write_lp(path, A, b, c):
    m, n = A.shape
    with open(path, "w") as f:
        f.write(f"{m} {n}\n")
        for i in range(m):
            f.write(" ".join(repr(float(x)) for x in A[i]) + "\n")
        f.write(" ".join(repr(float(x)) for x in b) + "\n")
        f.write(" ".join(repr(float(x)) for x in c) + "\n")


def _cxx_float(x) -> str:
    """C++ ``ostream << real`` with default flags: %g with 6 significant digits."""
    return "%g" % float(x)


def format_result(sol: Solution) -> str:
    """The reference's stdout up to the timing block (v4:287, 426-445)."""
    out = io.StringIO()
    for i in range(sol.iterations):
        out.write(f"# Iteration {i + 1}\n")
    if sol.status == SolveStatus.OptimumFound:
        out.write(f"Optimum found: {_cxx_float(sol.z)}\n")
        for ix, val in zip(sol.b_ixs, sol.x_b):
            out.write(f"\tx_{int(ix)} = {_cxx_float(val)}\n")
    elif sol.status == SolveStatus.Unbounded:
        out.write("Problem unbounded.\n")
    elif sol.status == SolveStatus.ThetaOverflow:
        out.write("Theta overflow.\n")
    elif sol.status == SolveStatus.Infeasible:
        out.write("Problem infeasible.\n")
    elif sol.status == SolveStatus.NotDualFeasible:
        out.write("Start not dual feasible.\n")
    else:
        out.write("MAX_ITER exceeded.\n")
    out.write("\n")
    return out.getvalue()
