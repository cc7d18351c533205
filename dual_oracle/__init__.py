"""TEST INFRASTRUCTURE — NOT PRODUCT CODE.

ctypes front-end of the CPU reference of the dual simplex loop and of the composite method built on it
(``libdualoracle.so``, built in-tree with gcc by ``build()``), the check of the engine's ``algorithm=1`` path with and
without ``cost_shift=1``.  Order 1 replays the engine's summation orders, so the
two compare bit for bit.  Only ``tests/``, ``tools/`` and ``__graft_entry__`` import it; the product path never does.

Also ``gen_covering``: the synthetic dense LP negated, whose slack basis is dual feasible and primal infeasible, and
``gen_general``: LPs whose slack basis is neither (the composite method's inputs).
"""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
from dataclasses import dataclass, field

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_ORACLE = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB_PATH = os.path.join(_HERE, "libdualoracle.so")
_SRCS = [os.path.join(_HERE, f) for f in ("dual_oracle.c", "dual_oracle_impl.h")] + \
        [os.path.join(_ORACLE, f) for f in ("simplex_oracle_impl.h", "simplex_oracle.h")]

MAX_ITER, OPTIMUM, UNBOUNDED, INFEASIBLE, NOT_DUAL_FEASIBLE = 0, 1, 2, 4, 5


class _Result(C.Structure):
    _fields_ = [("status", C.c_int), ("iterations", C.c_long), ("pivots", C.c_long), ("z", C.c_double),
                ("min_e", C.c_double), ("phase", C.c_int), ("shifted", C.c_long), ("phase1_pivots", C.c_long)]


def _cc() -> str:
    # the primal oracle's choice (oracle/Makefile): a gcc that ships libgomp
    for cand in ("/usr/bin/gcc-13", "/usr/bin/gcc"):
        if os.path.exists(cand):
            return cand
    return shutil.which("gcc") or "gcc"


def build(force: bool = False) -> str:
    """Compile libdualoracle.so in-tree (gcc, a few seconds) when a source is newer."""
    stale = (not os.path.exists(_LIB_PATH)) or any(os.path.getmtime(s) > os.path.getmtime(_LIB_PATH) for s in _SRCS)
    if force or stale:
        tmp = _LIB_PATH + f".{os.getpid()}.tmp"
        subprocess.run([_cc(), "-O3", "-march=x86-64-v3", "-fopenmp", "-ffp-contract=off", "-fPIC", "-Wall", "-Wextra",
                        "-Wno-unknown-pragmas", "-shared", "-o", tmp, _SRCS[0], "-lm"], check=True, capture_output=True)
        os.replace(tmp, _LIB_PATH)
    return _LIB_PATH


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(_LIB_PATH)
        for name, real in (("dual_solve_f64", C.c_double), ("dual_solve_f32", C.c_float)):
            fn = getattr(L, name)
            fn.restype = C.c_int
            fn.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.c_long, real, C.c_long, C.c_int, C.c_double,
                           C.c_int, C.c_double,
                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                           C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_long, C.POINTER(_Result)]
        _lib = L
    return _lib


@dataclass
class DualSolution:
    status: int
    iterations: int
    pivots: int
    z: float
    min_e: float
    x_b: np.ndarray
    b_ixs: np.ndarray
    y: np.ndarray
    trace_p: np.ndarray
    trace_q: np.ndarray
    gap_p: np.ndarray            # runner-up distance of the entering column (dual ratio test; phase 2: pricing)
    gap_q: np.ndarray            # runner-up distance of the leaving row (x_b argmin; phase 2: primal ratio test)
    Binv: np.ndarray | None = field(default=None, repr=False)
    phase: int = 0               # composite method: 1 (ended in the dual loop) or 2 (in the primal loop)
    shifted: int = 0             # columns the cost shift moved
    phase1_pivots: int = 0

    def x(self, n: int) -> np.ndarray:
        out = np.zeros(n, dtype=self.x_b.dtype)
        out[self.b_ixs] = self.x_b
        return out


def _ptr(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def solve(A, b, c, eps=1e-9, max_iter=100000, order=0, pivot_tol=0.0, want_Binv=False,
          trace_cap=None, cost_shift=0, shift_delta=0.0) -> DualSolution:
    """Dual simplex from the slack basis; with ``cost_shift=1`` the composite method (dual loop on shifted costs, then
    the primal loop).  A: (m, n), slack block last; float32 or float64."""
    dt = np.dtype(A.dtype)
    assert dt in (np.float32, np.float64)
    A = np.asfortranarray(A, dtype=dt)
    b = np.ascontiguousarray(b, dtype=dt)
    c = np.ascontiguousarray(c, dtype=dt)
    m, n = A.shape
    cap = int(trace_cap if trace_cap is not None else min(max_iter, 1 << 22))
    x_b = np.zeros(m, dt)
    y = np.zeros(m, dt)
    b_ixs = np.zeros(m, np.int32)
    Binv = np.zeros((m, m), dt, order="F") if want_Binv else None
    tp = np.full(cap, -1, np.int32)
    tq = np.full(cap, -1, np.int32)
    gp = np.zeros(cap, np.float64)
    gq = np.zeros(cap, np.float64)
    res = _Result()
    fn = lib().dual_solve_f64 if dt == np.float64 else lib().dual_solve_f32
    rc = fn(_ptr(A), _ptr(b), _ptr(c), m, n, eps, int(max_iter), int(order), float(pivot_tol),
            int(cost_shift), float(shift_delta),
            _ptr(x_b), _ptr(b_ixs), _ptr(y), _ptr(Binv), _ptr(tp), _ptr(tq), _ptr(gp), _ptr(gq), cap, C.byref(res))
    if rc != 0:
        raise ValueError(f"dual_solve failed with code {rc} (m={m}, n={n})")
    k = min(res.pivots, cap)
    return DualSolution(res.status, res.iterations, res.pivots, res.z, res.min_e, x_b, b_ixs, y,
                        tp[:k], tq[:k], gp[:k], gq[:k], Binv, res.phase, res.shifted, res.phase1_pivots)


def gen_covering(m: int, n: int, seed: int = 1, dtype=np.float64):
    """The dense generator's LP negated: A = [-A_s, I], b = -b_s, c = [-c_s, 0], i.e. min c_s.x s.t. A_s x >= b_s,
    x >= 0 written as a max over <= rows.  The slack basis is dual feasible (e_j = c_s,j > 0) and primal infeasible
    (x_b = -b_s < 0); the LP has a finite optimum (A_s > 0, c_s > 0)."""
    import oracle
    A, b, c = oracle.gen_dense(m, n, seed, dtype)
    ns = n - m
    A[:, :ns] = -A[:, :ns]
    c = -c
    c[ns:] = 0                     # +0, not -0
    return A, -b, c


GENERAL_KINDS = ("feasible", "infeasible", "unbounded", "degenerate")


def gen_general(m: int, n: int, seed: int = 1, kind: str = "feasible", dtype=np.float64):
    """max c.x, A_s x <= b, x >= 0 with mixed-sign b and c: the slack basis is neither primal nor dual feasible.
    A = [A_s, I] (m x n, n - m >= 2 structural columns), c = [c_s, 0].
      feasible    A_s ~ U(-1, 1), b = A_s x0 + U(0.1, 1) for a known x0 ~ U(0, 1), c_s ~ U(-1, 1); the last row is
                  sum(x) <= sum(x0) + 1, so the LP is bounded and x0 strictly feasible
      infeasible  as feasible, with row m-2 = -(row 0) and b = -b_0 - 1, which contradicts row 0 (needs m >= 3)
      unbounded   as feasible without the bounding row (a random row instead) and with column 0 = -U(0, 1),
                  c_0 ~ U(0.5, 1): x_0 grows without bound
      degenerate  integer data: A_s in {-3..3}, x0 in {0, 1, 2}, b = A_s x0 + {0, 1}, c_s in {-3..3}, every third row
                  a copy of the row before it, bounding row as in feasible"""
    if kind not in GENERAL_KINDS:
        raise ValueError(f"kind must be one of {GENERAL_KINDS}")
    ns = n - m
    assert ns >= 2 and m >= 1
    rng = np.random.default_rng([seed, GENERAL_KINDS.index(kind)])
    if kind == "degenerate":
        As = rng.integers(-3, 4, size=(m, ns)).astype(np.float64)
        x0 = rng.integers(0, 3, size=ns).astype(np.float64)
        for i in range(2, m - 1, 3):
            As[i] = As[i - 1]
        b = As @ x0 + rng.integers(0, 2, size=m)
        for i in range(2, m - 1, 3):
            b[i] = b[i - 1]
        cs = rng.integers(-3, 4, size=ns).astype(np.float64)
    else:
        As = rng.uniform(-1.0, 1.0, size=(m, ns))
        x0 = rng.uniform(0.0, 1.0, size=ns)
        b = As @ x0 + rng.uniform(0.1, 1.0, size=m)
        cs = rng.uniform(-1.0, 1.0, size=ns)
    if kind != "unbounded":
        As[m - 1] = 1.0
        b[m - 1] = x0.sum() + 1.0
    if kind == "infeasible":
        assert m >= 3
        As[m - 2] = -As[0]
        b[m - 2] = -b[0] - 1.0
    if kind == "unbounded":
        As[:, 0] = -rng.uniform(0.0, 1.0, size=m)
        cs[0] = rng.uniform(0.5, 1.0)
    A = np.zeros((m, n), dtype=dtype, order="F")
    A[:, :ns] = As
    A[:, ns:] = np.eye(m)
    c = np.zeros(n, dtype=dtype)
    c[:ns] = cs
    return A, b.astype(dtype), c
