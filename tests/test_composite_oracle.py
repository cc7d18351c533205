"""CPU reference of the composite method (dual_oracle with cost_shift=1: dual loop on shifted costs, then the primal
loop) against HiGHS and against the two loops it is made of.  The GPU engine is held to this reference bit for bit
(tests/test_composite_gpu.py)."""
import numpy as np
import pytest
from scipy.optimize import linprog

import dual_oracle as D
import oracle as O

EPS = 1e-9


def _solve(A, b, c, order=1, **kw):
    kw.setdefault("max_iter", 100000)
    return D.solve(A, b, c, eps=EPS, order=order, cost_shift=1, **kw)


def _highs(A, b, c):
    ns = A.shape[1] - A.shape[0]
    return linprog(-c[:ns], A_ub=A[:, :ns], b_ub=b, bounds=(0, None), method="highs")


def _check_optimum(sol, A, b, c):
    m, n = A.shape
    ref = _highs(A, b, c)
    assert ref.status == 0
    assert sol.status == D.OPTIMUM and sol.phase == 2
    assert abs(sol.z - (-ref.fun)) <= 1e-9 * max(1.0, abs(ref.fun))
    x = sol.x(n)
    assert np.all(x >= -1e-9)
    assert np.max(A @ x - b) <= 1e-9 * max(1.0, np.max(np.abs(b)))
    # optimality from the returned basis: every reduced cost e_j = y.a_j - c_j >= -eps (up to the recomputation)
    e = A.T @ sol.y - c
    assert e.min() >= -1e-9 * max(1.0, np.max(np.abs(c)))
    assert np.array_equal(np.sort(sol.b_ixs), np.unique(sol.b_ixs))


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("m,n,seed", [(5, 13, 2), (30, 71, 2), (64, 200, 3), (120, 301, 4), (250, 600, 5)])
def test_feasible_family_matches_highs(m, n, seed, order):
    A, b, c = D.gen_general(m, n, seed, "feasible")
    assert b.min() < 0 and c.max() > 0                 # the slack basis is neither primal nor dual feasible
    sol = _solve(A, b, c, order)
    assert sol.shifted > 0 and 0 < sol.phase1_pivots <= sol.pivots
    _check_optimum(sol, A, b, c)


@pytest.mark.parametrize("m,n,seed", [(10, 25, 1), (50, 131, 2), (200, 501, 3)])
def test_degenerate_family_matches_highs(m, n, seed):
    """integer data with repeated rows; the textbook ratio tests need pivot_tol against noise pivots here"""
    A, b, c = D.gen_general(m, n, seed, "degenerate")
    _check_optimum(_solve(A, b, c, pivot_tol=1e-9), A, b, c)


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("m,n,seed", [(3, 7, 1), (10, 25, 2), (50, 131, 2), (200, 501, 3)])
def test_infeasible_with_farkas_certificate(m, n, seed, order):
    A, b, c = D.gen_general(m, n, seed, "infeasible")
    assert _highs(A, b, c).status == 2
    sol = _solve(A, b, c, order, pivot_tol=1e-9, want_Binv=True)
    assert sol.status == D.INFEASIBLE and sol.phase == 1
    r = int(np.argmin(sol.x_b))
    rho = sol.Binv[r, :]
    assert rho @ b < 0
    assert (rho @ A).min() >= -1e-12 * max(1.0, np.abs(rho).max())


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("m,n,seed", [(4, 9, 1), (50, 131, 2), (200, 501, 3)])
def test_unbounded(m, n, seed, order):
    A, b, c = D.gen_general(m, n, seed, "unbounded")
    assert _highs(A, b, c).status == 3
    sol = _solve(A, b, c, order)
    assert sol.status == D.UNBOUNDED and sol.phase == 2


@pytest.mark.parametrize("kind", ["feasible", "unbounded", "infeasible"])
@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_orders_agree(kind, dt):
    A, b, c = D.gen_general(40, 101, 7, kind, dt)
    eps = np.float32(EPS) if dt == np.float32 else EPS
    s0, s1 = (D.solve(A, b, c, eps=eps, max_iter=100000, order=o, cost_shift=1, pivot_tol=1e-7) for o in (0, 1))
    assert s0.status == s1.status
    tol = 1e-9 if dt == np.float64 else 1e-4
    if kind == "feasible":
        assert abs(s0.z - s1.z) <= tol * max(1.0, abs(s1.z))


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("m,n", [(1, 4), (20, 61), (100, 257)])
def test_feasible_start_is_the_primal_run_plus_one_iteration(m, n, dt):
    """b >= 0: phase 1 stops at once (one iteration, no pivot), the hand-over keeps y, phase 2 is the primal loop"""
    A, b, c = O.gen_dense(m, n, 11, dt)
    eps = np.float32(EPS) if dt == np.float32 else EPS
    ref = O.solve(A, b, c, eps=eps, max_iter=100000, order=1)
    sol = D.solve(A, b, c, eps=eps, max_iter=100001, order=1, cost_shift=1)
    assert sol.shifted == n - m and sol.phase1_pivots == 0 and sol.phase == 2
    assert (sol.status, sol.iterations, sol.pivots) == (ref.status, ref.iterations + 1, ref.pivots)
    assert np.array_equal(sol.trace_p, ref.trace_p) and np.array_equal(sol.trace_q, ref.trace_q)
    assert np.array_equal(sol.x_b, ref.x_b) and np.array_equal(sol.b_ixs, ref.b_ixs) and np.array_equal(sol.y, ref.y)
    assert sol.z == ref.z


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("m,n", [(3, 8), (40, 101)])
def test_dual_feasible_start_is_the_dual_run(m, n, dt):
    """c <= 0: nothing is shifted and the run is the plain dual loop, status and all"""
    A, b, c = D.gen_covering(m, n, 12, dt)
    eps = np.float32(EPS) if dt == np.float32 else EPS
    ref = D.solve(A, b, c, eps=eps, order=1)
    sol = D.solve(A, b, c, eps=eps, order=1, cost_shift=1)
    assert sol.shifted == 0 and sol.phase == 1 and sol.phase1_pivots == sol.pivots
    assert (sol.status, sol.iterations, sol.pivots, sol.z, sol.min_e) == (ref.status, ref.iterations, ref.pivots, ref.z, ref.min_e)
    assert np.array_equal(sol.trace_p, ref.trace_p) and np.array_equal(sol.x_b, ref.x_b) and np.array_equal(sol.y, ref.y)


def test_window_ending_on_the_phase1_optimum_hands_over():
    """max_iter that ends on the phase-1 optimum: MAX_ITER, phase 2 entered, z for the original costs"""
    A, b, c = D.gen_general(30, 71, 2, "feasible")
    full = _solve(A, b, c)
    k = full.phase1_pivots + 1
    cut = _solve(A, b, c, max_iter=k)
    assert (cut.status, cut.iterations, cut.pivots, cut.phase) == (D.MAX_ITER, k, full.phase1_pivots, 2)
    assert np.isclose(cut.z, c[cut.b_ixs] @ cut.x_b, rtol=1e-12, atol=1e-12)
    assert np.array_equal(cut.trace_p, full.trace_p[:k - 1])


def test_gen_general_shapes_and_kinds():
    for kind in D.GENERAL_KINDS:
        A, b, c = D.gen_general(6, 15, 3, kind, np.float32)
        assert A.shape == (6, 15) and b.shape == (6,) and c.shape == (15,) and A.dtype == np.float32
        assert np.array_equal(A[:, 9:], np.eye(6))
        assert np.all(c[9:] == 0)
    with pytest.raises(ValueError):
        D.gen_general(6, 15, 3, "bogus")
