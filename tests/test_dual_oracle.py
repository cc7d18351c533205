"""CPU reference of the dual simplex (dual_oracle) against HiGHS and closed forms: optimum, x, INFEASIBLE with its
Farkas certificate, NOT_DUAL_FEASIBLE, both summation orders.  The GPU engine is held to this reference bit for bit
(tests/test_dual_gpu.py)."""
import numpy as np
import pytest
from scipy.optimize import linprog

import dual_oracle as D


def _highs(A, b, c):
    ns = A.shape[1] - A.shape[0]
    return linprog(-c[:ns], A_ub=A[:, :ns], b_ub=b, bounds=(0, None), method="highs-ds",
                   options={"presolve": False})


def _mixed(m, ns, seed, scale=1.0):
    """Mixed-sign b with c <= 0: rows with negative b are ">=" rows written as "<=" (negated)."""
    rng = np.random.default_rng(seed)
    As = rng.uniform(0.0, 1.0, (m, ns))
    sign = np.where(rng.uniform(size=m) < 0.5, -1.0, 1.0)
    b = np.where(sign > 0, ns * rng.uniform(0.5, 1.0, m), -scale * ns * rng.uniform(0.05, 0.2, m))
    A = np.asfortranarray(np.hstack([As * sign[:, None], np.eye(m)]))
    c = np.concatenate([-rng.uniform(0.5, 1.5, ns), np.zeros(m)])
    return A, b * 1.0, c


def _check_optimum(sol, A, b, c, ref):
    m, n = A.shape
    assert sol.status == D.OPTIMUM
    assert abs(sol.z - (-ref.fun)) <= 1e-9 * max(1.0, abs(ref.fun))
    x = sol.x(n)
    assert np.all(sol.x_b >= -1e-9)
    assert np.max(np.abs(A @ x - b)) <= 1e-8 * max(1.0, np.max(np.abs(b)))
    ns = n - m
    # the LPs below have unique optima (random data): same x as HiGHS
    assert np.allclose(x[:ns], ref.x, rtol=1e-7, atol=1e-8 * max(1.0, np.max(np.abs(ref.x))))


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("m,n,seed", [(1, 3, 1), (7, 20, 2), (40, 101, 3), (120, 250, 4), (300, 700, 5)])
def test_covering_matches_highs(order, m, n, seed):
    A, b, c = D.gen_covering(m, n, seed)
    sol = D.solve(A, b, c, eps=1e-9, max_iter=100000, order=order)
    ref = _highs(A, b, c)
    assert ref.status == 0
    _check_optimum(sol, A, b, c, ref)
    # the start is dual feasible and stays so: reduced costs never below -eps
    assert sol.min_e >= -1e-9
    assert sol.pivots == sol.iterations - 1 and len(sol.trace_p) == sol.pivots


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("seed", range(12))
def test_mixed_sign_b_matches_highs(order, seed):
    m, ns = [(5, 7), (30, 41), (64, 130), (200, 310)][seed % 4]
    A, b, c = _mixed(m, ns, seed, scale=1.0 if seed < 8 else 12.0)
    sol = D.solve(A, b, c, eps=1e-9, max_iter=100000, order=order, want_Binv=True)
    ref = _highs(A, b, c)
    assert ref.status in (0, 2)
    if ref.status == 2:
        assert sol.status == D.INFEASIBLE
        _check_farkas(sol, A, b)
    else:
        _check_optimum(sol, A, b, c, ref)


def _check_farkas(sol, A, b):
    """row r of the returned B^-1 (r = the row that had no entering column) proves infeasibility:
    rho.b < 0 while rho.a_j >= 0 for every column (basic ones give 0 or 1)."""
    m, n = A.shape
    r = int(np.argmin(sol.x_b))
    rho = sol.Binv[r]
    assert rho @ b < -1e-9 * max(1.0, np.abs(b).max())
    assert np.all(rho @ A >= -1e-9 * max(1.0, np.abs(rho).max()))
    assert abs(rho @ b - sol.x_b[r]) <= 1e-8 * max(1.0, abs(sol.x_b[r]))


@pytest.mark.parametrize("order", [0, 1])
def test_infeasible_closed_form(order):
    # x1 + x2 <= 1 and x1 + x2 >= 3
    A = np.asfortranarray([[1.0, 1.0, 1.0, 0.0], [-1.0, -1.0, 0.0, 1.0]])
    b = np.array([1.0, -3.0])
    c = np.array([-1.0, -2.0, 0.0, 0.0])
    sol = D.solve(A, b, c, order=order, want_Binv=True)
    assert sol.status == D.INFEASIBLE
    _check_farkas(sol, A, b)
    assert _highs(A, b, c).status == 2


@pytest.mark.parametrize("order", [0, 1])
@pytest.mark.parametrize("dt", [np.float64, np.float32])
def test_two_rows_by_hand(order, dt):
    """min x1 + x2  s.t.  x1 + 2 x2 >= 4,  3 x1 + x2 >= 6.
    Slack basis: x_b = (-4, -6), e = (1, 1, 0, 0).  Iteration 1: r = 1, rho = (0, 1), alpha_r = (-3, -1, 0, 1),
    ratios 1/3 and 1 -> x1 enters at row 1.  Iteration 2: x_b = (-2, 2), r = 0, rho = (1, -1/3),
    e = (0, 2/3, 0, 1/3), alpha_r = (0, -5/3, 1, -1/3), ratios 2/5 and 1 -> x2 enters at row 0.
    Iteration 3: x_b = (6/5, 8/5) >= 0: optimum -14/5 at x = (8/5, 6/5)."""
    A = np.asfortranarray([[-1.0, -2.0, 1.0, 0.0], [-3.0, -1.0, 0.0, 1.0]], dtype=dt)
    b = np.array([-4.0, -6.0], dt)
    c = np.array([-1.0, -1.0, 0.0, 0.0], dt)
    sol = D.solve(A, b, c, eps=1e-6, order=order)
    assert (sol.status, sol.iterations, sol.pivots) == (D.OPTIMUM, 3, 2)
    assert sol.trace_p.tolist() == [0, 1] and sol.trace_q.tolist() == [1, 0]
    assert sol.b_ixs.tolist() == [1, 0]
    tol = 1e-14 if dt == np.float64 else 1e-6
    assert np.allclose(sol.x_b, [1.2, 1.6], atol=tol, rtol=0)
    assert abs(sol.z + 2.8) <= tol * 10
    assert np.allclose(sol.y, [2.0 / 5.0, 1.0 / 5.0], atol=tol * 10)     # duals: u1 + 3 u2 = 1, 2 u1 + u2 = 1


@pytest.mark.parametrize("order", [0, 1])
def test_not_dual_feasible_start(order):
    A, b, c = D.gen_covering(20, 50, 7)
    c = c.copy()
    c[3] = 0.5                           # e_3 = -0.5 at the slack basis
    sol = D.solve(A, b, c, eps=1e-9, order=order)
    assert (sol.status, sol.iterations, sol.pivots) == (D.NOT_DUAL_FEASIBLE, 1, 0)
    assert sol.min_e == pytest.approx(-0.5)
    assert np.array_equal(sol.x_b, b)


@pytest.mark.parametrize("order", [0, 1])
def test_primal_feasible_start_is_optimal_at_once(order):
    """b >= 0 and c <= 0: the slack basis is optimal, the dual loop says so after one column pass."""
    A, b, c = D.gen_covering(10, 30, 2)
    sol = D.solve(A, -b, c, eps=1e-9, order=order)
    assert (sol.status, sol.iterations, sol.pivots) == (D.OPTIMUM, 1, 0)
    assert sol.z == 0.0


@pytest.mark.parametrize("order", [0, 1])
def test_only_slack_columns(order):
    """m = n: the slack columns are the whole LP; x = 0 is the only point, infeasible as soon as some b_i < 0."""
    m = 6
    A = np.asfortranarray(np.eye(m))
    c = np.zeros(m)
    b = np.array([1.0, -2.0, 3.0, 0.0, -1.0, 2.0])
    sol = D.solve(A, b, c, order=order, want_Binv=True)
    assert (sol.status, sol.iterations, sol.pivots) == (D.INFEASIBLE, 1, 0)
    _check_farkas(sol, A, b)
    sol = D.solve(A, np.abs(b), c, order=order)
    assert (sol.status, sol.iterations, sol.pivots) == (D.OPTIMUM, 1, 0)


@pytest.mark.parametrize("order", [0, 1])
def test_max_iter_and_pivot_tol(order):
    A, b, c = D.gen_covering(60, 150, 9)
    full = D.solve(A, b, c, eps=1e-9, order=order)
    part = D.solve(A, b, c, eps=1e-9, order=order, max_iter=5)
    assert (part.status, part.iterations, part.pivots) == (D.MAX_ITER, 5, 5)
    assert np.array_equal(part.trace_p, full.trace_p[:5]) and np.array_equal(part.trace_q, full.trace_q[:5])
    # a pivot tolerance above every |alpha_rj| leaves no entering column
    tol = D.solve(A, b, c, eps=1e-9, order=order, pivot_tol=1e6)
    assert (tol.status, tol.pivots) == (D.INFEASIBLE, 0)
    # a small one changes nothing on this LP
    small = D.solve(A, b, c, eps=1e-9, order=order, pivot_tol=1e-12)
    assert np.array_equal(small.trace_p, full.trace_p) and small.z == full.z


def test_gap_records_and_orders_agree():
    A, b, c = D.gen_covering(100, 230, 11)
    s0 = D.solve(A, b, c, eps=1e-9, order=0)
    s1 = D.solve(A, b, c, eps=1e-9, order=1)
    assert np.all(s1.gap_p >= 0) and np.all(s1.gap_q >= 0)
    if min(s1.gap_p.min(), s1.gap_q.min()) > 1e-9:       # no near-tie: both orders take the same path
        assert np.array_equal(s0.trace_p, s1.trace_p) and np.array_equal(s0.trace_q, s1.trace_q)
    assert abs(s0.z - s1.z) <= 1e-9 * abs(s0.z)


def test_covering_generator():
    import oracle
    A, b, c = D.gen_covering(8, 20, 3)
    A0, b0, c0 = oracle.gen_dense(8, 20, 3)
    assert np.array_equal(A[:, :12], -A0[:, :12]) and np.array_equal(A[:, 12:], np.eye(8))
    assert np.array_equal(b, -b0) and np.all(b < 0)
    assert np.array_equal(c[:12], -c0[:12]) and np.all(c[12:] == 0) and not np.any(np.signbit(c[12:]))
