"""Dual simplex on the B200 (options.algorithm = 1, simplex_dual) against the order-1 CPU reference bit for bit:
status, iterations, pivots, trace, x_b, b_ixs, z, y and min_reduced_cost."""
import numpy as np
import pytest

import dual_oracle as D

pytestmark = pytest.mark.gpu

EPS = 1e-9


def _run(A, b, c, dt, max_iter, windows=None, **opts):
    import simplex_method_gpu_b200 as lp
    m, n = A.shape
    eps = float(np.float32(EPS)) if dt == np.float32 else EPS
    with lp.Engine(m, n, dtype=dt, eps=eps, max_iter=max_iter, algorithm=1, **opts) as e:
        e.upload(A.astype(dt, order="F"), b.astype(dt), c.astype(dt))
        for w in (windows or [max_iter]):
            r = e.run(w)
        x_b, b_ixs, y = e.download()
        return r, e.trace(), x_b, b_ixs, y


def _ref(A, b, c, dt, max_iter, pivot_tol=0.0):
    eps = np.float32(EPS) if dt == np.float32 else EPS
    return D.solve(A.astype(dt, order="F"), b.astype(dt), c.astype(dt), eps=eps, max_iter=max_iter, order=1,
                   pivot_tol=pivot_tol)


def _same(got, ref):
    r, tr, x_b, b_ixs, y = got
    assert (int(r["status"]), r["iterations"], r["pivots"]) == (ref.status, ref.iterations, ref.pivots)
    assert np.array_equal(tr[:, 0], ref.trace_p) and np.array_equal(tr[:, 1], ref.trace_q)
    assert np.array_equal(b_ixs, ref.b_ixs)
    assert np.array_equal(x_b, ref.x_b) and np.array_equal(y, ref.y)
    assert r["z"] == ref.z
    assert r["min_reduced_cost"] == ref.min_e


def _infeasible(m, n, seed):
    """covering rows plus one row sum(x) <= 0.01: no solution, dual feasible start"""
    A, b, c = D.gen_covering(m, n, seed)
    ns = n - m
    A[m - 1, :ns] = 1.0
    b[m - 1] = 0.01
    return A, b, c


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("m", [1, 7, 63, 64, 65, 200, 1000, 2100])
def test_ragged_shapes_bit_exact(m, dt):
    n = m + 2 * m + 3                                   # n - m odd: ragged pricing groups
    A, b, c = D.gen_covering(m, n, 100 + m)
    cap = 100000 if m <= 200 else 400
    ref = _ref(A, b, c, dt, cap)
    assert ref.pivots > 0
    _same(_run(A, b, c, dt, cap), ref)


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_slack_block_as_data(dt):
    """last m columns not the identity: all n columns are stored and priced from A (ns = n)"""
    m, n = 70, 181
    A, b, c = D.gen_covering(m, n, 5)
    A[0, n - 1] = 0.25
    ref = _ref(A, b, c, dt, 300)
    _same(_run(A, b, c, dt, 300), ref)


@pytest.mark.parametrize("grid", [1, 3, 0])
@pytest.mark.parametrize("tile", [0, 1, 2, 4, 8])
def test_grid_and_tile_shape(grid, tile):
    A, b, c = D.gen_covering(300, 677, 21)
    ref = _ref(A, b, c, np.float64, 100000)
    _same(_run(A, b, c, np.float64, 100000, grid_ctas=grid, tile_shape=tile), ref)


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_windows_equal_one_run(dt):
    A, b, c = D.gen_covering(150, 333, 8)
    ref = _ref(A, b, c, dt, 100000)
    w = [7] * (ref.iterations // 7) + [100000]
    _same(_run(A, b, c, dt, 100000, windows=w), ref)


def test_statuses():
    A, b, c = D.gen_covering(120, 301, 13)
    full = _ref(A, b, c, np.float64, 100000)
    assert full.status == D.OPTIMUM
    _same(_run(A, b, c, np.float64, 100000), full)
    part = _ref(A, b, c, np.float64, 9)                        # max_iter
    assert (part.status, part.pivots) == (D.MAX_ITER, 9)
    _same(_run(A, b, c, np.float64, 9), part)
    Ai, bi, ci = _infeasible(120, 301, 14)                     # infeasible after some pivots
    inf = _ref(Ai, bi, ci, np.float64, 100000)
    assert inf.status == D.INFEASIBLE and inf.pivots > 0
    _same(_run(Ai, bi, ci, np.float64, 100000), inf)
    c2 = c.copy()                                              # not dual feasible at the start
    c2[17] = 0.25
    ndf = _ref(A, b, c2, np.float64, 100000)
    assert (ndf.status, ndf.pivots) == (D.NOT_DUAL_FEASIBLE, 0)
    _same(_run(A, b, c2, np.float64, 100000), ndf)


@pytest.mark.parametrize("tol", [1e-3, 1e6])
def test_pivot_tol(tol):
    A, b, c = D.gen_covering(90, 211, 31)
    ref = _ref(A, b, c, np.float64, 100000, pivot_tol=tol)
    _same(_run(A, b, c, np.float64, 100000, pivot_tol=tol), ref)


def test_only_slack_columns():
    m = 40
    A = np.asfortranarray(np.eye(m))
    b = np.linspace(-1.0, 1.0, m)
    c = np.zeros(m)
    ref = _ref(A, b, c, np.float64, 100)
    assert ref.status == D.INFEASIBLE
    _same(_run(A, b, c, np.float64, 100), ref)


def test_solve_and_batch_equal_single_calls():
    import simplex_method_gpu_b200 as lp
    m, n, k = 24, 61, 5
    lps = [D.gen_covering(m, n, 40 + i) for i in range(k)]
    lps[3] = _infeasible(m, n, 43)
    A = np.stack([x[0] for x in lps])
    b = np.stack([x[1] for x in lps])
    c = np.stack([x[2] for x in lps])
    bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=1000, trace_cap=1000, algorithm=1)
    for i in range(k):
        one = lp.solve(A[i], b[i], c[i], eps=EPS, max_iter=1000, algorithm=1)
        ref = _ref(A[i], b[i], c[i], np.float64, 1000)
        assert (int(one.status), one.iterations, one.pivots, one.z) == (ref.status, ref.iterations, ref.pivots, ref.z)
        assert np.array_equal(one.x_b, ref.x_b) and np.array_equal(one.trace[:, 0], ref.trace_p)
        s = bs.solution(i)
        assert (s.status, s.iterations, s.pivots, s.z) == (one.status, one.iterations, one.pivots, one.z)
        assert np.array_equal(s.x_b, one.x_b) and np.array_equal(s.b_ixs, one.b_ixs)
        assert np.array_equal(s.trace, one.trace) and np.array_equal(bs.y[i], ref.y)
    assert int(bs.status[3]) == int(lp.SolveStatus.Infeasible)
    assert "Problem infeasible." in lp.format_result(bs.solution(3))


def test_primal_default_unchanged_on_the_same_engine_options():
    """algorithm = 0 on a covering LP still runs the primal loop (infeasible start: it never pivots right)."""
    import oracle
    import simplex_method_gpu_b200 as lp
    A, b, c = D.gen_covering(50, 120, 3)
    prim = lp.solve(A, b, c, eps=EPS, max_iter=50)
    ref = oracle.solve(A, b, c, eps=EPS, max_iter=50, order=1)
    assert (int(prim.status), prim.pivots, prim.z) == (ref.status, ref.pivots, ref.z)


def test_large_covering_to_optimality():
    """m = 8192, n = 16384 (fp64): optimum with a duality gap <= 1e-9, checked on the host from x_b, b_ixs and y."""
    import simplex_method_gpu_b200 as lp
    m, n = 8192, 16384
    A, b, c = D.gen_covering(m, n, 1)
    with lp.Engine(m, n, dtype=np.float64, eps=EPS, max_iter=10 ** 6, algorithm=1) as e:
        e.upload(A, b, c)
        r = e.run(10 ** 6)
        x_b, b_ixs, y = e.download()
    assert r["status"] == lp.SolveStatus.OptimumFound and r["pivots"] > 0
    x = np.zeros(n)
    x[b_ixs] = x_b
    assert x.min() >= -1e-9 * np.abs(b).max()
    assert np.abs(A @ x - b).max() <= 1e-9 * np.abs(b).max()
    e_red = y @ A - c
    assert e_red.min() >= -1e-9 * np.abs(c).max()
    primal, dual = c @ x, y @ b
    assert abs(primal - dual) <= 1e-9 * abs(primal)
    assert abs(r["z"] - primal) <= 1e-9 * abs(primal)


def test_cli_dual(tmp_path):
    """bin/solver.out --dual on the two-row example of tests/test_dual_oracle.py and on an infeasible LP"""
    import os
    import subprocess
    import simplex_method_gpu_b200 as lp
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "bin", "solver.out")
    f = tmp_path / "two_rows.txt"
    lp.write_lp(str(f), np.array([[-1.0, -2.0, 1.0, 0.0], [-3.0, -1.0, 0.0, 1.0]]), np.array([-4.0, -6.0]),
                np.array([-1.0, -1.0, 0.0, 0.0]))
    out = subprocess.run([cli, str(f), "--f64", "--dual", "--max-iter", "10"], capture_output=True, text=True, check=True).stdout
    assert out.startswith("# Iteration 1\n# Iteration 2\n# Iteration 3\nOptimum found: -2.8\n\tx_1 = 1.2\n\tx_0 = 1.6\n"), out
    g = tmp_path / "infeasible.txt"
    lp.write_lp(str(g), np.array([[1.0, 1.0, 1.0, 0.0], [-1.0, -1.0, 0.0, 1.0]]), np.array([1.0, -3.0]),
                np.array([-1.0, -2.0, 0.0, 0.0]))
    out = subprocess.run([cli, str(g), "--f64", "--dual", "--max-iter", "10"], capture_output=True, text=True, check=True).stdout
    assert "Problem infeasible.\n" in out, out
    out = subprocess.run([cli, str(f), "--f64", "--max-iter", "10"], capture_output=True, text=True, check=True).stdout
    assert out.startswith("# Iteration 1\nOptimum found: 0\n"), out       # the primal loop cannot see the ">=" rows
