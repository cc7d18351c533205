"""Composite method on the B200 (options.algorithm = 1, cost_shift = 1: k_cost_shift, simplex_dual on the shifted
costs, the hand-over, then simplex_tiny / simplex_resident / simplex_persistent on the original costs) against the
order-1 CPU reference bit for bit: status, iterations, pivots, trace, x_b, b_ixs, y, z, min_reduced_cost and the
phase information."""
import numpy as np
import pytest

import dual_oracle as D

pytestmark = pytest.mark.gpu

EPS = 1e-9


def _eps(dt):
    # fp32: the primal loop needs a tolerance above its rounding noise to stop
    return float(np.float32(1e-5)) if dt == np.float32 else EPS


def _run(A, b, c, dt, max_iter, windows=None, **opts):
    import simplex_method_gpu_b200 as lp
    m, n = A.shape
    with lp.Engine(m, n, dtype=dt, eps=_eps(dt), max_iter=max_iter, algorithm=1, cost_shift=1, **opts) as e:
        e.upload(A.astype(dt, order="F"), b.astype(dt), c.astype(dt))
        assert e.phase_info()["phase"] == 0
        for w in (windows or [max_iter]):
            r = e.run(w)
        x_b, b_ixs, y = e.download()
        return r, e.trace(), x_b, b_ixs, y, e.phase_info()


def _ref(A, b, c, dt, max_iter, **kw):
    eps = np.float32(_eps(dt)) if dt == np.float32 else EPS
    return D.solve(A.astype(dt, order="F"), b.astype(dt), c.astype(dt), eps=eps, max_iter=max_iter, order=1,
                   cost_shift=1, **kw)


def _same(got, ref):
    r, tr, x_b, b_ixs, y, ph = got
    assert (int(r["status"]), r["iterations"], r["pivots"]) == (ref.status, ref.iterations, ref.pivots)
    assert np.array_equal(tr[:, 0], ref.trace_p) and np.array_equal(tr[:, 1], ref.trace_q)
    assert np.array_equal(b_ixs, ref.b_ixs)
    assert np.array_equal(x_b, ref.x_b) and np.array_equal(y, ref.y)
    assert r["z"] == ref.z
    assert r["min_reduced_cost"] == ref.min_e
    assert (ph["phase"], ph["shifted_columns"], ph["phase1_pivots"]) == (ref.phase, ref.shifted, ref.phase1_pivots)


def _few_negative_rows(m, n, seed, k=1):
    """the feasible family with only k rows of negative b (raising b_i keeps x0 feasible): a short phase 1, so a
    capped run reaches phase 2 at every size"""
    A, b, c = D.gen_general(m, n, seed, "feasible")
    neg = np.flatnonzero(b < 0)[:k]
    keep = np.zeros(m, bool)
    keep[neg] = True
    b = np.where(keep, b, np.abs(b) + 0.1)
    return A, b, c


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
@pytest.mark.parametrize("m", [1, 7, 63, 64, 65, 200, 1000, 2100])
def test_ragged_shapes_bit_exact(m, dt):
    n = m + 2 * m + 3                                   # n - m odd: ragged pricing groups
    if m <= 200:
        A, b, c = D.gen_general(m, n, 100 + m, "feasible")
        cap = 100000 if dt == np.float64 else 3000      # fp32: a capped run where the textbook loop does not settle
    else:
        A, b, c = _few_negative_rows(m, n, 100 + m)
        cap = 600
    ref = _ref(A, b, c, dt, cap)
    assert ref.phase == 2
    _same(_run(A, b, c, dt, cap), ref)


def test_phase2_reaches_each_primal_kernel():
    """phase 2 runs where algorithm = 0 would: simplex_tiny (m = 7), simplex_resident (m = 200) and the general
    simplex_persistent (m = 2100), after k_cost_shift and simplex_dual"""
    import torch
    from torch.profiler import ProfilerActivity, profile
    for m, want in ((7, "simplex_tiny"), (200, "simplex_resident"), (2100, "simplex_persistent")):
        n = 3 * m + 3
        A, b, c = _few_negative_rows(m, n, 5 + m) if m > 200 else D.gen_general(m, n, 5 + m, "feasible")
        cap = 600 if m > 200 else 100000
        ref = _ref(A, b, c, np.float64, cap)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            got = _run(A, b, c, np.float64, cap)
            torch.cuda.synchronize()
        _same(got, ref)
        names = " ".join(ev.name for ev in prof.events())
        for k in ("k_cost_shift", "simplex_dual", want):
            assert k in names, (m, k)


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_slack_block_as_data(dt):
    """last m columns not the identity: all n columns are stored, shifted and priced from A (ns = n)"""
    m, n = 70, 181
    A, b, c = D.gen_general(m, n, 5, "feasible")
    A[0, n - 1] = 0.25
    ref = _ref(A, b, c, dt, 100000)
    assert ref.phase == 2
    _same(_run(A, b, c, dt, 100000), ref)


@pytest.mark.parametrize("grid", [1, 3, 0])
@pytest.mark.parametrize("tile", [0, 1, 2, 4, 8])
def test_grid_and_tile_shape(grid, tile):
    A, b, c = D.gen_general(300, 677, 21, "feasible")
    ref = _ref(A, b, c, np.float64, 100000)
    _same(_run(A, b, c, np.float64, 100000, grid_ctas=grid, tile_shape=tile), ref)


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_windows_equal_one_run(dt):
    """windows of 7, one that ends exactly on the phase-1 optimum (hand-over, MAX_ITER), then the rest"""
    A, b, c = D.gen_general(150, 333, 8, "feasible")
    cap = 100000 if dt == np.float64 else 3000
    ref = _ref(A, b, c, dt, cap)
    k1 = ref.phase1_pivots + 1                       # the pivots of phase 1 and its final check
    _same(_run(A, b, c, dt, cap, windows=[7] * (ref.iterations // 7) + [cap - 7 * (ref.iterations // 7)]), ref)
    cut = _ref(A, b, c, dt, k1)
    assert (cut.status, cut.phase) == (D.MAX_ITER, 2)
    _same(_run(A, b, c, dt, cap, windows=[k1]), cut)
    _same(_run(A, b, c, dt, cap, windows=[k1 - 3, 3, 5, cap - k1 - 5]), ref)


def test_abort_and_continue():
    import simplex_method_gpu_b200 as lp
    A, b, c = D.gen_general(400, 901, 9, "feasible")
    ref = _ref(A, b, c, np.float64, 100000)
    with lp.Engine(400, 901, dtype=np.float64, eps=EPS, max_iter=100000, algorithm=1, cost_shift=1, grid_ctas=2) as e:
        e.upload(A, b, c)
        e.run_async(100000)
        e.abort()
        r = e.wait()
        assert r["aborted"] or r["status"] == lp.SolveStatus.OptimumFound
        r = e.run(100000 - r["iterations"])
        x_b, b_ixs, y = e.download()
        _same((r, e.trace(), x_b, b_ixs, y, e.phase_info()), ref)


@pytest.mark.parametrize("m,n", [(7, 20), (200, 503), (2100, 4203)])
def test_feasible_start_equals_the_primal_run(m, n):
    """b >= 0: bit for bit algorithm = 0's run on the same kernel, one iteration more"""
    import oracle
    import simplex_method_gpu_b200 as lp
    A, b, c = oracle.gen_dense(m, n, 3)
    cap = 100000 if m <= 200 else 300
    prim = lp.solve(A, b, c, eps=EPS, max_iter=cap, trace_cap=cap)
    comp = _run(A, b, c, np.float64, cap + 1)
    r, tr, x_b, b_ixs, y, ph = comp
    assert (int(r["status"]), r["iterations"], r["pivots"], r["z"]) == (int(prim.status), prim.iterations + 1, prim.pivots, prim.z)
    assert np.array_equal(tr, prim.trace) and np.array_equal(x_b, prim.x_b) and np.array_equal(b_ixs, prim.b_ixs)
    assert (ph["phase"], ph["shifted_columns"], ph["phase1_pivots"]) == (2, n - m, 0)


@pytest.mark.parametrize("m,n", [(24, 61), (300, 677)])
def test_dual_feasible_start_equals_the_dual_run(m, n):
    """c <= 0 (covering LP): bit for bit algorithm = 1's run, nothing shifted"""
    import simplex_method_gpu_b200 as lp
    A, b, c = D.gen_covering(m, n, 4)
    with lp.Engine(m, n, dtype=np.float64, eps=EPS, max_iter=100000, algorithm=1) as e:
        e.upload(A, b, c)
        r0 = e.run(100000)
        x0, bix0, y0 = e.download()
        tr0 = e.trace()
    r, tr, x_b, b_ixs, y, ph = _run(A, b, c, np.float64, 100000)
    for k in ("status", "iterations", "pivots", "z", "min_reduced_cost"):
        assert r[k] == r0[k], k
    assert np.array_equal(tr, tr0) and np.array_equal(x_b, x0) and np.array_equal(b_ixs, bix0) and np.array_equal(y, y0)
    assert (ph["phase"], ph["shifted_columns"], ph["phase1_pivots"]) == (1, 0, r0["pivots"])


def test_statuses_and_phase_info():
    A, b, c = D.gen_general(120, 301, 13, "feasible")
    full = _ref(A, b, c, np.float64, 100000)                           # OPTIMUM in phase 2
    assert (full.status, full.phase) == (D.OPTIMUM, 2)
    _same(_run(A, b, c, np.float64, 100000), full)
    late = _ref(A, b, c, np.float64, full.phase1_pivots + 5)            # MAX_ITER in phase 2
    assert (late.status, late.phase) == (D.MAX_ITER, 2)
    _same(_run(A, b, c, np.float64, full.phase1_pivots + 5), late)
    early = _ref(A, b, c, np.float64, 4)                               # MAX_ITER in phase 1 (z, min e of c')
    assert (early.status, early.phase, early.pivots) == (D.MAX_ITER, 1, 4)
    _same(_run(A, b, c, np.float64, 4), early)
    Au, bu, cu = D.gen_general(120, 301, 14, "unbounded")              # UNBOUNDED in phase 2
    unb = _ref(Au, bu, cu, np.float64, 100000)
    assert (unb.status, unb.phase) == (D.UNBOUNDED, 2)
    _same(_run(Au, bu, cu, np.float64, 100000), unb)
    Ai, bi, ci = D.gen_general(120, 301, 15, "infeasible")             # INFEASIBLE in phase 1
    inf = _ref(Ai, bi, ci, np.float64, 100000, pivot_tol=1e-9)
    assert (inf.status, inf.phase) == (D.INFEASIBLE, 1) and inf.pivots > 0
    _same(_run(Ai, bi, ci, np.float64, 100000, pivot_tol=1e-9), inf)


def test_degenerate_family():
    A, b, c = D.gen_general(50, 131, 2, "degenerate")
    ref = _ref(A, b, c, np.float64, 100000, pivot_tol=1e-9)
    assert ref.status == D.OPTIMUM
    _same(_run(A, b, c, np.float64, 100000, pivot_tol=1e-9), ref)


def test_reset_starts_over():
    import simplex_method_gpu_b200 as lp
    A, b, c = D.gen_general(90, 211, 16, "feasible")
    ref = _ref(A, b, c, np.float64, 100000)
    with lp.Engine(90, 211, dtype=np.float64, eps=EPS, max_iter=100000, algorithm=1, cost_shift=1) as e:
        e.upload(A, b, c)
        e.run(ref.phase1_pivots // 2)               # stop inside phase 1: the engine prices with c'
        e.reset()
        assert e.phase_info() == {"phase": 0, "shifted_columns": 0, "phase1_pivots": 0}
        r = e.run(100000)
        x_b, b_ixs, y = e.download()
        _same((r, e.trace(), x_b, b_ixs, y, e.phase_info()), ref)


def test_solve_and_batch_equal_single_calls():
    import simplex_method_gpu_b200 as lp
    m, n, k = 24, 61, 5
    lps = [D.gen_general(m, n, 40 + i, "feasible") for i in range(k)]
    lps[3] = D.gen_general(m, n, 43, "infeasible")
    A = np.stack([x[0] for x in lps])
    b = np.stack([x[1] for x in lps])
    c = np.stack([x[2] for x in lps])
    opts = dict(eps=EPS, max_iter=1000, algorithm=1, cost_shift=1, pivot_tol=1e-9)
    bs = lp.solve_batch(A, b, c, trace_cap=1000, **opts)
    for i in range(k):
        one = lp.solve(A[i], b[i], c[i], **opts)
        ref = _ref(A[i], b[i], c[i], np.float64, 1000, pivot_tol=1e-9)
        assert (int(one.status), one.iterations, one.pivots, one.z) == (ref.status, ref.iterations, ref.pivots, ref.z)
        assert np.array_equal(one.x_b, ref.x_b) and np.array_equal(one.trace[:, 0], ref.trace_p)
        s = bs.solution(i)
        assert (s.status, s.iterations, s.pivots, s.z) == (one.status, one.iterations, one.pivots, one.z)
        assert np.array_equal(s.x_b, one.x_b) and np.array_equal(s.b_ixs, one.b_ixs)
        assert np.array_equal(s.trace, one.trace) and np.array_equal(bs.y[i], ref.y)
    assert int(bs.status[3]) == int(lp.SolveStatus.Infeasible)


def test_large_feasible_to_optimality():
    """m = 4096, n = 8192 (fp64), feasible family: optimum with primal and dual residuals and the duality gap checked
    on the host from x_b, b_ixs and y"""
    import simplex_method_gpu_b200 as lp
    m, n = 4096, 8192
    A, b, c = D.gen_general(m, n, 1, "feasible")
    with lp.Engine(m, n, dtype=np.float64, eps=EPS, max_iter=10 ** 6, algorithm=1, cost_shift=1, pivot_tol=1e-9) as e:
        e.upload(A, b, c)
        r = e.run(10 ** 6)
        x_b, b_ixs, y = e.download()
        ph = e.phase_info()
    assert r["status"] == lp.SolveStatus.OptimumFound and ph["phase"] == 2 and ph["phase1_pivots"] > 0
    x = np.zeros(n)
    x[b_ixs] = x_b
    scale_b = max(1.0, np.abs(b).max())
    assert x.min() >= -1e-9 * scale_b
    assert (A @ x - b).max() <= 1e-9 * scale_b
    assert (y @ A - c).min() >= -1e-9 * max(1.0, np.abs(c).max())
    primal, dual = c @ x, y @ b
    assert abs(primal - dual) <= 1e-9 * max(1.0, abs(primal))
    assert abs(r["z"] - primal) <= 1e-9 * max(1.0, abs(primal))


def test_cli_cost_shift(tmp_path):
    """bin/solver.out --dual --cost-shift: max x0 + x1, x0 + x1 >= 1, x0 + 2 x1 <= 4, 3 x0 + x1 <= 6 (optimum 2.8 at
    (1.6, 1.2)), and an infeasible LP with positive costs"""
    import os
    import subprocess
    import simplex_method_gpu_b200 as lp
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cli = os.path.join(root, "bin", "solver.out")
    f = tmp_path / "mixed.txt"
    lp.write_lp(str(f), np.array([[-1.0, -1.0, 1.0, 0.0, 0.0], [1.0, 2.0, 0.0, 1.0, 0.0], [3.0, 1.0, 0.0, 0.0, 1.0]]),
                np.array([-1.0, 4.0, 6.0]), np.array([1.0, 1.0, 0.0, 0.0, 0.0]))
    out = subprocess.run([cli, str(f), "--f64", "--dual", "--cost-shift", "--max-iter", "20"], capture_output=True,
                         text=True, check=True).stdout
    assert "Optimum found: 2.8\n" in out and "\tx_0 = 1.6\n" in out and "\tx_1 = 1.2\n" in out, out
    g = tmp_path / "infeasible.txt"
    lp.write_lp(str(g), np.array([[1.0, 1.0, 1.0, 0.0], [-1.0, -1.0, 0.0, 1.0]]), np.array([1.0, -3.0]),
                np.array([1.0, 2.0, 0.0, 0.0]))
    out = subprocess.run([cli, str(g), "--f64", "--dual", "--cost-shift", "--max-iter", "20"], capture_output=True,
                         text=True, check=True).stdout
    assert "Problem infeasible.\n" in out, out
