"""Dual simplex and composite method in the batch kernel (simplex_tiny_batch_dual: solve_batch with algorithm=1, with
and without cost_shift=1): every output of LP k equals, bit for bit, the order-1 CPU reference on LP k and the single
call on LP k alone (y: Engine.download() after a run)."""
import re

import numpy as np
import pytest

import dual_oracle as D

pytestmark = pytest.mark.gpu

EPS = 1e-9
LD = {np.float64: 64, np.float32: 128}        # one warp-wide vector row: the largest m of the tiny kernels


@pytest.fixture(scope="module")
def lp(engine_lib):
    import simplex_method_gpu_b200 as s
    was = s.set_memory_cache(True)            # single calls of one shape reuse their engine: the loops stay quick
    yield s
    s.set_memory_cache(was)


def bits(a):
    return np.ascontiguousarray(a).view(np.uint8)


def same_float(x, y):
    return np.float64(x).tobytes() == np.float64(y).tobytes()


def _eps(dt, composite=False):
    # fp32 composite: the primal phase needs a tolerance above its rounding noise to stop
    if dt == np.float32:
        return float(np.float32(1e-5 if composite else EPS))
    return EPS


def check(lp, bs, A, b, c, k, dt, eps, max_iter, tag, **opts):
    """LP k of the batch against the CPU reference (every output, y included) and the single call."""
    ref = D.solve(np.asfortranarray(A[k]), b[k], c[k], eps=dt(eps), max_iter=max_iter, order=1,
                  pivot_tol=float(dt(opts.get("pivot_tol", 0.0))), cost_shift=opts.get("cost_shift", 0),
                  shift_delta=opts.get("shift_delta", 0.0))
    assert (int(bs.status[k]), bs.iterations[k], bs.pivots[k]) == (ref.status, ref.iterations, ref.pivots), tag
    h = min(int(bs.pivots[k]), bs.trace.shape[1])
    assert bs.trace[k, :h, 0].tolist() == ref.trace_p[:h].tolist(), tag
    assert bs.trace[k, :h, 1].tolist() == ref.trace_q[:h].tolist(), tag
    assert (bs.trace[k, h:] == -1).all(), tag
    assert np.array_equal(bits(bs.x_b[k]), bits(ref.x_b)) and np.array_equal(bs.b_ixs[k], ref.b_ixs), tag
    assert np.array_equal(bits(bs.y[k]), bits(ref.y)), tag
    assert same_float(bs.z[k], ref.z) and same_float(bs.min_reduced_cost[k], ref.min_e), tag
    sol = lp.solve(A[k], b[k], c[k], eps=eps, max_iter=max_iter, algorithm=1, **opts)
    assert (int(bs.status[k]), bs.iterations[k], bs.pivots[k]) == (int(sol.status), sol.iterations, sol.pivots), tag
    assert np.array_equal(bs.trace[k, :h], sol.trace[:h]), tag
    assert np.array_equal(bits(bs.x_b[k]), bits(sol.x_b)) and np.array_equal(bs.b_ixs[k], sol.b_ixs), tag
    assert same_float(bs.z[k], sol.z) and same_float(bs.min_reduced_cost[k], sol.min_reduced_cost), tag
    assert lp.format_result(bs.solution(k)) == lp.format_result(sol), tag
    return ref


def check_y_vs_engine(lp, bs, A, b, c, ks, dt, eps, max_iter, tag, **opts):
    _, m, n = A.shape
    with lp.Engine(m, n, dt, eps=eps, max_iter=max_iter, algorithm=1, **opts) as e:
        for k in ks:
            e.upload(np.asfortranarray(A[k]), b[k], c[k])
            e.run(max_iter)
            x_b, _, y = e.download()
            assert np.array_equal(bits(bs.y[k]), bits(y)) and np.array_equal(bits(bs.x_b[k]), bits(x_b)), (tag, k)


def covering(rng, m, n):
    """gen_covering's family with random numbers: min c_s.x, A_s x >= b_s written as <= rows (negative b)."""
    ns = n - m
    A = np.zeros((m, n))
    A[:, :ns] = -rng.uniform(0.0, 1.0, (m, ns))
    A[:, ns:] = np.eye(m)
    b = -(max(ns, 1) / 2) * rng.uniform(1.0, 2.0, m)
    c = np.zeros(n)
    c[:ns] = -rng.uniform(0.5, 1.5, ns)
    return A, b, c


def dual_batch(rng, batch, m, n, dt, data_slack=True):
    """Mixed kinds: covering, infeasible (a row sum(x) <= 0.01 next to the covering rows), a positive cost (not dual
    feasible), b >= 0 with c <= 0 (optimal at the start), and covering LPs whose slack block is data (data_slack; else
    a sixth covering LP)."""
    ns = n - m
    As, bs, cs = [], [], []
    for k in range(batch):
        A, b, c = covering(rng, m, n)
        kind = k % 6
        if kind == 2:
            A[m - 1, :ns] = 1.0
            b[m - 1] = 0.01
        elif kind == 3 and ns > 0:
            c[int(rng.integers(0, ns))] = 0.5
        elif kind == 4:
            b = -b
        elif kind == 5 and data_slack:
            A[:, ns:] += np.diag(rng.uniform(0.1, 0.5, m))
            A[0, n - 1] = 0.25
        As.append(A)
        bs.append(b)
        cs.append(c)
    return np.stack(As).astype(dt), np.stack(bs).astype(dt), np.stack(cs).astype(dt)


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_dual_mixed_statuses_bit_exact(lp, dt):
    """Ragged tiny shapes (n == m, m == LD and n - m odd included), every status of the dual loop in one run."""
    ld = LD[dt]
    eps = _eps(dt)
    rng = np.random.default_rng(20261022 + ld)
    seen = set()
    shapes = [(1, 1), (1, 7), (ld, ld), (ld - 1, 2 * ld), (17, 60), (33, 90), (24, 70)]
    for m, n in shapes:
        batch = int(rng.integers(40, 90))
        # LPs with the slack block stored (ns = n) only where that still fits the kernel: at (LD - 1, 2 LD) in fp32
        # all 256 columns of A do not fit 200 KB of shared memory, and such a batch runs on the one-engine path
        A, b, c = dual_batch(rng, batch, m, n, dt, data_slack=_dual_fits(m, n, n, np.dtype(dt).itemsize)[1])
        max_iter = 3 if (m, n) == (24, 70) else int(rng.integers(m + 2, 3 * m + 8))   # (24, 70): capped runs
        bs = lp.solve_batch(A, b, c, eps=eps, max_iter=max_iter, trace_cap=max_iter, algorithm=1)
        assert bs.kernel_launches == 1, (m, n)
        for k in range(batch):
            seen.add(check(lp, bs, A, b, c, k, dt, eps, max_iter, (m, n, k, dt.__name__)).status)
        check_y_vs_engine(lp, bs, A, b, c, range(0, batch, 5), dt, eps, max_iter, (m, n))
    assert seen == {D.MAX_ITER, D.OPTIMUM, D.INFEASIBLE, D.NOT_DUAL_FEASIBLE}
    # the slack-basis optimum (b >= 0, c <= 0) stops in the first iteration without a pivot
    A, b, c = dual_batch(rng, 5, 9, 20, dt)
    bs = lp.solve_batch(A[4:5], b[4:5], c[4:5], eps=eps, max_iter=50, algorithm=1)
    assert (bs.status[0], bs.iterations[0], bs.pivots[0]) == (D.OPTIMUM, 1, 0)


def general_batch(m, n, seed0, kinds, dt):
    probs = [D.gen_general(m, n, seed0 + i, kind) for i, kind in enumerate(kinds)]
    return (np.stack([p[0] for p in probs]).astype(dt), np.stack([p[1] for p in probs]).astype(dt),
            np.stack([p[2] for p in probs]).astype(dt))


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["f64", "f32"])
def test_composite_kinds_bit_exact(lp, dt):
    """gen_general's four families (pivot_tol = 1e-9 for the degenerate one's sake), b >= 0 LPs (every column with
    e_j < -eps is shifted, phase 1 stops at once, phase 2 does the work) and covering LPs (nothing is shifted)."""
    m, n = 32, 96
    eps = _eps(dt, True)
    cap = 100000 if dt == np.float64 else 3000
    kinds = [D.GENERAL_KINDS[i % 4] for i in range(48)]
    A, b, c = general_batch(m, n, 300, kinds, dt)
    rng = np.random.default_rng(3)
    for k in range(48, 60):                            # b >= 0
        Ak, bk, ck = D.gen_general(m, n, 300 + k, "feasible")
        A = np.concatenate([A, Ak[None].astype(dt)])
        b = np.concatenate([b, np.abs(bk)[None].astype(dt)])
        c = np.concatenate([c, ck[None].astype(dt)])
    for k in range(60, 70):                            # covering
        Ak, bk, ck = covering(rng, m, n)
        A = np.concatenate([A, Ak[None].astype(dt)])
        b = np.concatenate([b, bk[None].astype(dt)])
        c = np.concatenate([c, ck[None].astype(dt)])
    opts = dict(cost_shift=1, pivot_tol=1e-9)
    bs = lp.solve_batch(A, b, c, eps=eps, max_iter=cap, trace_cap=cap, algorithm=1, **opts)
    assert bs.kernel_launches == 1
    refs = [check(lp, bs, A, b, c, k, dt, eps, cap, (k, dt.__name__), **opts) for k in range(len(b))]
    check_y_vs_engine(lp, bs, A, b, c, range(0, len(b), 3), dt, eps, cap, "composite", **opts)
    assert all(r.phase == 2 and r.shifted > 0 and r.phase1_pivots == 0 for r in refs[48:60])
    assert all(r.shifted == 0 for r in refs[60:])
    if dt == np.float64:                               # fp32: the same bits, whatever status the rounding leads to
        assert {r.status for r in refs[:48]} == {D.OPTIMUM, D.INFEASIBLE, D.UNBOUNDED}
        assert all(r.status == D.OPTIMUM for r in refs[60:])


def test_composite_caps_and_shift_delta(lp):
    """Budgets that end inside phase 1, exactly on the phase-1 optimum (phase-1 pivots + 1: MAX_ITER with the
    original-c z) and inside phase 2; and a non-default shift_delta."""
    m, n = 32, 96
    A, b, c = general_batch(m, n, 500, ["feasible"] * 24, np.float64)
    full = [D.solve(np.asfortranarray(A[k]), b[k], c[k], eps=EPS, max_iter=100000, order=1, cost_shift=1)
            for k in range(24)]
    k0 = next(k for k, r in enumerate(full) if r.phase == 2 and r.phase1_pivots > 0 and r.pivots > r.phase1_pivots + 3)
    p1 = full[k0].phase1_pivots
    for budget in (p1, p1 + 1, p1 + 3):
        bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=budget, trace_cap=budget, algorithm=1, cost_shift=1)
        assert bs.kernel_launches == 1
        refs = [check(lp, bs, A, b, c, k, np.float64, EPS, budget, (budget, k), cost_shift=1) for k in range(24)]
        r = refs[k0]
        want = {p1: (1, p1), p1 + 1: (2, p1), p1 + 3: (2, p1 + 2)}[budget]
        assert (r.status, r.phase, r.pivots) == (D.MAX_ITER, *want), budget
        check_y_vs_engine(lp, bs, A, b, c, [k0], np.float64, EPS, budget, budget, cost_shift=1)
    bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=100000, trace_cap=0, algorithm=1, cost_shift=1, shift_delta=1e-3)
    assert bs.kernel_launches == 1
    for k in range(24):
        check(lp, bs, A, b, c, k, np.float64, EPS, 100000, ("delta", k), cost_shift=1, shift_delta=1e-3)


def test_many_waves(lp):
    """20 000 dual LPs: every CTA takes many tickets; every LP equals the reference."""
    m, n, batch = 16, 48, 20000
    rng = np.random.default_rng(17)
    A, b, c = dual_batch(rng, batch, m, n, np.float64)
    bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=200, trace_cap=200, algorithm=1)
    assert bs.kernel_launches == 1
    for k in range(batch):
        ref = D.solve(np.asfortranarray(A[k]), b[k], c[k], eps=EPS, max_iter=200, order=1)
        assert (int(bs.status[k]), bs.iterations[k], bs.pivots[k]) == (ref.status, ref.iterations, ref.pivots), k
        assert np.array_equal(bits(bs.x_b[k]), bits(ref.x_b)) and np.array_equal(bits(bs.y[k]), bits(ref.y)), k
        assert np.array_equal(bs.b_ixs[k], ref.b_ixs) and same_float(bs.z[k], ref.z), k
        h = int(ref.pivots)
        assert bs.trace[k, :h, 0].tolist() == ref.trace_p.tolist(), k
    for k in range(0, batch, 997):
        check(lp, bs, A, b, c, k, np.float64, EPS, 200, k)


def _dual_fits(m, n, ns, itemsize):
    """tiny_fits and tiny_dual_fits of engine.cu from TinyLayout / TinyDualLayout: (primal, dual)"""
    ld = 512 // itemsize                               # one warp of 16-byte vectors
    end = ld * ns + ld * m + 15 * ld + (n + 3) // 4 * 4
    primal = end * itemsize + 4 * m + 16
    return m <= ld and primal <= 200 * 1024, m <= ld and primal + n <= 200 * 1024


def test_fallback_paths(lp):
    """Outside the kernel's conditions the LPs run one after another on one engine: still the single call's bits."""
    rng = np.random.default_rng(9)
    # f64 beyond the tiny limit (m = 100 > 64 doubles)
    A, b, c = dual_batch(rng, 6, 100, 180, np.float64)
    bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=400, trace_cap=400, algorithm=1)
    assert bs.kernel_launches > 1
    for k in range(6):
        check(lp, bs, A, b, c, k, np.float64, EPS, 400, ("m100", k))
    # max_iter = 0: nothing runs, the slack basis comes back
    A, b, c = dual_batch(rng, 4, 10, 30, np.float64)
    for opts in ({}, {"cost_shift": 1}):
        bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=0, algorithm=1, **opts)
        assert bs.kernel_launches > 1
        for k in range(4):
            sol = lp.solve(A[k], b[k], c[k], eps=EPS, max_iter=0, algorithm=1, **opts)
            assert bs.iterations[k] == 0 and int(bs.status[k]) == int(sol.status), k
            assert np.array_equal(bits(bs.x_b[k]), bits(sol.x_b)) and same_float(bs.z[k], sol.z), k
    # a shape inside tiny_fits (the primal batch kernel takes it) but outside tiny_dual_fits (the mask does not fit)
    m, n = next((m, n) for m in range(1, 65) for n in range(m, 400) if _dual_fits(m, n, n - m, 8) == (True, False))
    A, b, c = dual_batch(rng, 3, m, n, np.float64)
    assert lp.solve_batch(A, np.abs(b), c, eps=EPS, max_iter=5).kernel_launches == 1
    assert lp.solve_batch(A, b, c, eps=EPS, max_iter=5, algorithm=1, cost_shift=1).kernel_launches > 1
    m2, n2 = m, n - 4                                    # just inside: the dual kernel
    assert _dual_fits(m2, n2, n2 - m2, 8)[1]
    A2, b2, c2 = dual_batch(rng, 3, m2, n2, np.float64)
    assert lp.solve_batch(A2, b2, c2, eps=EPS, max_iter=5, algorithm=1).kernel_launches == 1
    bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=60, trace_cap=60, algorithm=1)
    assert bs.kernel_launches > 1
    for k in range(3):
        check(lp, bs, A, b, c, k, np.float64, EPS, 60, ("edge", k))


def _kernel_names(prof):
    """base names of the CUDA kernels the profiler saw ("void b200lp::simplex_tiny<double>(...)" -> simplex_tiny)"""
    out = set()
    for ev in prof.events():
        s = re.sub(r"^void ", "", ev.name)
        s = re.split(r"[<(]", s, maxsplit=1)[0]
        out.add(s.rsplit("::", 1)[-1])
    return out


def test_profiler_one_kernel(lp):
    """A dual and a composite batch each launch the dual batch kernel once, and none of the single-LP kernels."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    rng = np.random.default_rng(4)
    A, b, c = dual_batch(rng, 200, 32, 96, np.float64)
    Ag, bg, cg = general_batch(32, 96, 700, ["feasible"] * 50, np.float64)
    for args, opts in (((A, b, c), {}), ((Ag, bg, cg), {"cost_shift": 1})):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            bs = lp.solve_batch(*args, eps=EPS, max_iter=1000, algorithm=1, **opts)
            torch.cuda.synchronize()
        assert bs.kernel_launches == 1
        names = [n for n in _kernel_names(prof) if n.startswith(("simplex_", "k_"))]
        kern = [ev for ev in prof.events() if "simplex_tiny_batch_dual" in ev.name]
        assert names == ["simplex_tiny_batch_dual"], (opts, names)
        assert len(kern) == 1, opts
        for k in (0, 7, 13):
            check(lp, bs, *args, k, np.float64, EPS, 1000, (opts, k), **opts)


def test_covering_optimum_against_highs(lp):
    """Independent of the reference: the optimal objectives of a covering batch equal HiGHS's to 1e-9 relative."""
    from scipy.optimize import linprog
    rng = np.random.default_rng(31)
    m, n, batch = 32, 96, 64
    A, b, c = (np.stack(x) for x in zip(*[covering(rng, m, n) for _ in range(batch)]))
    bs = lp.solve_batch(A, b, c, eps=EPS, max_iter=100000, algorithm=1)
    assert bs.kernel_launches == 1
    ns = n - m
    for k in range(batch):
        r = linprog(-c[k, :ns], A_ub=A[k, :, :ns], b_ub=b[k], bounds=(0, None), method="highs")
        assert r.status == 0 and bs.status[k] == D.OPTIMUM, k
        assert abs(bs.z[k] - (-r.fun)) <= 1e-9 * abs(r.fun), (k, bs.z[k], -r.fun)
