"""Batched solve (b200lp_solve_batch_*, solve_batch) on the GPU: every output of LP k equals, bit for bit, the
engine-order oracle on LP k and the single call on LP k alone (y: Engine.download() after a run)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


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


def assert_vs_oracle(bs, k, ref, tag):
    assert int(bs.status[k]) == ref.status and bs.iterations[k] == ref.iterations and bs.pivots[k] == ref.pivots, tag
    h = min(int(bs.pivots[k]), bs.trace.shape[1])
    assert bs.trace[k, :h, 0].tolist() == ref.trace_p[:h].tolist(), tag
    assert bs.trace[k, :h, 1].tolist() == ref.trace_q[:h].tolist(), tag
    assert (bs.trace[k, h:] == -1).all(), tag
    assert np.array_equal(bits(bs.x_b[k]), bits(ref.x_b)) and np.array_equal(bs.b_ixs[k], ref.b_ixs), tag
    assert same_float(bs.z[k], ref.z), tag


def assert_vs_single(bs, k, sol, tag):
    assert int(bs.status[k]) == int(sol.status) and bs.iterations[k] == sol.iterations and bs.pivots[k] == sol.pivots, tag
    h = min(int(bs.pivots[k]), bs.trace.shape[1])
    assert np.array_equal(bs.trace[k, :h], sol.trace[:h]), tag
    assert np.array_equal(bits(bs.x_b[k]), bits(sol.x_b)) and np.array_equal(bs.b_ixs[k], sol.b_ixs), tag
    assert same_float(bs.z[k], sol.z) and same_float(bs.min_reduced_cost[k], sol.min_reduced_cost), tag
    s = bs.solution(k)
    assert s.status == sol.status and np.array_equal(s.trace, sol.trace[:h]) and s.z == sol.z, tag


def assert_y_vs_engine(lp, bs, As, bs_b, bs_c, ks, eps, max_iter, dt, tag, **opts):
    _, m, n = As.shape
    with lp.Engine(m, n, dt, eps=eps, max_iter=max_iter, **opts) as e:
        for k in ks:
            e.upload(np.asfortranarray(As[k]), bs_b[k], bs_c[k])
            e.run(max_iter)
            x_b, b_ixs, y = e.download()
            assert np.array_equal(bits(bs.y[k]), bits(y)) and np.array_equal(bits(bs.x_b[k]), bits(x_b)), (tag, k)


def fuzz_batch(rng, batch, m, n, dt):
    """LPs of one shape, mixed kinds: regular, optimal at the slack basis, degenerate (b_i = 0), unbounded."""
    ns = n - m
    A = np.zeros((batch, m, n))
    b = np.zeros((batch, m))
    c = np.zeros((batch, n))
    for k in range(batch):
        kind = k % 5
        A[k, :, :ns] = rng.uniform(-0.3 if kind == 4 else 0.0, 1.0, (m, ns))
        A[k, :, ns:] = np.eye(m)
        b[k] = rng.uniform(1.0, 2.0, m) * max(ns, 1)
        c[k, :ns] = rng.uniform(-0.5 if kind == 4 else 0.1, 1.0, ns)
        if kind == 1:
            c[k, :ns] = -np.abs(c[k, :ns])                          # optimal at the slack basis
        elif kind == 2:
            b[k, rng.integers(0, m)] = 0.0                          # degenerate vertex, zero-length steps
        elif kind == 3 and ns > 0:
            A[k, :, 0] = -np.abs(A[k, :, 0])                         # column 0 never blocks
            c[k, 0] = 10.0                                          # ... and enters first: unbounded
    return A.astype(dt), b.astype(dt), c.astype(dt)


@pytest.mark.parametrize("dt,eps,mmax", [(np.float64, 1e-9, 64), (np.float32, 1e-4, 128)])
def test_fuzz_mixed_statuses_bit_exact(lp, oracle, dt, eps, mmax):
    """Ragged tiny shapes (n == m included): optimal-at-start, degenerate, unbounded and max_iter-capped LPs in one
    batch, each equal to the oracle and to its single call."""
    rng = np.random.default_rng(20261021 + mmax)
    seen = set()
    shapes = [(1, 1), (1, 7), (5, 5), (mmax, mmax), (mmax, mmax + 40), (mmax - 1, 2 * mmax), (17, 60), (33, 90)]
    for si, (m, n) in enumerate(shapes):
        batch = int(rng.integers(50, 301)) if si < 4 else int(rng.integers(50, 120))
        A, b, c = fuzz_batch(rng, batch, m, n, dt)
        max_iter = int(rng.integers(m // 2 + 2, 2 * m + 8))       # some LPs need more: capped
        bs = lp.solve_batch(A, b, c, eps=eps, max_iter=max_iter, trace_cap=max_iter)
        assert bs.kernel_launches == 1, (m, n)                      # the batch kernel
        for k in range(batch):
            tag = (m, n, k, dt.__name__)
            ref = oracle.solve(np.asfortranarray(A[k]), b[k], c[k], eps=eps, max_iter=max_iter, order=1)
            assert_vs_oracle(bs, k, ref, tag)
            assert_vs_single(bs, k, lp.solve(A[k], b[k], c[k], eps=eps, max_iter=max_iter), tag)
            seen.add(ref.status)
        assert_y_vs_engine(lp, bs, A, b, c, range(0, batch, 7), eps, max_iter, dt, (m, n))
    assert seen == {oracle.MAX_ITER, oracle.OPTIMUM, oracle.UNBOUNDED}


def test_slack_blocks_mixed(lp, oracle):
    """LPs whose last m columns are the identity next to LPs where they are data (all n columns stored)."""
    rng = np.random.default_rng(7)
    m, n, batch = 20, 50, 60
    A, b, c = fuzz_batch(rng, batch, m, n, np.float64)
    for k in range(1, batch, 2):
        A[k, :, n - m:] += np.diag(rng.uniform(0.1, 0.5, m))          # slack block is data
        A[k, 0, n - 1] = 0.25
    bs = lp.solve_batch(A, b, c, eps=1e-9, max_iter=500, trace_cap=500)
    assert bs.kernel_launches == 1
    for k in range(batch):
        sol = lp.solve(A[k], b[k], c[k], eps=1e-9, max_iter=500)
        assert_vs_single(bs, k, sol, k)
        ref = oracle.solve(np.asfortranarray(A[k]), b[k], c[k], eps=1e-9, max_iter=500, order=1)
        assert_vs_oracle(bs, k, ref, k)
    assert_y_vs_engine(lp, bs, A, b, c, range(batch), 1e-9, 500, np.float64, "slack")


def test_klee_minty_uneven_work(lp, oracle):
    """256 Klee-Minty d = 12 copies (4095 pivots each, b scaled by 2^k) interleaved with LPs that are optimal at the
    start: the tickets see very uneven work, the results stay exact."""
    d = 12
    A0, b0, c0 = oracle.gen_klee_minty(d)
    m, n = A0.shape
    A = np.empty((512, m, n))
    b = np.empty((512, m))
    c = np.empty((512, n))
    for i in range(512):
        A[i] = A0
        if i % 2 == 0:
            b[i] = b0 * 2.0 ** ((i // 2) % 8)
            c[i] = c0
        else:
            b[i] = b0
            c[i] = -np.abs(c0)
    bs = lp.solve_batch(A, b, c, eps=1e-4, max_iter=1 << 13, trace_cap=16)
    assert bs.kernel_launches == 1
    ref = oracle.solve(A0, b0, c0, eps=1e-4, max_iter=1 << 13, order=1)
    for i in range(512):
        if i % 2 == 0:
            s = (i // 2) % 8
            assert bs.status[i] == 1 and bs.pivots[i] == 2 ** d - 1 and bs.z[i] == 5.0 ** d * 2.0 ** s, i
            assert bs.trace[i, :, 0].tolist() == ref.trace_p[:16].tolist(), i
            assert np.array_equal(bs.b_ixs[i], ref.b_ixs) and np.array_equal(bs.x_b[i], ref.x_b * 2.0 ** s), i
        else:
            assert bs.status[i] == 1 and bs.pivots[i] == 0 and bs.iterations[i] == 1 and (bs.trace[i] == -1).all(), i
    for i in (0, 2, 14, 1):
        sol = lp.solve(A[i], b[i], c[i], eps=1e-4, max_iter=1 << 13, trace_cap=16)
        assert_vs_single(bs, i, sol, i)


def test_assignment_against_scipy(lp, oracle):
    """200 assignment LPs: the optimum equals the maximum-weight assignment (independent of the oracle)."""
    from scipy.optimize import linear_sum_assignment
    k = 6
    probs = [oracle.gen_assignment(k, seed) for seed in range(1, 201)]
    A = np.stack([p[0] for p in probs])
    b = np.stack([p[1] for p in probs])
    c = np.stack([p[2] for p in probs])
    bs = lp.solve_batch(A, b, c, eps=1e-4, max_iter=1 << 12, trace_cap=1 << 12)
    assert bs.kernel_launches == 1
    for i, (Ai, bi, ci, w) in enumerate(probs):
        r, cidx = linear_sum_assignment(w, maximize=True)
        assert bs.status[i] == 1 and bs.z[i] == w[r, cidx].sum(), i
        ref = oracle.solve(Ai, bi, ci, eps=1e-4, max_iter=1 << 12, order=1)
        assert_vs_oracle(bs, i, ref, i)


def test_many_waves(lp, oracle):
    """20 000 LPs: every CTA takes many tickets; every LP equals the oracle."""
    m, n, batch = 16, 48, 20000
    rng = np.random.default_rng(11)
    A, b, c = fuzz_batch(rng, batch, m, n, np.float64)
    bs = lp.solve_batch(A, b, c, eps=1e-9, max_iter=200, trace_cap=200, want_y=False)
    assert bs.y is None and bs.kernel_launches == 1
    for k in range(batch):
        ref = oracle.solve(np.asfortranarray(A[k]), b[k], c[k], eps=1e-9, max_iter=200, order=1)
        assert_vs_oracle(bs, k, ref, k)
    for k in range(0, batch, 997):
        assert_vs_single(bs, k, lp.solve(A[k], b[k], c[k], eps=1e-9, max_iter=200), k)


def test_fallback_paths(lp, oracle):
    """Shapes and options outside the batch kernel run one LP after another on one engine: still the single call's
    bits.  kernel_launches tells the paths apart."""
    rng = np.random.default_rng(5)
    # f64 beyond the tiny limit (m = 100 > 64 doubles)
    A, b, c = fuzz_batch(rng, 6, 100, 180, np.float64)
    bs = lp.solve_batch(A, b, c, eps=1e-9, max_iter=400, trace_cap=400)
    assert bs.kernel_launches > 1
    for k in range(6):
        assert_vs_single(bs, k, lp.solve(A[k], b[k], c[k], eps=1e-9, max_iter=400), k)
        assert_vs_oracle(bs, k, oracle.solve(np.asfortranarray(A[k]), b[k], c[k], eps=1e-9, max_iter=400, order=1), k)
    assert_y_vs_engine(lp, bs, A, b, c, range(6), 1e-9, 400, np.float64, "m100")
    # steepest edge on a tiny shape
    A, b, c = fuzz_batch(rng, 8, 12, 30, np.float64)
    bs = lp.solve_batch(A, b, c, eps=1e-9, max_iter=300, trace_cap=300, pricing_rule=1)
    assert bs.kernel_launches > 1
    for k in range(8):
        assert_vs_single(bs, k, lp.solve(A[k], b[k], c[k], eps=1e-9, max_iter=300, pricing_rule=1), k)
    assert_y_vs_engine(lp, bs, A, b, c, range(8), 1e-9, 300, np.float64, "se", pricing_rule=1)


def test_trace_cap_and_optional_outputs(lp, oracle):
    A0, b0, c0 = oracle.gen_klee_minty(6)
    A, b, c = A0[None], b0[None], c0[None]
    ref = oracle.solve(A0, b0, c0, eps=1e-4, max_iter=1 << 10, order=1)
    assert ref.pivots == 63
    bs = lp.solve_batch(A, b, c, eps=1e-4, max_iter=1 << 10, trace_cap=10)   # batch == 1, cap < pivots
    assert bs.trace.shape == (1, 10, 2)
    assert_vs_oracle(bs, 0, ref, "cap10")
    bs0 = lp.solve_batch(A, b, c, eps=1e-4, max_iter=1 << 10, trace_cap=0, want_y=False)
    assert bs0.trace.shape == (1, 0, 2) and bs0.y is None
    assert bs0.pivots[0] == 63 and np.array_equal(bs0.x_b, bs.x_b) and same_float(bs0.z[0], bs.z[0])
    # a non-NULL trace buffer with trace_cap = 0 receives nothing
    import ctypes as C
    from simplex_method_gpu_b200 import capi
    L = capi.lib()
    o = capi.default_options(eps=1e-4, max_iter=1 << 10)
    Ac = np.ascontiguousarray(A.transpose(0, 2, 1))
    x_b = np.zeros((1, 6))
    bix = np.zeros((1, 6), np.int32)
    tr = np.full((4, 2), 7, np.int32)
    res = (capi.Result * 1)()
    vp = lambda a: a.ctypes.data_as(C.c_void_p)
    capi.check(L.b200lp_solve_batch_f64(vp(Ac), vp(b), vp(c), 1, 6, 12, C.byref(o), vp(x_b), vp(bix), None, vp(tr), 0, res))
    assert (tr == 7).all() and res[0].pivots == 63 and res[0].aborted == 0
