"""Touched-column passes of simplex_persistent (Engine(binv_sparse=...)): streaming only the columns of B^-1 that have
left e_j must not change a single bit.  Every case runs the same LP with an explicit K* (m unless stated: every
pass sparse, below the auto setting's size gate too) and with -1 (every pass dense) and compares trace, x_b, b_ixs,
y, z and B^-1 through their raw bits (a -0 shows), and, with steepest edge, v = B^-T alpha and the weights; b200lp_binv_info shows that the sparse arm took the sparse
pass; then the trace, x_b, b_ixs and z against the oracle in the engine's summation order (order = 1)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def _state(e, se):
    x_b, b_ixs, y = e.download()
    st = {"trace": e.trace(), "x_b": _bits(x_b), "b_ixs": b_ixs, "y": _bits(y)}
    if se:                                           # steepest edge: v = B^-T alpha of the last pivot and the weights
        st["vbt"], st["gamma"] = _bits(e.vector("vbt")), _bits(e.vector("gamma"))
    info = e.binv_info()                             # before download_binv, which applies a pending update densely
    st["binv"] = _bits(e.download_binv())
    return st, info


def _run(lp, A, b, c, dtype, eps, windows, sparse, after=None, **kw):
    """windows of the persistent kernel (resident = -1); `after(e, k)` runs between windows"""
    m, n = A.shape
    with lp.Engine(m, n, dtype, eps=eps, max_iter=1 << 20, resident=-1, binv_sparse=sparse, **kw) as e:
        e.upload(A, b, c)
        zs = []
        for k, w in enumerate(windows):
            r = e.run(w)
            zs.append((r["z"], int(r["status"]), r["pivots"]))
            if after:
                after(e, k)
        st, info = _state(e, kw.get("pricing_rule", 0) == 1)
        return st, zs, info


def _compare(lp, oracle, A, b, c, dtype, eps, windows, sparse=None, after=None, want_oracle=True, **kw):
    m = A.shape[0]
    sparse = m if sparse is None else sparse         # default: sparse passes whatever |K| and m
    s, zs, si = _run(lp, A, b, c, dtype, eps, windows, sparse, after, **kw)
    d, zd, di = _run(lp, A, b, c, dtype, eps, windows, -1, after, **kw)
    assert si["sparse_passes"] > 0 and di["sparse_passes"] == 0, (si, di)   # the sparse arm did take the sparse pass
    assert si["touched"] == di["touched"] > 0
    assert zs == zd
    for k in s:
        assert np.array_equal(s[k], d[k]), k
    assert len(s["trace"]) > 0
    if want_oracle:
        okw = {k: kw[k] for k in ("pivot_tol", "ratio_mode", "harris_delta", "pricing_rule") if k in kw}
        ref = oracle.solve(A, b, c, eps=eps, max_iter=sum(windows), order=1, **okw)
        assert s["trace"][:, 0].tolist() == ref.trace_p.tolist() and s["trace"][:, 1].tolist() == ref.trace_q.tolist()
        assert np.array_equal(s["x_b"], _bits(ref.x_b)) and np.array_equal(s["b_ixs"], ref.b_ixs)
        assert zs[-1][0] == ref.z
    return s


CASES = [
    # m, n, dtype, eps, windows, options
    (300, 701, np.float64, 1e-9, [1 << 20], {}),                                  # ragged m, ns % 4 != 0
    (1024, 2048, np.float64, 1e-9, [1 << 20], {}),
    (1000, 2003, np.float64, 1e-9, [37, 100, 1 << 20], {"tile_shape": 1}),        # windows: pending update at the edge
    (777, 1600, np.float64, 1e-9, [1 << 20], {"grid_ctas": 3, "tile_shape": 2}),
    (513, 1100, np.float64, 1e-9, [50, 1 << 20], {"grid_ctas": 1, "tile_shape": 8}),
    (500, 1203, np.float32, 1e-4, [1 << 20], {"tile_shape": 4}),
    (640, 1500, np.float64, 1e-9, [1 << 20], {"pivot_tol": 1e-9}),
    (640, 1500, np.float64, 1e-9, [1 << 20], {"ratio_mode": 1}),
    (640, 1500, np.float64, 1e-9, [1 << 20], {"ratio_mode": 2, "harris_delta": 1e-9}),
    (600, 1300, np.float64, 1e-9, [41, 1 << 20], {"pricing_rule": 1}),            # steepest edge: sparse BTRAN
    (300, 800, np.float32, 1e-4, [1 << 20], {"pricing_rule": 1}),
]


@pytest.mark.parametrize("m,n,dtype,eps,windows,kw", CASES)
def test_sparse_equals_dense(oracle, engine_lib, m, n, dtype, eps, windows, kw):
    import simplex_method_gpu_b200 as lp
    A, b, c = oracle.gen_dense(m, n, 1, dtype)
    s = _compare(lp, oracle, A, b, c, dtype, eps, windows, **kw)
    basis = s["b_ixs"]
    assert (basis < n - m).any()                    # structural columns entered


def test_threshold_crossed_inside_a_window(oracle, engine_lib):
    """an explicit K* of 20: the kernel switches to the dense pass in the middle of the window"""
    import simplex_method_gpu_b200 as lp
    m, n = 800, 1700
    A, b, c = oracle.gen_dense(m, n, 3)
    for sparse in (20, 1):
        _compare(lp, oracle, A, b, c, np.float64, 1e-9, [300], sparse=sparse)
    _compare(lp, oracle, A, b, c, np.float64, 1e-9, [60], sparse=20, pricing_rule=1)


def test_slack_columns_reenter(oracle, engine_lib):
    """a long solve: slack columns leave and enter again (unit a_p), the touched set keeps growing"""
    import simplex_method_gpu_b200 as lp
    m, n = 256, 520
    A, b, c = oracle.gen_dense(m, n, 7)
    s = _compare(lp, oracle, A, b, c, np.float64, 1e-9, [1 << 20])
    tr = s["trace"]
    assert (tr[:, 0] >= n - m).any()                 # a slack column entered


def test_slack_block_stored_as_data(oracle, engine_lib):
    import simplex_method_gpu_b200 as lp
    m, n = 320, 700
    A, b, c = oracle.gen_dense(m, n, 2)
    A = A.copy(order="F")
    A[3, n - 1] = 0.25                               # not the identity: all n columns are stored and priced
    _compare(lp, oracle, A, b, c, np.float64, 1e-9, [40, 1 << 20])


def test_refactor_and_check_basis_mid_solve(oracle, engine_lib):
    """refactor rebuilds B^-1 (and the touched set through its replays), then more pivots; check_basis between"""
    import simplex_method_gpu_b200 as lp
    m, n = 700, 1500
    A, b, c = oracle.gen_dense(m, n, 4)
    def after(e, k):
        err, scale = e.check_basis()
        assert err <= 1e-6 * max(1.0, scale)
        if k == 0:
            assert e.refactor() > 0
    _compare(lp, oracle, A, b, c, np.float64, 1e-9, [120, 1 << 20], after=after, want_oracle=False)
    with lp.Engine(m, n, np.float64, eps=1e-9, max_iter=1 << 20, resident=-1, binv_sparse=m) as e:
        e.upload(A, b, c)
        r, nref = e.run_guarded(1 << 20, 100, 1e-30)         # a refactorisation after every window
        assert nref >= 1 and r["status"] == lp.SolveStatus.OptimumFound
        assert e.binv_info()["sparse_passes"] > 0
        z_sparse = r["z"]
    with lp.Engine(m, n, np.float64, eps=1e-9, max_iter=1 << 20, resident=-1, binv_sparse=-1) as e:
        e.upload(A, b, c)
        r, nref2 = e.run_guarded(1 << 20, 100, 1e-30)
        assert nref2 == nref and r["z"] == z_sparse


def test_auto_setting(oracle, engine_lib):
    """auto (binv_sparse = 0): LPs below the size gate stream all of B^-1; above it, sparse while |K| <= m / 8"""
    import simplex_method_gpu_b200 as lp
    for m, n, want in ((1024, 2048, False), (4096, 8192, True)):
        A, b, c = oracle.gen_dense(m, n, 1)
        with lp.Engine(m, n, np.float64, eps=1e-9, max_iter=1 << 20, resident=-1, pricing_rule=1) as e:
            e.upload(A, b, c)
            e.run(30)
            assert (e.binv_info()["sparse_passes"] > 0) == want, m


def test_binv_sparse_rejects_bad_values(engine_lib):
    import simplex_method_gpu_b200 as lp
    with pytest.raises(lp.capi.B200LPError):
        lp.Engine(300, 600, np.float64, binv_sparse=-2)
