"""Dual simplex (options.algorithm = 1) on the host side: every combination it does not support is an argument
error returned before any device call, so these hold with or without a GPU; without one, a supported call fails
loudly (there is no CPU fallback)."""
import ctypes as C

import numpy as np
import pytest

# options that the dual loop rejects, each with algorithm = 1
_BAD = [dict(algorithm=2), dict(algorithm=-1), dict(algorithm=1, pricing_rule=1), dict(algorithm=1, ratio_mode=1),
        dict(algorithm=1, ratio_mode=2), dict(algorithm=1, mode=1), dict(algorithm=1, fuse_ratio=1)]


def _vp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _lp(m=2, n=4, dt=np.float64):
    A = np.zeros((m, n), dt, order="F")
    A[:, n - m:] = np.eye(m)
    A[:, :n - m] = -1
    return A, -np.ones(m, dt), -np.ones(n, dt)


def test_options_mirror_the_header(engine_lib):
    from simplex_method_gpu_b200 import capi
    assert C.sizeof(capi.Options) == engine_lib.b200lp_sizeof_options()
    o = capi.default_options()
    assert o.algorithm == 0                          # primal by default
    assert (capi.STATUS_INFEASIBLE, capi.STATUS_NOT_DUAL_FEASIBLE) == (4, 5)
    import simplex_method_gpu_b200 as s
    assert int(s.SolveStatus.Infeasible) == 4 and int(s.SolveStatus.NotDualFeasible) == 5


@pytest.mark.parametrize("bad", _BAD, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()))
def test_rejected_before_any_device_call(engine_lib, bad):
    from simplex_method_gpu_b200 import capi
    L = engine_lib
    A, b, c = _lp()
    o = capi.default_options(max_iter=10, **bad)
    h = C.c_void_p()
    assert L.b200lp_create(capi.F64, 2, 4, C.byref(o), C.byref(h)) == capi.ERR_ARG
    assert not h
    assert b"algorithm" in L.b200lp_last_error() or b"dual" in L.b200lp_last_error()
    x_b, bix, res = np.zeros(2), np.zeros(2, np.int32), capi.Result()
    assert L.b200lp_solve_f64(_vp(A), _vp(b), _vp(c), 2, 4, C.byref(o), _vp(x_b), _vp(bix), None, 0, C.byref(res)) == capi.ERR_ARG
    A3 = np.ascontiguousarray(np.stack([A, A]).transpose(0, 2, 1))
    b3, c3 = np.stack([b, b]), np.stack([c, c])
    xb3, bix3, res3 = np.zeros((2, 2)), np.zeros((2, 2), np.int32), (capi.Result * 2)()
    assert L.b200lp_solve_batch_f64(_vp(A3), _vp(b3), _vp(c3), 2, 2, 4, C.byref(o), _vp(xb3), _vp(bix3), None, None, 0,
                                    res3) == capi.ERR_ARG


@pytest.mark.parametrize("ndev", [2, 4])
def test_dual_on_several_gpus_rejected(engine_lib, ndev):
    from simplex_method_gpu_b200 import capi
    L = engine_lib
    A, b, c = _lp()
    o = capi.default_options(max_iter=10, algorithm=1)
    devs = (C.c_int32 * ndev)(*([0] * ndev))
    h = C.c_void_p()
    assert L.b200lp_create_multi(capi.F64, 2, 4, devs, ndev, C.byref(o), C.byref(h)) == capi.ERR_ARG
    assert L.b200lp_create_sharded(capi.F64, 2, 4, 0, ndev, C.byref(o), C.byref(h)) == capi.ERR_ARG
    x_b, bix, res = np.zeros(2), np.zeros(2, np.int32), capi.Result()
    assert L.b200lp_solve_f64_multi(_vp(A), _vp(b), _vp(c), 2, 4, C.byref(o), devs, ndev, _vp(x_b), _vp(bix), None, 0,
                                    C.byref(res)) == capi.ERR_ARG
    Af = A.astype(np.float32, order="F")
    assert L.b200lp_solve_f32_multi(_vp(Af), _vp(b.astype(np.float32)), _vp(c.astype(np.float32)), 2, 4, C.byref(o),
                                    devs, ndev, _vp(x_b.astype(np.float32)), _vp(bix), None, 0, C.byref(res)) == capi.ERR_ARG
    assert b"one GPU" in L.b200lp_last_error()


def test_python_front_ends_pass_algorithm_through(engine_lib):
    import simplex_method_gpu_b200 as s
    from simplex_method_gpu_b200 import capi
    A, b, c = _lp()
    with pytest.raises(capi.B200LPError) as ei:
        s.solve(A, b, c, algorithm=1, pricing_rule=1)
    assert ei.value.code == capi.ERR_ARG
    with pytest.raises(capi.B200LPError) as ei:
        s.solve_batch(np.stack([A, A]), np.stack([b, b]), np.stack([c, c]), algorithm=3)
    assert ei.value.code == capi.ERR_ARG
    with pytest.raises(capi.B200LPError) as ei:
        s.Engine(2, 4, algorithm=1, devices=[0, 0])
    assert ei.value.code == capi.ERR_ARG


def test_dual_without_gpu_fails_loudly(engine_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import simplex_method_gpu_b200 as s
    from simplex_method_gpu_b200 import capi
    A, b, c = _lp()
    for call in (lambda: s.solve(A, b, c, algorithm=1), lambda: s.Engine(2, 4, algorithm=1),
                 lambda: s.solve_batch(np.stack([A, A]), np.stack([b, b]), np.stack([c, c]), algorithm=1)):
        with pytest.raises(capi.B200LPError) as ei:
            call()
        assert ei.value.code == capi.ERR_NO_GPU


def test_format_result_prints_the_new_statuses():
    import simplex_method_gpu_b200 as s
    base = dict(z=0.0, x_b=np.zeros(1), b_ixs=np.zeros(1, np.int32), iterations=2, pivots=1,
                trace=np.zeros((1, 2), np.int32))
    out = s.format_result(s.Solution(status=s.SolveStatus.Infeasible, **base))
    assert out == "# Iteration 1\n# Iteration 2\nProblem infeasible.\n\n"
    out = s.format_result(s.Solution(status=s.SolveStatus.NotDualFeasible, **base))
    assert out.endswith("Start not dual feasible.\n\n")
