"""Composite method (options.cost_shift = 1) on the host side: every option combination it does not support is an
argument error returned before any device call, so these hold with or without a GPU."""
import ctypes as C
import math

import numpy as np
import pytest

# each rejected with ERR_ARG: cost_shift without the dual loop, with an option the dual loop rejects, out of range,
# and a bad shift_delta
_BAD = [dict(cost_shift=1), dict(cost_shift=1, algorithm=0),
        dict(cost_shift=1, algorithm=1, pricing_rule=1), dict(cost_shift=1, algorithm=1, ratio_mode=1),
        dict(cost_shift=1, algorithm=1, ratio_mode=2), dict(cost_shift=1, algorithm=1, mode=1),
        dict(cost_shift=1, algorithm=1, fuse_ratio=1), dict(cost_shift=2, algorithm=1), dict(cost_shift=-1, algorithm=1),
        dict(cost_shift=1, algorithm=1, shift_delta=-1e-7), dict(cost_shift=1, algorithm=1, shift_delta=math.nan),
        dict(algorithm=1, shift_delta=-1.0)]


def _vp(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


def _lp(m=2, n=4, dt=np.float64):
    """max x1 + x2 with x1 + x2 >= 1 written as -x1 - x2 <= -1 (both rows), bounded by nothing: mixed signs"""
    A = np.zeros((m, n), dt, order="F")
    A[:, n - m:] = np.eye(m)
    A[:, :n - m] = -1
    return A, -np.ones(m, dt), np.ones(n, dt)


def test_options_mirror_the_header(engine_lib):
    from simplex_method_gpu_b200 import capi
    assert C.sizeof(capi.Options) == engine_lib.b200lp_sizeof_options()
    o = capi.default_options()
    assert (o.cost_shift, o.shift_delta, o.algorithm) == (0, 0.0, 0)
    # the int fills the padding after algorithm, the double follows it
    assert capi.Options.cost_shift.offset == capi.Options.algorithm.offset + 4
    assert capi.Options.shift_delta.offset == capi.Options.cost_shift.offset + 4
    assert C.sizeof(capi.Options) == capi.Options.shift_delta.offset + 8


@pytest.mark.parametrize("bad", _BAD, ids=lambda d: ",".join(f"{k}={v}" for k, v in d.items()))
def test_rejected_before_any_device_call(engine_lib, bad):
    from simplex_method_gpu_b200 import capi
    L = engine_lib
    A, b, c = _lp()
    o = capi.default_options(max_iter=10, **bad)
    h = C.c_void_p()
    assert L.b200lp_create(capi.F64, 2, 4, C.byref(o), C.byref(h)) == capi.ERR_ARG
    assert not h
    err = L.b200lp_last_error()
    assert b"cost_shift" in err or b"shift_delta" in err or b"dual" in err
    x_b, bix, res = np.zeros(2), np.zeros(2, np.int32), capi.Result()
    assert L.b200lp_solve_f64(_vp(A), _vp(b), _vp(c), 2, 4, C.byref(o), _vp(x_b), _vp(bix), None, 0, C.byref(res)) == capi.ERR_ARG
    A3 = np.ascontiguousarray(np.stack([A, A]).transpose(0, 2, 1))
    b3, c3 = np.stack([b, b]), np.stack([c, c])
    xb3, bix3, res3 = np.zeros((2, 2)), np.zeros((2, 2), np.int32), (capi.Result * 2)()
    assert L.b200lp_solve_batch_f64(_vp(A3), _vp(b3), _vp(c3), 2, 2, 4, C.byref(o), _vp(xb3), _vp(bix3), None, None, 0,
                                    res3) == capi.ERR_ARG


@pytest.mark.parametrize("ndev", [2, 4])
def test_composite_on_several_gpus_rejected(engine_lib, ndev):
    from simplex_method_gpu_b200 import capi
    L = engine_lib
    A, b, c = _lp()
    o = capi.default_options(max_iter=10, algorithm=1, cost_shift=1)
    devs = (C.c_int32 * ndev)(*([0] * ndev))
    h = C.c_void_p()
    assert L.b200lp_create_multi(capi.F64, 2, 4, devs, ndev, C.byref(o), C.byref(h)) == capi.ERR_ARG
    assert L.b200lp_create_sharded(capi.F64, 2, 4, 0, ndev, C.byref(o), C.byref(h)) == capi.ERR_ARG
    x_b, bix, res = np.zeros(2), np.zeros(2, np.int32), capi.Result()
    assert L.b200lp_solve_f64_multi(_vp(A), _vp(b), _vp(c), 2, 4, C.byref(o), devs, ndev, _vp(x_b), _vp(bix), None, 0,
                                    C.byref(res)) == capi.ERR_ARG


def test_python_front_ends_pass_cost_shift_through(engine_lib):
    import simplex_method_gpu_b200 as s
    from simplex_method_gpu_b200 import capi
    A, b, c = _lp()
    for call in (lambda: s.solve(A, b, c, cost_shift=1),
                 lambda: s.solve_batch(np.stack([A, A]), np.stack([b, b]), np.stack([c, c]), cost_shift=1),
                 lambda: s.Engine(2, 4, algorithm=1, cost_shift=1, shift_delta=-2.0),
                 lambda: s.Engine(2, 4, algorithm=1, cost_shift=1, devices=[0, 0])):
        with pytest.raises(capi.B200LPError) as ei:
            call()
        assert ei.value.code == capi.ERR_ARG


def test_phase_info_needs_an_engine(engine_lib):
    from simplex_method_gpu_b200 import capi
    ph, k, p1 = C.c_int32(7), C.c_int64(7), C.c_int64(7)
    assert engine_lib.b200lp_phase_info(None, C.byref(ph), C.byref(k), C.byref(p1)) == capi.ERR_ARG


def test_composite_without_gpu_fails_loudly(engine_lib):
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    import simplex_method_gpu_b200 as s
    from simplex_method_gpu_b200 import capi
    A, b, c = _lp()
    for call in (lambda: s.solve(A, b, c, algorithm=1, cost_shift=1), lambda: s.Engine(2, 4, algorithm=1, cost_shift=1)):
        with pytest.raises(capi.B200LPError) as ei:
            call()
        assert ei.value.code == capi.ERR_NO_GPU
