"""Batched solve on the host side: argument errors before any device call, no silent CPU path, shape checks."""
import ctypes as C

import numpy as np
import pytest


def _call(L, capi, A, b, c, batch, m, n, x_b, b_ixs, res, trace=None, trace_cap=0, y=None, f32=False):
    vp = lambda a: a.ctypes.data_as(C.c_void_p) if a is not None else None
    o = capi.default_options()
    fn = L.b200lp_solve_batch_f32 if f32 else L.b200lp_solve_batch_f64
    return fn(vp(A), vp(b), vp(c), batch, m, n, C.byref(o), vp(x_b), vp(b_ixs), vp(y), vp(trace), trace_cap, res)


def _lp(batch=3, m=2, n=4, dt=np.float64):
    A = np.zeros((batch, n, m), dt)
    A[:, n - m:, :] = np.eye(m)
    return A, np.ones((batch, m), dt), np.ones((batch, n), dt), np.zeros((batch, m), dt), np.zeros((batch, m), np.int32)


@pytest.mark.parametrize("f32", [False, True])
def test_batch_argument_errors(engine_lib, f32):
    from simplex_method_gpu_b200 import capi
    L = engine_lib
    dt = np.float32 if f32 else np.float64
    A, b, c, x_b, bix = _lp(dt=dt)
    res = (capi.Result * 3)()
    assert _call(L, capi, A, b, c, 0, 2, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG          # batch <= 0
    assert _call(L, capi, A, b, c, -1, 2, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG
    assert _call(L, capi, A, b, c, 3, 0, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG          # m <= 0
    assert _call(L, capi, A, b, c, 3, 5, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG          # m > n (v4:402)
    assert _call(L, capi, None, b, c, 3, 2, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG
    assert _call(L, capi, A, None, c, 3, 2, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG
    assert _call(L, capi, A, b, None, 3, 2, 4, x_b, bix, res, f32=f32) == capi.ERR_ARG
    assert b"NULL" in L.b200lp_last_error()
    assert _call(L, capi, A, b, c, 3, 2, 4, None, bix, res, f32=f32) == capi.ERR_ARG
    assert _call(L, capi, A, b, c, 3, 2, 4, x_b, None, res, f32=f32) == capi.ERR_ARG
    assert _call(L, capi, A, b, c, 3, 2, 4, x_b, bix, None, f32=f32) == capi.ERR_ARG
    tr = np.zeros((3, 1, 2), np.int32)
    assert _call(L, capi, A, b, c, 3, 2, 4, x_b, bix, res, trace=tr, trace_cap=-1, f32=f32) == capi.ERR_ARG
    assert b"trace_cap" in L.b200lp_last_error()


def test_batch_without_gpu_fails_loudly(engine_lib):
    """No device: the batched call refuses like the single one (there is no CPU fallback)."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from simplex_method_gpu_b200 import capi
    A, b, c, x_b, bix = _lp()
    res = (capi.Result * 3)()
    tr = np.zeros((3, 2, 2), np.int32)
    assert _call(engine_lib, capi, A, b, c, 3, 2, 4, x_b, bix, res) == capi.ERR_NO_GPU
    assert _call(engine_lib, capi, A, b, c, 3, 2, 4, x_b, bix, res, trace=tr, trace_cap=0) == capi.ERR_NO_GPU
    import simplex_method_gpu_b200 as s
    with pytest.raises(capi.B200LPError) as ei:
        s.solve_batch(np.ones((3, 2, 4)), np.ones((3, 2)), np.ones((3, 4)))
    assert ei.value.code == capi.ERR_NO_GPU


def test_solve_batch_shape_validation(engine_lib):
    import simplex_method_gpu_b200 as s
    with pytest.raises(ValueError, match="stack of matrices"):
        s.solve_batch(np.ones((2, 4)), np.ones(2), np.ones(4))
    with pytest.raises(ValueError, match="shape mismatch"):
        s.solve_batch(np.ones((3, 2, 4)), np.ones((3, 3)), np.ones((3, 4)))
    with pytest.raises(ValueError, match="shape mismatch"):
        s.solve_batch(np.ones((3, 2, 4)), np.ones((3, 2)), np.ones((2, 4)))
    with pytest.raises(ValueError, match="shape mismatch"):
        s.solve_batch(np.ones((3, 2, 4)), np.ones(6), np.ones((3, 4)))
    with pytest.raises(ValueError, match="m > n"):
        s.solve_batch(np.ones((3, 4, 2)), np.ones((3, 4)), np.ones((3, 2)))
    with pytest.raises(ValueError, match="empty"):
        s.solve_batch(np.ones((0, 2, 4)), np.ones((0, 2)), np.ones((0, 4)))
    with pytest.raises(ValueError, match="trace_cap"):
        s.solve_batch(np.ones((3, 2, 4)), np.ones((3, 2)), np.ones((3, 4)), trace_cap=-2)
    with pytest.raises(TypeError):
        s.solve_batch(np.ones((3, 2, 4), np.int64), np.ones((3, 2)), np.ones((3, 4)))
    assert "solve_batch" in s.__all__ and "BatchSolution" in s.__all__
