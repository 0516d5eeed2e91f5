"""CPU tests of the free-constraint entry points (minsnap_derivative_gradient, minsnap_free_objective,
minsnap_optimize_free_constraints): argument errors come back as codes before any device work, the collision
entries refuse shapes other than D = 3, N = 10, and without a GPU the host entry point fails loudly."""
import ctypes as C

import numpy as np
import pytest

from helpers import standard_mask

K = 4
DIMS = np.array([8, 8, 8], np.int32)
ORIGIN = np.zeros(3)
LO, HI = np.zeros(3), np.full(3, 4.0)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _fake_device_pointer():
    # never dereferenced: every call below returns before it touches device memory
    return C.c_void_p(0x1000)


def _objective(lib, B=2, S=2, D=3, N=10, mask=None, objective=True, w_d=0.1):
    mask = standard_mask(K, N) if mask is None else mask
    dp = _fake_device_pointer()
    return lib.minsnap_free_objective(B, S, K, D, N, min(4, N // 2 - 1), _p(mask), dp, dp, dp, w_d, 1.0, 1.0, dp,
                                      _p(DIMS), _p(ORIGIN), 0.5, 0.0, _p(LO), _p(HI), 1, 0.1, 0.5, 0.5, 0.5, 1.0,
                                      dp if objective else None, None, None, None, None)


def _optimize(lib, B=2, D=3, N=10, w_d=0.1, n_steps=4, iterations=3, times=True, sdf=True, mask=None):
    mask = standard_mask(K, N) if mask is None else mask
    dp = _fake_device_pointer()
    return lib.minsnap_optimize_free_constraints(B, K, D, N, min(4, N // 2 - 1), _p(mask), dp, dp, dp if times else None,
                                                 1, w_d, 1.0, 1.0, dp if sdf else None, _p(DIMS), _p(ORIGIN), 0.5, 0.0,
                                                 _p(LO), _p(HI), 1, 0.1, 0.5, 0.5, 0.5, 1.0, iterations, n_steps, 0.5,
                                                 0.1, 1e-3, None, None, None)


def test_driver_rejects_bad_arguments(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    for w_d in (0.0, -1.0, float("nan")):       # the step divides by w_d
        assert _optimize(lib, w_d=w_d) == capi.ERR_ARG
    assert _optimize(lib, n_steps=0) == capi.ERR_ARG
    assert _optimize(lib, iterations=-1) == capi.ERR_ARG
    assert _optimize(lib, times=False) == capi.ERR_ARG
    assert _optimize(lib, sdf=False) == capi.ERR_ARG
    dp = _fake_device_pointer()
    assert lib.minsnap_optimize_free_constraints(2, K, 3, 10, 4, None, dp, dp, dp, 0, 0.1, 1.0, 1.0, dp, _p(DIMS),
                                                 _p(ORIGIN), 0.5, 0.0, _p(LO), _p(HI), 1, 0.1, 0.5, 0.5, 0.5, 1.0, 3, 4,
                                                 0.5, 0.1, 1e-3, None, None, None) == capi.ERR_ARG
    # an empty batch is a no-op, not an error
    assert _optimize(lib, B=0, times=False, sdf=False) == capi.OK


def test_objective_and_gradient_reject_bad_arguments(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _objective(lib, S=0) == capi.ERR_ARG
    assert _objective(lib, objective=False) == capi.ERR_ARG
    mask = standard_mask(K)
    dp = _fake_device_pointer()
    ws = lib.minsnap_solve_workspace_bytes(10, K)
    # NULL times, NULL J_d, NULL gradient, NULL free values, NULL mask
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 4, _p(mask), dp, dp, None, None, dp, dp, None, dp, ws,
                                           None) == capi.ERR_ARG
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 4, _p(mask), dp, dp, dp, None, None, dp, None, dp, ws,
                                           None) == capi.ERR_ARG
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 4, _p(mask), dp, dp, dp, None, dp, None, None, dp, ws,
                                           None) == capi.ERR_ARG
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 4, _p(mask), dp, None, dp, None, dp, dp, None, dp, ws,
                                           None) == capi.ERR_ARG
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 4, None, dp, dp, dp, None, dp, dp, None, dp, ws,
                                           None) == capi.ERR_ARG
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 5, _p(mask), dp, dp, dp, None, dp, dp, None, dp, ws,
                                           None) == capi.ERR_ARG                       # derivative > N/2 - 1
    assert lib.minsnap_derivative_gradient(2, K, 3, 10, 4, _p(mask), dp, dp, dp, None, dp, dp, None, dp, ws - 1,
                                           None) == capi.ERR_WORKSPACE
    assert lib.minsnap_derivative_gradient_host(2, K, 3, 10, 4, _p(mask), None, None, None, None, None, None,
                                                None) == capi.ERR_ARG


@pytest.mark.parametrize("D,N", [(2, 10), (1, 10), (3, 8), (3, 12)])
def test_collision_entries_need_three_dimensions_and_degree_nine(ms, D, N):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _objective(lib, D=D, N=N) == capi.ERR_UNSUPPORTED
    assert _optimize(lib, D=D, N=N) == capi.ERR_UNSUPPORTED


def test_derivative_gradient_host_fails_loudly_without_gpu(ms):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the loud-failure path is exercised on CPU-only machines")
    mask = standard_mask(K)
    fixed = np.zeros((2, K + 9, 3))
    free = np.zeros((2, (K - 1) * 4, 3))
    with pytest.raises(ms.MinsnapError) as ei:
        ms.derivative_gradient_host(mask, fixed, free, np.ones((2, K)))
    assert ei.value.code in (2, 4)
