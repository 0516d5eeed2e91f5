"""CPU tests of the soft-constraint entry points (minsnap_soft_constraint_cost, minsnap_time_objective_soft,
minsnap_optimize_segment_times_soft): argument errors come back as MINSNAP_ERR_ARG before any device work, shapes
minsnap_solve_standard does not take come back as MINSNAP_ERR_UNSUPPORTED, an empty batch is a no-op, and without a
GPU the calls fail loudly."""
import ctypes as C

import numpy as np
import pytest

K = 4
KS = np.array([1, 2], np.int32)
LIMITS = np.array([3.0, 5.0])
NAN, INF = float("nan"), float("inf")


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _fake_device_pointer():
    # never dereferenced: every call below returns before it touches device memory
    return C.c_void_p(0x1000)


def _soft(ks=KS, limits=LIMITS, n_c=None, weight=100.0, maximum_cost=1e12, flags=0):
    """The constraint arguments in ABI order; None for an array passes NULL."""
    n_c = len(KS) if n_c is None else n_c
    return (n_c, None if ks is None else _p(ks), None if limits is None else _p(limits), weight, maximum_cost, flags)


def _cost(lib, B=2, D=3, N=10, out=True, coeffs=True, **kw):
    dp = _fake_device_pointer()
    return lib.minsnap_soft_constraint_cost(B, K, D, N, dp if coeffs else None, dp, *_soft(**kw), dp if out else None,
                                            None, None, None)


def _objective(lib, B=2, S=3, D=3, N=10, derivative=None, out=True, **kw):
    dp = _fake_device_pointer()
    derivative = min(4, N // 2 - 1) if derivative is None else derivative
    return lib.minsnap_time_objective_soft(B, S, K, D, N, derivative, dp, None, dp, 0.5, *_soft(**kw),
                                           dp if out else None, None, None, None, None)


def _optimize(lib, B=2, D=3, N=10, derivative=None, iterations=3, n_steps=4, min_time=0.1, step=0.5, increment=1e-3,
              times=True, **kw):
    dp = _fake_device_pointer()
    derivative = min(4, N // 2 - 1) if derivative is None else derivative
    return lib.minsnap_optimize_segment_times_soft(B, K, D, N, derivative, dp, None, dp if times else None, iterations,
                                                   0.5, n_steps, step, min_time, increment, *_soft(**kw), None, None,
                                                   None)


def _calls():
    return (_cost, _objective, _optimize)


@pytest.mark.parametrize("call", _calls())
def test_constraint_arguments_are_checked(ms, call):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    # 1..4 constraints
    for n_c in (0, 5, -1):
        ks = np.ones(max(n_c, 1), np.int32)
        assert call(lib, ks=ks, limits=np.ones(max(n_c, 1)), n_c=n_c) == capi.ERR_ARG
    # a derivative outside 0..N-2
    for N, k in ((10, 9), (10, -1), (6, 5), (4, 3)):
        assert call(lib, N=N, ks=np.array([1, k], np.int32)) == capi.ERR_ARG
    # limit <= 0 or not finite
    for bad in (0.0, -1.0, NAN, INF):
        assert call(lib, limits=np.array([3.0, bad])) == capi.ERR_ARG
    # weight and maximum_cost positive and finite
    for bad in (0.0, -1.0, NAN, INF):
        assert call(lib, weight=bad) == capi.ERR_ARG
        assert call(lib, maximum_cost=bad) == capi.ERR_ARG
    # extrema_flags: 0 or MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS only (mode 1 has no meaning here)
    for bad in (1, 17, 32, -1):
        assert call(lib, flags=bad) == capi.ERR_ARG
    # NULL host arrays
    assert call(lib, ks=None) == capi.ERR_ARG
    assert call(lib, limits=None) == capi.ERR_ARG


def test_null_outputs_and_inputs_are_rejected(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _cost(lib, out=False) == capi.ERR_ARG
    assert _cost(lib, coeffs=False) == capi.ERR_ARG
    assert _cost(lib, D=33) == capi.ERR_ARG
    assert _objective(lib, out=False) == capi.ERR_ARG
    assert _objective(lib, S=0) == capi.ERR_ARG
    assert _optimize(lib, times=False) == capi.ERR_ARG


def test_driver_rejects_bad_arguments(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _optimize(lib, n_steps=0) == capi.ERR_ARG
    assert _optimize(lib, iterations=-1) == capi.ERR_ARG
    for bad in (0.0, -0.1, NAN):
        assert _optimize(lib, min_time=bad) == capi.ERR_ARG
        assert _optimize(lib, step=bad) == capi.ERR_ARG
        assert _optimize(lib, increment=bad) == capi.ERR_ARG


def test_empty_batch_is_a_no_op(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _cost(lib, B=0, out=False, coeffs=False) == capi.OK
    assert _objective(lib, B=0, out=False) == capi.OK
    assert _optimize(lib, B=0, times=False) == capi.OK


@pytest.mark.parametrize("D,N,derivative", [(3, 8, 3), (3, 12, 4), (3, 10, 3), (6, 10, 4)])
def test_shapes_outside_the_standard_solve_are_unsupported(ms, D, N, derivative):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _objective(lib, D=D, N=N, derivative=derivative) == capi.ERR_UNSUPPORTED
    assert _optimize(lib, D=D, N=N, derivative=derivative) == capi.ERR_UNSUPPORTED


def test_calls_fail_loudly_without_gpu(ms):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the loud-failure path is exercised on CPU-only machines")
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    for call in _calls():
        assert call(lib) in (capi.ERR_CUDA, capi.ERR_NO_DEVICE)
