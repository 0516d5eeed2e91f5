"""CPU tests of the soft limits in the free-derivative problem (minsnap_soft_constraint_gradient,
minsnap_free_objective_soft, minsnap_optimize_free_constraints_soft): argument errors and unsupported shapes come back
before any device work, an empty batch is a no-op, and without a GPU the calls fail loudly.

The file also holds a long-double restatement of the closed-form gradient (`restated_gradient`), which the GPU tests
compare the kernel with.  Here it is checked against central differences of the oracle's own soft term, with the
maximum from Oracle.minmax_magnitude over Oracle.coeffs_from_constraints, so the math is checked before any GPU run.
"""
import ctypes as C
from fractions import Fraction

import numpy as np
import pytest

from helpers import compact_fixed, random_batch, standard_mask, vertex_values

K = 4
KS = np.array([1, 2], np.int32)
LIMITS = np.array([3.0, 5.0])
NAN, INF = float("nan"), float("inf")
MAP_DIMS = np.array([4, 4, 4], np.int32)
MAP_VEC = np.zeros(3)


def _p(a):
    return a.ctypes.data_as(C.c_void_p)


def _fake_device_pointer():
    # never dereferenced: every call below returns before it touches device memory
    return C.c_void_p(0x1000)


def _soft(ks=KS, limits=LIMITS, n_c=None, weight=100.0, maximum_cost=1e12, flags=0):
    n_c = len(KS) if n_c is None else n_c
    return (n_c, None if ks is None else _p(ks), None if limits is None else _p(limits), weight, maximum_cost, flags)


def _map(dt=0.1):
    return (_fake_device_pointer(), _p(MAP_DIMS), _p(MAP_VEC), 0.5, 0.0, _p(MAP_VEC), _p(MAP_VEC), 1, dt, 0.5, 0.5, 0.5,
            1.0)


def _gradient(lib, B=2, k_=K, D=3, N=10, mask=True, grad=True, coeffs=True, **kw):
    dp = _fake_device_pointer()
    m = standard_mask(k_, N)
    return lib.minsnap_soft_constraint_gradient(B, k_, D, N, _p(m) if mask else None, dp if coeffs else None, dp,
                                                *_soft(**kw), None, dp if grad else None, None, None, None, None, None)


def _objective(lib, B=2, S=3, D=3, N=10, w_sc=1.0, out=True, **kw):
    dp = _fake_device_pointer()
    m = standard_mask(K, N)
    return lib.minsnap_free_objective_soft(B, S, K, D, N, min(4, N // 2 - 1), _p(m), dp, dp, dp, 0.1, 1.0, 1.0, *_map(),
                                           *_soft(**kw), w_sc, dp if out else None, None, None, None, None, None)


def _optimize(lib, B=2, k_=K, D=3, N=10, w_sc=1.0, iterations=3, n_steps=4, w_d=0.1, times=True, **kw):
    dp = _fake_device_pointer()
    m = standard_mask(k_, N)
    return lib.minsnap_optimize_free_constraints_soft(B, k_, D, N, min(4, N // 2 - 1), _p(m), dp, dp,
                                                      dp if times else None, 1, w_d, 1.0, 1.0, *_map(), *_soft(**kw),
                                                      w_sc, iterations, n_steps, 0.5, 0.1, 1e-3, None, None, None, None)


def _calls():
    return (_gradient, _objective, _optimize)


@pytest.mark.parametrize("call", _calls())
def test_constraint_arguments_are_checked(ms, call):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    for n_c in (0, 5, -1):
        ks = np.ones(max(n_c, 1), np.int32)
        assert call(lib, ks=ks, limits=np.ones(max(n_c, 1)), n_c=n_c) == capi.ERR_ARG
    for k in (9, -1):
        assert call(lib, ks=np.array([1, k], np.int32)) == capi.ERR_ARG
    for bad in (0.0, -1.0, NAN, INF):
        assert call(lib, limits=np.array([3.0, bad])) == capi.ERR_ARG
        assert call(lib, weight=bad) == capi.ERR_ARG
        assert call(lib, maximum_cost=bad) == capi.ERR_ARG
    for bad in (1, 17, -1):
        assert call(lib, flags=bad) == capi.ERR_ARG
    assert call(lib, ks=None) == capi.ERR_ARG
    assert call(lib, limits=None) == capi.ERR_ARG


@pytest.mark.parametrize("call", [_objective, _optimize])
def test_soft_weight_is_checked(ms, call):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    for bad in (-1.0, NAN, INF, -1e-300):
        assert call(lib, w_sc=bad) == capi.ERR_ARG


def test_null_and_out_of_range_arguments_are_rejected(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _gradient(lib, mask=False) == capi.ERR_ARG
    assert _gradient(lib, grad=False) == capi.ERR_ARG       # the standard mask has free derivatives
    assert _gradient(lib, coeffs=False) == capi.ERR_ARG
    assert _gradient(lib, D=33) == capi.ERR_ARG
    assert _gradient(lib, D=0) == capi.ERR_ARG
    assert _gradient(lib, N=7) == capi.ERR_ARG
    assert _gradient(lib, B=-1) == capi.ERR_ARG
    assert _objective(lib, out=False) == capi.ERR_ARG
    assert _objective(lib, S=0) == capi.ERR_ARG
    assert _optimize(lib, times=False) == capi.ERR_ARG
    assert _optimize(lib, w_d=0.0) == capi.ERR_ARG
    assert _optimize(lib, n_steps=0) == capi.ERR_ARG
    assert _optimize(lib, iterations=-1) == capi.ERR_ARG


def test_unsupported_shapes_return_before_device_work(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    # the collision walk needs D = 3 and N = 10
    for D, N in ((2, 10), (3, 8), (3, 12)):
        assert _objective(lib, D=D, N=N) == capi.ERR_UNSUPPORTED
        assert _optimize(lib, D=D, N=N) == capi.ERR_UNSUPPORTED
    # more segments than the recovery kernel's shared memory takes, and a mask beyond the packed-parameter limit
    assert _optimize(lib, k_=2000) == capi.ERR_UNSUPPORTED
    assert _gradient(lib, k_=4000, N=10) == capi.ERR_UNSUPPORTED


def test_empty_batch_is_a_no_op(ms):
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    assert _gradient(lib, B=0, grad=False, coeffs=False) == capi.OK
    assert _objective(lib, B=0, out=False) == capi.OK
    assert _optimize(lib, B=0, times=False) == capi.OK


def test_calls_fail_loudly_without_gpu(ms):
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present; the loud-failure path is exercised on CPU-only machines")
    from mav_trajectory_generation_cmake_b200 import capi
    lib = ms.load()
    for call in _calls():
        assert call(lib) in (capi.ERR_CUDA, capi.ERR_NO_DEVICE)


# ---- the closed-form gradient, restated in long double -------------------------------------------------------------
def _ff(k, n):
    r = 1
    for q in range(k):
        r *= n - q
    return r if n >= k else 0


def unit_a1inv(N):
    """A(1)^-1 exactly (Fractions), as long double: row r of A is derivative k_r = r mod N/2 at t = 0 (r < N/2) or
    t = 1 of the monomials t^n."""
    h = N // 2
    A = [[Fraction(_ff(r % h, n) if r >= h else (_ff(r, n) if n == r else 0)) for n in range(N)] for r in range(N)]
    inv = [[Fraction(int(i == j)) for j in range(N)] for i in range(N)]
    for c in range(N):
        p = next(r for r in range(c, N) if A[r][c] != 0)
        A[c], A[p], inv[c], inv[p] = A[p], A[c], inv[p], inv[c]
        f = A[c][c]
        A[c] = [x / f for x in A[c]]
        inv[c] = [x / f for x in inv[c]]
        for r in range(N):
            if r != c and A[r][c] != 0:
                g = A[r][c]
                A[r] = [x - g * y for x, y in zip(A[r], A[c])]
                inv[r] = [x - g * y for x, y in zip(inv[r], inv[c])]
    return np.array([[float(x.numerator) / float(x.denominator) for x in row] for row in inv], np.longdouble)


def _deriv_value(c, k, t):
    """p^(k)(t) of one dimension's coefficients c (increasing powers), long double."""
    t = np.longdouble(t)
    return sum(np.longdouble(_ff(k, n)) * c[n] * t ** (n - k) for n in range(k, len(c)))


def restated_gradient(coeffs, times, col_of_row, n_fixed, n_free, constraints, weight, maximum_cost, argmax,
                      want_bound=False):
    """The gradient minsnap_soft_constraint_gradient computes, in long double.  coeffs [K][D][N], times [K];
    argmax: one (segment, time) per constraint.  Returns (soft, grad_free [n_free][D], grad_times [K]); with
    want_bound also the same sums taken over the absolute values of their terms, which bound the rounding error of a
    double evaluation (an entry that vanishes, such as a fixed vertex's, is a cancellation of terms of that size)."""
    c = np.asarray(coeffs, np.longdouble)
    T_all = np.asarray(times, np.longdouble)
    K, D, N = c.shape
    h = N // 2
    A1inv = unit_a1inv(N)
    soft = np.longdouble(0)
    gf = np.zeros((n_free, D), np.longdouble)
    gt = np.zeros(K, np.longdouble)
    bf = np.zeros((n_free, D), np.longdouble)
    bt_abs = np.zeros(K, np.longdouble)
    for (k, L), (s, t) in zip(constraints, argmax):
        T = T_all[s]
        p = np.array([_deriv_value(c[s, d], k, t) for d in range(D)])
        m = np.sqrt((p * p).sum())
        x = np.exp((m - L) / np.longdouble(L) * weight)
        soft += min(x, np.longdouble(maximum_cost))
        if not (x < maximum_cost) or m == 0:
            continue
        w = x * weight / L * p / m                                     # dtau/dm p_dim / m
        u = np.longdouble(t) / T
        for r in range(N):
            kr = r % h
            bd = sum(_ff(k, n) * u ** (n - k) * A1inv[n, r] for n in range(k, N))
            bt = sum(_ff(k, n) * u ** (n - k) * (kr - n) * A1inv[n, r] for n in range(k, N))
            ad = sum(abs(_ff(k, n) * u ** (n - k) * A1inv[n, r]) for n in range(k, N))
            at = sum(abs(_ff(k, n) * u ** (n - k) * (kr - n) * A1inv[n, r]) for n in range(k, N))
            col = col_of_row[s * N + r] - n_fixed
            if col >= 0:
                gf[col] += w * bd * T ** (kr - k)
                bf[col] += np.abs(w) * ad * T ** (kr - k)
            d_r = np.array([_deriv_value(c[s, d], kr, 0.0 if r < h else T) for d in range(D)])
            gt[s] += (w * d_r).sum() * bt * T ** (kr - k - 1)
            bt_abs[s] += np.abs(w * d_r).sum() * at * T ** (kr - k - 1)
        if s == K - 1 and t == times[s]:
            drift = w * np.array([_deriv_value(c[s, d], k + 1, T) for d in range(D)])
            gt[s] += drift.sum()
            bt_abs[s] += np.abs(drift).sum()
    if want_bound:
        return soft, gf, gt, bf, bt_abs
    return soft, gf, gt


def oracle_soft(oracle, N, K, D, col, d_all, times, constraints, weight, maximum_cost):
    """The oracle's soft term at [d_f; d_p] = d_all [D][n_all] and times, with the maxima's (segment, time)."""
    coeffs = oracle.coeffs_from_constraints(N, K, D, col, d_all, times)
    soft, where = 0.0, []
    for k, L in constraints:
        t, v, s = oracle.minmax_magnitude(coeffs, times, k, 0)["max"]
        soft += min(maximum_cost, np.exp((float(v) - L) / L * weight))
        where.append((int(s), float(t)))
    return soft, where, coeffs


def general_mask(K, N):
    h = N // 2
    m = standard_mask(K, N).copy()
    m[2, 1] = 1
    m[3, h - 1] = 1
    m[K, h - 1] = 0
    m[0, 1] = 0
    return m


@pytest.mark.parametrize("N,D,ks", [(10, 3, (1, 2)), (10, 1, (1, 3)), (6, 2, (1,)), (8, 3, (2, 3)), (12, 2, (2,))])
@pytest.mark.parametrize("mask_kind", ["standard", "general"])
def test_restated_gradient_matches_central_differences_of_the_oracle(oracle, N, D, ks, mask_kind):
    """The restatement against central differences of the oracle's soft term, d_p +/- h e_j and T +/- h with d fixed,
    within 1e-5 of the largest component, where each maximum is an isolated interior root."""
    Kt = 5
    mask = standard_mask(Kt, N) if mask_kind == "standard" else general_mask(Kt, N)
    col, n_fixed, n_free = oracle.reorder(N, Kt, mask)
    weight, maximum_cost = 10.0, 1e12
    checked = 0
    for seed in range(80):
        pos, times = random_batch(oracle, 1, Kt, D=D, seed=900 + seed)
        times = np.asarray(times[0], np.float64)
        fixed = compact_fixed(mask, vertex_values(pos[0], N)).T                        # [D][n_fixed]
        rng = np.random.default_rng(seed)
        free = rng.normal(size=(D, n_free)) * 0.5
        d_all = np.concatenate([fixed, free], axis=1)
        # limits below the maxima: the terms are live and not saturated
        _, where, coeffs = oracle_soft(oracle, N, Kt, D, col, d_all, times, [(k, 1.0) for k in ks], weight, maximum_cost)
        peaks = [float(oracle.minmax_magnitude(coeffs, times, k, 0)["max"][1]) for k in ks]
        constraints = [(k, 0.95 * v) for k, v in zip(ks, peaks)]
        if any(t <= 1e-3 * times[s] or t >= (1 - 1e-3) * times[s] for s, t in where):
            continue                                                                    # not an interior root
        soft, gf, gt = restated_gradient(coeffs, times, col, n_fixed, n_free, constraints, weight, maximum_cost, where)
        f = lambda da, tt: oracle_soft(oracle, N, Kt, D, col, da, tt, constraints, weight, maximum_cost)
        s0, w0, _ = f(d_all, times)
        assert abs(s0 - float(soft)) <= 1e-9 * abs(s0)
        fd_free = np.zeros((n_free, D))
        for j in range(n_free):
            for d in range(D):
                hstep = 1e-5 * max(1.0, abs(free[d, j]))
                dp, dm = d_all.copy(), d_all.copy()
                dp[d, n_fixed + j] += hstep
                dm[d, n_fixed + j] -= hstep
                sp, wp, _ = f(dp, times)
                sm, wm, _ = f(dm, times)
                assert [s for s, _ in wp] == [s for s, _ in w0] == [s for s, _ in wm]
                fd_free[j, d] = (sp - sm) / (2 * hstep)
        fd_t = np.zeros(Kt)
        for s in range(Kt):
            hstep = 1e-6 * times[s]
            tp, tm = times.copy(), times.copy()
            tp[s] += hstep
            tm[s] -= hstep
            fd_t[s] = (f(d_all, tp)[0] - f(d_all, tm)[0]) / (2 * hstep)
        scale_f = max(np.abs(fd_free).max(), 1e-300)
        scale_t = max(np.abs(fd_t).max(), 1e-300)
        assert np.abs(gf.astype(np.float64) - fd_free).max() <= 1e-5 * scale_f
        assert np.abs(gt.astype(np.float64) - fd_t).max() <= 1e-5 * scale_t
        checked += 1
        if checked == 2:
            break
    assert checked >= 1
