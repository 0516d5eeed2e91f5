"""Python plumbing over the C ABI: torch tensors for device memory and streams, numpy arrays
for the host-buffer entry points.  Every function is a thin argument marshaller around one
C-ABI call -- there is no arithmetic and no fallback here.  The exceptions are the torch-glue
versions kept as the tests' checkers (time_objective_with_soft_constraints and the *_reference_glue
drivers), which chain several C-ABI calls on the device and glue them with elementwise torch
operations (step ladders, exp / clamp of the soft-constraint terms), and the cost_time term that
time_objective_soft reports with want_terms.

Layouts are those of include/minsnap_b200.h (h = N/2):
  fixed_values [B][n_fixed][D], free_values [B][n_free][D], positions [B][K+1][D],
  times [B][K], coeffs [B][K][D][N], samples [B][M][n_deriv][D].
"""
import ctypes as C

import numpy as np

from . import capi

SNAP = 4


def _lib():
    return capi.load()


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def _torch():
    import torch
    return torch


def _dptr(t, dtype=None):
    if t is None:
        return None
    torch = _torch()
    assert t.is_cuda and t.is_contiguous(), "expected a contiguous CUDA tensor"
    if dtype is not None:
        assert t.dtype == dtype, "expected dtype %s, got %s" % (dtype, t.dtype)
    return C.c_void_p(t.data_ptr())


def _stream():
    torch = _torch()
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


def _hptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _np(a, dtype):
    return None if a is None else np.ascontiguousarray(a, dtype=dtype)


def standard_mask(K, N=10, max_fixed_derivative=None):
    """Mask of createRandomVertices (ref src/vertex.cpp:59,71-76)."""
    h = N // 2
    if max_fixed_derivative is None:
        max_fixed_derivative = h - 1
    m = np.zeros((K + 1, h), np.uint8)
    m[:, 0] = 1
    m[0, : max_fixed_derivative + 1] = 1
    m[K, : max_fixed_derivative + 1] = 1
    return m


def mask_counts(mask):
    mask = np.asarray(mask)
    n_fixed = int((mask != 0).sum())
    return n_fixed, mask.size - n_fixed


def device_info():
    dev, sms, maj, mnr = C.c_int(), C.c_int(), C.c_int(), C.c_int()
    mem = C.c_size_t()
    capi.check(_lib().minsnap_device_info(C.byref(dev), C.byref(sms), C.byref(maj), C.byref(mnr), C.byref(mem)),
               "minsnap_device_info")
    return dict(device=dev.value, sm_count=sms.value, cc=(maj.value, mnr.value), global_mem_bytes=mem.value)


def fp64_peak(repeats=5):
    out = C.c_double()
    capi.check(_lib().minsnap_fp64_peak(repeats, C.byref(out)), "minsnap_fp64_peak")
    return out.value


# ------------------------------------------------------------------------------------------
# device-pointer entry points (torch CUDA tensors, current stream, asynchronous)
# ------------------------------------------------------------------------------------------
def reorder(mask_dev, N, K):
    """mask_dev uint8 [n_masks][(K+1)*h] on the GPU -> (col_of_row int32 [n_masks][N*K], counts int32 [n_masks][2])."""
    torch = _torch()
    n_masks = mask_dev.shape[0]
    col = torch.empty((n_masks, N * K), dtype=torch.int32, device=mask_dev.device)
    counts = torch.empty((n_masks, 2), dtype=torch.int32, device=mask_dev.device)
    capi.check(_lib().minsnap_reorder(N, K, n_masks, _dptr(mask_dev, torch.uint8), _dptr(col), _dptr(counts), _stream()),
               "minsnap_reorder")
    return col, counts


def estimate_segment_times(positions, v_max, a_max, magic=6.5):
    torch = _torch()
    B, K1, D = positions.shape
    times = torch.empty((B, K1 - 1), dtype=torch.float64, device=positions.device)
    capi.check(_lib().minsnap_estimate_segment_times(B, K1 - 1, D, _dptr(positions, torch.float64), v_max, a_max, magic,
                                                     _dptr(times), _stream()), "minsnap_estimate_segment_times")
    return times


def segment_matrices(T, N=10, derivative=SNAP):
    """T float64 [n] on the GPU -> dict(A, Ainv, Q, H), each [n][N][N]."""
    torch = _torch()
    n = T.shape[0]
    out = {k: torch.empty((n, N, N), dtype=torch.float64, device=T.device) for k in ("A", "Ainv", "Q", "H")}
    capi.check(_lib().minsnap_segment_matrices(n, N, derivative, _dptr(T, torch.float64), _dptr(out["A"]),
                                               _dptr(out["Ainv"]), _dptr(out["Q"]), _dptr(out["H"]), _stream()),
               "minsnap_segment_matrices")
    return out


def solve(mask, fixed_values, times, N=10, derivative=SNAP, want_cost=True):
    """General batched setupFromVertices + solveLinear.  mask: host uint8 [(K+1)][h]."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, n_fixed, D = fixed_values.shape
    nf, n_free = mask_counts(mask)
    assert nf == n_fixed and times.shape == (B, K)
    dev = times.device
    coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev)
    free = torch.empty((B, n_free, D), dtype=torch.float64, device=dev)
    cost = torch.empty((B,), dtype=torch.float64, device=dev) if want_cost else None
    status = torch.empty((B,), dtype=torch.int32, device=dev)
    col = torch.empty((N * K,), dtype=torch.int32, device=dev)
    ws_bytes = _lib().minsnap_solve_workspace_bytes(N, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    capi.check(_lib().minsnap_solve(B, K, D, N, derivative, _hptr(mask), _dptr(fixed_values, torch.float64),
                                    _dptr(times, torch.float64), _dptr(coeffs), _dptr(free), _dptr(cost), _dptr(status),
                                    _dptr(col), _dptr(ws), ws_bytes, _stream()), "minsnap_solve")
    return dict(coeffs=coeffs, free_values=free, cost=cost, status=status, col_of_row=col)


def coeffs_from_constraints(mask, fixed_values, free_values, times, N=10):
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, _, D = fixed_values.shape
    coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=times.device)
    ws_bytes = _lib().minsnap_solve_workspace_bytes(N, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=times.device)
    capi.check(_lib().minsnap_coeffs_from_constraints(B, K, D, N, _hptr(mask), _dptr(fixed_values), _dptr(free_values),
                                                      _dptr(times), _dptr(coeffs), _dptr(ws), ws_bytes, _stream()),
               "minsnap_coeffs_from_constraints")
    return coeffs


def cost(coeffs, times, derivative=SNAP):
    torch = _torch()
    B, K, D, N = coeffs.shape
    out = torch.empty((B,), dtype=torch.float64, device=coeffs.device)
    capi.check(_lib().minsnap_cost(B, K, D, N, derivative, _dptr(coeffs, torch.float64), _dptr(times, torch.float64),
                                   _dptr(out), _stream()), "minsnap_cost")
    return out


def solve_standard(positions, times=None, end_derivatives=None, v_max=0.0, a_max=0.0, magic=6.5, N=10,
                   derivative=SNAP, coeffs=None, want_free=False, want_cost=False, want_status=True,
                   want_times=False):
    """Standard-mask batched solve.  times=None => estimated on the device from (v_max, a_max, magic)."""
    torch = _torch()
    B, K1, D = positions.shape
    K = K1 - 1
    h = N // 2
    dev = positions.device
    if coeffs is None:
        coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev)
    free = torch.empty((B, (K - 1) * (h - 1), D), dtype=torch.float64, device=dev) if want_free else None
    cost_t = torch.empty((B,), dtype=torch.float64, device=dev) if want_cost else None
    status = torch.empty((B,), dtype=torch.int32, device=dev) if want_status else None
    times_out = torch.empty((B, K), dtype=torch.float64, device=dev) if (want_times and times is None) else None
    capi.check(_lib().minsnap_solve_standard(B, K, D, N, derivative, _dptr(positions, torch.float64),
                                             _dptr(end_derivatives), _dptr(times), v_max, a_max, magic,
                                             _dptr(times_out), _dptr(coeffs), _dptr(free), _dptr(cost_t), _dptr(status),
                                             _stream()), "minsnap_solve_standard")
    return dict(coeffs=coeffs, free_values=free, cost=cost_t, status=status,
                times=times if times is not None else times_out)


def sample_uniform(coeffs, times, M, n_deriv=5, out=None, want_times=False):
    torch = _torch()
    B, K, D, N = coeffs.shape
    if out is None:
        out = torch.empty((B, M, n_deriv, D), dtype=torch.float64, device=coeffs.device)
    t_out = torch.empty((B, M), dtype=torch.float64, device=coeffs.device) if want_times else None
    capi.check(_lib().minsnap_sample_uniform(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64), M,
                                             n_deriv, _dptr(out), _dptr(t_out), _stream()), "minsnap_sample_uniform")
    return (out, t_out) if want_times else out


def sample_at(coeffs, times, t, n_deriv=5, want_segment=False):
    """t: [B][M] per-trajectory instants or [M] shared by the whole batch."""
    torch = _torch()
    B, K, D, N = coeffs.shape
    M = t.shape[-1]
    stride = 0 if t.dim() == 1 else M
    out = torch.empty((B, M, n_deriv, D), dtype=torch.float64, device=coeffs.device)
    seg = torch.empty((B, M), dtype=torch.int32, device=coeffs.device) if want_segment else None
    capi.check(_lib().minsnap_sample_at(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64), M,
                                        _dptr(t, torch.float64), stride, n_deriv, _dptr(out), _dptr(seg), _stream()),
               "minsnap_sample_at")
    return (out, seg) if want_segment else out


def evaluate_range(coeffs, times, t_start, t_end, dt, derivative, max_samples):
    torch = _torch()
    B, K, D, N = coeffs.shape
    out = torch.zeros((B, max_samples, D), dtype=torch.float64, device=coeffs.device)
    t_out = torch.zeros((B, max_samples), dtype=torch.float64, device=coeffs.device)
    count = torch.zeros((B,), dtype=torch.int32, device=coeffs.device)
    capi.check(_lib().minsnap_evaluate_range(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64),
                                             t_start, t_end, dt, derivative, max_samples, _dptr(out), _dptr(t_out),
                                             _dptr(count), _stream()), "minsnap_evaluate_range")
    return out, t_out, count


def cost_sweep(positions, times, end_derivatives=None, N=10, derivative=SNAP, want_status=False):
    """positions [B][K+1][D], times [B][S][K] -> cost [B][S]."""
    torch = _torch()
    B, K1, D = positions.shape
    S = times.shape[1]
    out = torch.empty((B, S), dtype=torch.float64, device=positions.device)
    status = torch.empty((B, S), dtype=torch.int32, device=positions.device) if want_status else None
    capi.check(_lib().minsnap_cost_sweep(B, S, K1 - 1, D, N, derivative, _dptr(positions, torch.float64),
                                         _dptr(end_derivatives), _dptr(times, torch.float64), _dptr(out), _dptr(status),
                                         _stream()), "minsnap_cost_sweep")
    return (out, status) if want_status else out


def time_objective(positions, times, time_penalty, end_derivatives=None, N=10, derivative=SNAP, want_cost=False):
    """positions [B][K+1][D], times [B][S][K] -> objective [B][S] = computeCost + time_penalty * total_time^2
    (ref objectiveFunctionTime, NL.i:765-832, derivative and time terms)."""
    torch = _torch()
    B, K1, D = positions.shape
    S = times.shape[1]
    out = torch.empty((B, S), dtype=torch.float64, device=positions.device)
    cost_t = torch.empty((B, S), dtype=torch.float64, device=positions.device) if want_cost else None
    capi.check(_lib().minsnap_time_objective(B, S, K1 - 1, D, N, derivative, _dptr(positions, torch.float64),
                                             _dptr(end_derivatives), _dptr(times, torch.float64), float(time_penalty),
                                             _dptr(out), _dptr(cost_t), None, _stream()), "minsnap_time_objective")
    return (out, cost_t) if want_cost else out


def time_objective_with_soft_constraints(positions, times, time_penalty, constraints, soft_constraint_weight=100.0,
                                         maximum_cost=1.0e12, end_derivatives=None, N=10, derivative=SNAP,
                                         want_terms=False):
    """The reference's time-only objective with its soft limits on the magnitude of derivatives
    (objectiveFunctionTime with use_soft_constraints, NL.i:765-832; evaluateMaximumMagnitudeAsSoftConstraint,
    NL.i:2396-2426; evaluateMaximumMagnitudeConstraint, NL.i:2346-2392):

        objective = computeCost + time_penalty * total_time^2
                    + sum over constraints min(maximum_cost, exp((max |p^(k)| - limit) / limit * weight))

    constraints: iterable of (derivative k, limit), e.g. [(1, v_max), (2, a_max)].  positions [B][K+1][D],
    times [B][S][K] -> objective [B][S].  Composition of three C-ABI calls per constraint set: one solve of the
    B * S allocations with coefficients, one minsnap_extrema per constraint (computeMaximumOfMagnitude
    semantics), one fused epilogue on the device."""
    torch = _torch()
    B, K1, D = positions.shape
    K = K1 - 1
    S = times.shape[1]
    flat_t = times.reshape(B * S, K).contiguous()
    rep_p = positions.repeat_interleave(S, dim=0).contiguous()
    rep_e = None if end_derivatives is None else end_derivatives.repeat_interleave(S, dim=0).contiguous()
    sol = solve_standard(rep_p, flat_t, end_derivatives=rep_e, N=N, derivative=derivative, want_cost=True,
                         want_status=False)
    total = flat_t.sum(1)
    cost_time = total * total * time_penalty
    terms = []
    for k, limit in constraints:
        peak = extrema(sol["coeffs"], flat_t, int(k), mode=EXTREMA_OPTIMIZATION)["max_value"]
        terms.append(torch.exp((peak - limit) / limit * soft_constraint_weight).clamp_max(maximum_cost))
    obj = sol["cost"] + cost_time
    for t in terms:
        obj = obj + t
    obj = obj.reshape(B, S)
    if want_terms:
        return obj, dict(cost_trajectory=sol["cost"].reshape(B, S), cost_time=cost_time.reshape(B, S),
                         cost_constraints=[t.reshape(B, S) for t in terms])
    return obj


def time_gradient(coeffs, times, increment=0.1, w_d=0.1, w_t=1.0, derivative=SNAP, want_segment_cost=False):
    """Numeric gradient of w_d J_d + w_t total_time in the segment times (ref getCostAndGradientTime,
    NL.i:2155-2243; defaults are the reference's increment_time and cost weights).  coeffs [B][K][D][N]
    are the solved coefficients -> gradient [B][K] (and the per-segment terms of J_d = 2 computeCost)."""
    torch = _torch()
    B, K, D, N = coeffs.shape
    grad = torch.empty((B, K), dtype=torch.float64, device=coeffs.device)
    seg = torch.empty((B, K), dtype=torch.float64, device=coeffs.device) if want_segment_cost else None
    capi.check(_lib().minsnap_time_gradient(B, K, D, N, derivative, _dptr(coeffs, torch.float64),
                                            _dptr(times, torch.float64), float(increment), float(w_d), float(w_t),
                                            _dptr(grad), _dptr(seg), _stream()), "minsnap_time_gradient")
    return (grad, seg) if want_segment_cost else grad


def optimize_segment_times(positions, times, iterations=20, time_penalty=500.0, n_steps=16, max_relative_step=0.5,
                           min_time=0.1, end_derivatives=None, gradient_increment=1e-3, N=10, derivative=SNAP):
    """Additive batched driver for the time-only problem (SURVEY 8(f)2): every trajectory of the batch
    descends objective = computeCost + time_penalty * total_time^2 along its own numeric gradient, the line
    search is one cost sweep over n_steps step lengths per trajectory.  One C-ABI call
    (minsnap_optimize_segment_times): the whole loop is enqueued on the current stream, five launches per
    iteration, nothing returns to the host.  The reference runs one NLopt instance per trajectory on the host.
    Returns (times, objective history [iterations + 1][B])."""
    torch = _torch()
    B, K1, D = positions.shape
    times = times.clone().contiguous()
    history = torch.empty((iterations + 1, B), dtype=torch.float64, device=positions.device)
    capi.check(_lib().minsnap_optimize_segment_times(B, K1 - 1, D, N, derivative, _dptr(positions, torch.float64),
                                                     _dptr(end_derivatives), _dptr(times, torch.float64), int(iterations),
                                                     float(time_penalty), int(n_steps), float(max_relative_step),
                                                     float(min_time), float(gradient_increment), _dptr(history), _stream()),
               "minsnap_optimize_segment_times")
    return times, history


def optimize_segment_times_reference_glue(positions, times, iterations=20, time_penalty=500.0, n_steps=16,
                                          max_relative_step=0.5, min_time=0.1, end_derivatives=None):
    """The same descent with its glue written in elementwise torch operations around three C-ABI calls per
    iteration (round 1's driver): kept as the checker of minsnap_optimize_segment_times in the tests."""
    torch = _torch()
    B, K1, D = positions.shape
    times = times.clone()
    history = [time_objective(positions, times[:, None, :].contiguous(), time_penalty, end_derivatives)[:, 0]]
    ladder = max_relative_step * 0.5 ** torch.arange(n_steps, dtype=torch.float64, device=positions.device)
    for _ in range(iterations):
        coeffs = solve_standard(positions, times, end_derivatives=end_derivatives, want_status=False)["coeffs"]
        g = time_gradient(coeffs, times, increment=1e-3, w_d=0.5, w_t=0.0)
        g = g + 2.0 * time_penalty * times.sum(1, keepdim=True)
        scale = (times / g.abs().clamp_min(1e-300)).min(1, keepdim=True).values
        cand = times[:, None, :] - (ladder[None, :, None] * scale[:, :, None]) * g[:, None, :]
        cand = cand.clamp_min(min_time).contiguous()
        obj = time_objective(positions, cand, time_penalty, end_derivatives)
        best, arg = obj.min(1)
        improved = best < history[-1]
        chosen = cand[torch.arange(B, device=cand.device), arg]
        times = torch.where(improved[:, None], chosen, times)
        history.append(torch.where(improved, best, history[-1]))
    return times, torch.stack(history)


# ---- the time-only objective with the reference's soft limits on max |p^(k)| ------------------------------------
def _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small):
    """The constraint arguments of the soft-constraint entries, in their order, and the host arrays they point into
    (which must outlive the call)."""
    ks = np.asarray([int(k) for k, _ in constraints], np.int32)
    limits = np.asarray([float(v) for _, v in constraints], np.float64)
    args = (len(ks), _hptr(ks), _hptr(limits), float(soft_constraint_weight), float(maximum_cost),
            EXTREMA_KEEP_SMALL_COEFFICIENTS if keep_small else 0)
    return (ks, limits), args


def soft_constraint_cost(coeffs, times, constraints, soft_constraint_weight=100.0, maximum_cost=1.0e12,
                         keep_small=False, want_terms=False):
    """Soft cost of solved trajectories (ref evaluateMaximumMagnitudeAsSoftConstraint, NL.i:2396-2426):
    sum over constraints (k, limit) of min(maximum_cost, exp((max |p^(k)| - limit) / limit * weight)), the maximum
    that of extrema(..., mode=EXTREMA_OPTIMIZATION) bit for bit.  coeffs [B][K][D][N], times [B][K] -> cost [B]
    (with want_terms also dict(terms, max_value), each [B][n_constraints]).  One C-ABI call
    (minsnap_soft_constraint_cost)."""
    torch = _torch()
    B, K, D, N = coeffs.shape
    n_c = len(constraints)
    dev = coeffs.device
    cost_t = torch.empty((B,), dtype=torch.float64, device=dev)
    terms = torch.empty((B, n_c), dtype=torch.float64, device=dev) if want_terms else None
    peak = torch.empty((B, n_c), dtype=torch.float64, device=dev) if want_terms else None
    host, sargs = _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small)
    capi.check(_lib().minsnap_soft_constraint_cost(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64),
                                                   *sargs, _dptr(cost_t), _dptr(terms), _dptr(peak), _stream()),
               "minsnap_soft_constraint_cost")
    return (cost_t, dict(terms=terms, max_value=peak)) if want_terms else cost_t


def time_objective_soft(positions, times, time_penalty, constraints, soft_constraint_weight=100.0, maximum_cost=1.0e12,
                        end_derivatives=None, keep_small=False, N=10, derivative=SNAP, want_terms=False):
    """The objective of time_objective_with_soft_constraints in one C-ABI call (minsnap_time_objective_soft):
    computeCost + time_penalty * total_time^2 + soft cost, NaN where the solve fails.  positions [B][K+1][D], times
    [B][S][K] -> objective [B][S]; with want_terms also dict(cost_trajectory, cost_time, cost_constraints) as
    time_objective_with_soft_constraints gives them (cost_constraints: one [B][S] tensor per constraint)."""
    torch = _torch()
    B, K1, D = positions.shape
    S = times.shape[1]
    n_c = len(constraints)
    dev = positions.device
    obj = torch.empty((B, S), dtype=torch.float64, device=dev)
    cost_t = torch.empty((B, S), dtype=torch.float64, device=dev) if want_terms else None
    terms = torch.empty((B, S, n_c), dtype=torch.float64, device=dev) if want_terms else None
    host, sargs = _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small)
    capi.check(_lib().minsnap_time_objective_soft(B, S, K1 - 1, D, N, derivative, _dptr(positions, torch.float64),
                                                  _dptr(end_derivatives), _dptr(times, torch.float64), float(time_penalty),
                                                  *sargs, _dptr(obj), _dptr(cost_t), None, _dptr(terms), _stream()),
               "minsnap_time_objective_soft")
    if not want_terms:
        return obj
    total = times[..., 0]
    for k in range(1, K1 - 1):       # left to right, as the objective sums it
        total = total + times[..., k]
    return obj, dict(cost_trajectory=cost_t, cost_time=total * total * time_penalty,
                     cost_constraints=[terms[..., j] for j in range(n_c)])


def optimize_segment_times_soft(positions, times, constraints, iterations=20, time_penalty=500.0, n_steps=16,
                                max_relative_step=0.5, min_time=0.1, end_derivatives=None, gradient_increment=1e-3,
                                soft_constraint_weight=100.0, maximum_cost=1.0e12, keep_small=False, N=10,
                                derivative=SNAP):
    """optimize_segment_times on the objective of time_objective_soft: the gradient adds the central difference of
    the soft cost over re-solved allocations T -/+ gradient_increment e_n.  One C-ABI call
    (minsnap_optimize_segment_times_soft): the whole loop is enqueued on the current stream.  Returns (times,
    objective history [iterations + 1][B], max_value [B][n_constraints] at the returned times)."""
    torch = _torch()
    B, K1, D = positions.shape
    times = times.clone().contiguous()
    history = torch.empty((iterations + 1, B), dtype=torch.float64, device=positions.device)
    peak = torch.empty((B, len(constraints)), dtype=torch.float64, device=positions.device)
    host, sargs = _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small)
    capi.check(_lib().minsnap_optimize_segment_times_soft(B, K1 - 1, D, N, derivative, _dptr(positions, torch.float64),
                                                          _dptr(end_derivatives), _dptr(times, torch.float64),
                                                          int(iterations), float(time_penalty), int(n_steps),
                                                          float(max_relative_step), float(min_time),
                                                          float(gradient_increment), *sargs, _dptr(history), _dptr(peak),
                                                          _stream()), "minsnap_optimize_segment_times_soft")
    return times, history, peak


def optimize_segment_times_soft_reference_glue(positions, times, constraints, iterations=20, time_penalty=500.0,
                                               n_steps=16, max_relative_step=0.5, min_time=0.1, end_derivatives=None,
                                               gradient_increment=1e-3, soft_constraint_weight=100.0,
                                               maximum_cost=1.0e12, keep_small=False):
    """The descent of optimize_segment_times_soft with its glue written in elementwise torch operations around the
    C-ABI calls (solve_standard, time_gradient, soft_constraint_cost, time_objective_soft): kept as the checker of
    minsnap_optimize_segment_times_soft in the tests."""
    torch = _torch()
    B, K1, D = positions.shape
    K = K1 - 1
    dev = positions.device
    soft_kw = dict(soft_constraint_weight=soft_constraint_weight, maximum_cost=maximum_cost, keep_small=keep_small)

    def objective(t):
        return time_objective_soft(positions, t.contiguous(), time_penalty, constraints, end_derivatives=end_derivatives,
                                   **soft_kw)

    times = times.clone()
    history = [objective(times[:, None, :])[:, 0]]
    ladder = max_relative_step * 0.5 ** torch.arange(n_steps, dtype=torch.float64, device=dev)
    eye = torch.eye(K, dtype=torch.bool, device=dev)
    rep_p = positions.repeat_interleave(2 * K, dim=0).contiguous()
    rep_e = None if end_derivatives is None else end_derivatives.repeat_interleave(2 * K, dim=0).contiguous()
    rows = torch.arange(B, device=dev)
    h = gradient_increment
    for _ in range(iterations):
        coeffs = solve_standard(positions, times, end_derivatives=end_derivatives, want_status=False)["coeffs"]
        g = time_gradient(coeffs, times, increment=h, w_d=0.5, w_t=0.0)
        short = times <= 0.1
        t_minus = torch.where(short, torch.full_like(times, 0.1), times - h)
        t_plus = torch.where(short, torch.full_like(times, 0.1), times + h)
        base = times[:, None, :].expand(B, K, K)
        moved = torch.stack([torch.where(eye[None], t_minus[:, None, :], base),
                             torch.where(eye[None], t_plus[:, None, :], base)], 2)     # [B][n][-/+][K]
        flat = moved.reshape(B * 2 * K, K).contiguous()
        c2 = solve_standard(rep_p, flat, end_derivatives=rep_e, want_status=False)["coeffs"]
        soft = soft_constraint_cost(c2, flat, constraints, **soft_kw).reshape(B, K, 2)
        g = g + (soft[..., 1] - soft[..., 0]) / (2.0 * h)
        g = g + 2.0 * time_penalty * times.sum(1, keepdim=True)
        scale = (times / g.abs().clamp_min(1e-300)).min(1, keepdim=True).values
        cand = times[:, None, :] - (ladder[None, :, None] * scale[:, :, None]) * g[:, None, :]
        cand = cand.clamp_min(min_time).contiguous()
        obj = objective(cand)
        best, arg = torch.where(torch.isfinite(obj), obj, torch.full_like(obj, float("inf"))).min(1)
        improved = torch.isfinite(best) & (best < history[-1])
        times = torch.where(improved[:, None], cand[rows, arg], times)
        history.append(torch.where(improved, best, history[-1]))
    return times, torch.stack(history)


def collision_cost(coeffs, times, sdf, origin, resolution, min_bound, max_bound, dt=0.1, map_resolution=None,
                   epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.0, use_continuous_distance=True, oob_value=0.0,
                   want_charged=False):
    """Collision cost of solved trajectories against a dense distance grid (ref getCostAndGradientCollision,
    NL.i:1523-1709; defaults are the reference's NonlinearOptimizationParameters).  coeffs [B][K][3][10], times
    [B][K], sdf [nx][ny][nz] (distance at the cell centres) are CUDA tensors -> dict(cost [B], is_collision [B])."""
    torch = _torch()
    B, K, D, N = coeffs.shape
    if map_resolution is None:
        map_resolution = resolution
    dims = np.asarray(sdf.shape, np.int32)
    org, lo, hi = _np(origin, np.float64), _np(min_bound, np.float64), _np(max_bound, np.float64)
    cost_t = torch.empty((B,), dtype=torch.float64, device=coeffs.device)
    hit = torch.empty((B,), dtype=torch.int32, device=coeffs.device)
    charged = torch.empty((B,), dtype=torch.int32, device=coeffs.device) if want_charged else None
    capi.check(_lib().minsnap_collision_cost(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64),
                                             _dptr(sdf, torch.float64), _hptr(dims), _hptr(org), float(resolution),
                                             float(oob_value), _hptr(lo), _hptr(hi), int(bool(use_continuous_distance)),
                                             float(dt), float(map_resolution), float(epsilon), float(robot_radius),
                                             float(coll_pot_multiplier), _dptr(cost_t), _dptr(hit), _dptr(charged),
                                             _stream()), "minsnap_collision_cost")
    return dict(cost=cost_t, is_collision=hit, charged=charged)


def collision_gradient(coeffs, times, sdf, origin, resolution, min_bound, max_bound, dt=0.1, map_resolution=None,
                       epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.0, use_continuous_distance=True, oob_value=0.0,
                       col_of_row=None, n_fixed=0, n_free=None):
    """Collision cost AND its gradient w.r.t. the free derivatives (ref getCostAndGradientCollision with gradients,
    NL.i:1666-1686).  col_of_row: the int32 [N K] constraint index map on the device (minsnap_reorder) with its
    n_fixed / n_free, or None for the standard mask.  -> dict(cost [B], gradient [B][n_free][3], is_collision [B],
    charged [B])."""
    torch = _torch()
    B, K, D, N = coeffs.shape
    if map_resolution is None:
        map_resolution = resolution
    if col_of_row is None:
        n_fixed, n_free = K + N - 1, (K - 1) * (N // 2 - 1)
    dims = np.asarray(sdf.shape, np.int32)
    org, lo, hi = _np(origin, np.float64), _np(min_bound, np.float64), _np(max_bound, np.float64)
    cost_t = torch.empty((B,), dtype=torch.float64, device=coeffs.device)
    grad = torch.empty((B, n_free, 3), dtype=torch.float64, device=coeffs.device)
    hit = torch.empty((B,), dtype=torch.int32, device=coeffs.device)
    charged = torch.empty((B,), dtype=torch.int32, device=coeffs.device)
    capi.check(_lib().minsnap_collision_gradient(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64),
                                                 _dptr(sdf, torch.float64), _hptr(dims), _hptr(org), float(resolution),
                                                 float(oob_value), _hptr(lo), _hptr(hi), int(bool(use_continuous_distance)),
                                                 float(dt), float(map_resolution), float(epsilon), float(robot_radius),
                                                 float(coll_pot_multiplier),
                                                 _dptr(col_of_row, torch.int32) if col_of_row is not None else None,
                                                 int(n_fixed), int(n_free), _dptr(cost_t), _dptr(grad), _dptr(hit),
                                                 _dptr(charged), _stream()), "minsnap_collision_gradient")
    return dict(cost=cost_t, gradient=grad, is_collision=hit, charged=charged)


# ---- the free derivatives (and times) against w_d J_d + w_c J_c + w_t sum(T) ---------------------------------------
def derivative_gradient(mask, fixed_values, free_values, times, N=10, derivative=SNAP, want_coeffs=False,
                        want_diag=False):
    """J_d = d^T R d (= 2 computeCost; ref getCostAndGradientDerivative, NL.i:1452-1521) and its gradient
    2 (R_pf d_f + R_pp d_p) in the free derivatives, at the given constraints.  mask: host uint8 [(K+1)][h];
    fixed_values [B][n_fixed][D], free_values [B][n_free][D], times [B][K] (CUDA tensors) -> dict(Jd [B],
    gradient [B][n_free][D], diag [B][n_free] = diag(R_pp) or None, coeffs [B][K][D][N] or None)."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, _, D = fixed_values.shape
    _, n_free = mask_counts(mask)
    dev = times.device
    jd = torch.empty((B,), dtype=torch.float64, device=dev)
    grad = torch.empty((B, n_free, D), dtype=torch.float64, device=dev)
    diag = torch.empty((B, n_free), dtype=torch.float64, device=dev) if want_diag else None
    coeffs = torch.empty((B, K, D, N), dtype=torch.float64, device=dev) if want_coeffs else None
    ws_bytes = _lib().minsnap_solve_workspace_bytes(N, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    capi.check(_lib().minsnap_derivative_gradient(B, K, D, N, derivative, _hptr(mask), _dptr(fixed_values, torch.float64),
                                                  _dptr(free_values, torch.float64), _dptr(times, torch.float64),
                                                  _dptr(coeffs), _dptr(jd), _dptr(grad), _dptr(diag), _dptr(ws), ws_bytes,
                                                  _stream()), "minsnap_derivative_gradient")
    return dict(Jd=jd, gradient=grad, diag=diag, coeffs=coeffs)


def _collision_map(sdf, origin, resolution, min_bound, max_bound, dt, map_resolution, epsilon, robot_radius,
                   coll_pot_multiplier, use_continuous_distance, oob_value):
    """The map and walk arguments of minsnap_collision_cost, in its order, and the host arrays they point into
    (which must outlive the call)."""
    torch = _torch()
    if map_resolution is None:
        map_resolution = resolution
    host = (np.asarray(sdf.shape, np.int32), _np(origin, np.float64), _np(min_bound, np.float64),
            _np(max_bound, np.float64))
    dims, org, lo, hi = host
    args = (_dptr(sdf, torch.float64), _hptr(dims), _hptr(org), float(resolution), float(oob_value), _hptr(lo), _hptr(hi),
            int(bool(use_continuous_distance)), float(dt), float(map_resolution), float(epsilon), float(robot_radius),
            float(coll_pot_multiplier))
    return host, args


def free_objective(mask, fixed_values, free_values, times, sdf, origin, resolution, min_bound, max_bound, w_c, w_d=0.1,
                   w_t=1.0, dt=0.1, map_resolution=None, epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.0,
                   use_continuous_distance=True, oob_value=0.0, N=10, derivative=SNAP, want_terms=False):
    """J = w_d J_d + w_c J_c + w_t sum(T) for S candidates per trajectory (minsnap_free_objective).  fixed_values
    [B][n_fixed][3] is shared by the candidates of a trajectory; free_values [B][S][n_free][3], times [B][S][K] ->
    objective [B][S] (with want_terms also dict(Jd, Jc, is_collision), each [B][S]).  The map arguments are those of
    collision_cost.  w_d and w_t default to the reference's cost weights; w_c has no default."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, S = times.shape[0], times.shape[1]
    D = fixed_values.shape[2]
    dev = times.device
    obj = torch.empty((B, S), dtype=torch.float64, device=dev)
    terms = dict(Jd=torch.empty((B, S), dtype=torch.float64, device=dev),
                 Jc=torch.empty((B, S), dtype=torch.float64, device=dev),
                 is_collision=torch.empty((B, S), dtype=torch.int32, device=dev)) if want_terms else {}
    host, margs = _collision_map(sdf, origin, resolution, min_bound, max_bound, dt, map_resolution, epsilon, robot_radius,
                                 coll_pot_multiplier, use_continuous_distance, oob_value)
    capi.check(_lib().minsnap_free_objective(B, S, K, D, N, derivative, _hptr(mask), _dptr(fixed_values, torch.float64),
                                             _dptr(free_values, torch.float64), _dptr(times, torch.float64), float(w_d),
                                             float(w_c), float(w_t), *margs, _dptr(obj), _dptr(terms.get("Jd")),
                                             _dptr(terms.get("Jc")), _dptr(terms.get("is_collision")), _stream()),
               "minsnap_free_objective")
    return (obj, terms) if want_terms else obj


def optimize_free_constraints(mask, fixed_values, free_values, times, sdf, origin, resolution, min_bound, max_bound, w_c,
                              w_d=0.1, w_t=1.0, optimize_times=False, iterations=20, n_steps=8, max_relative_step=0.5,
                              min_time=0.1, gradient_increment=1e-3, dt=0.1, map_resolution=None, epsilon=0.5,
                              robot_radius=0.5, coll_pot_multiplier=1.0, use_continuous_distance=True, oob_value=0.0,
                              N=10, derivative=SNAP):
    """Additive batched driver for the reference's nonlinear problem over the free derivatives (and, with
    optimize_times, the segment times): every trajectory descends J = w_d J_d + w_c J_c + w_t sum(T) along a
    Jacobi-scaled step, the line search is one evaluation of n_steps candidates.  One C-ABI call
    (minsnap_optimize_free_constraints): the whole loop is enqueued on the current stream.  The reference runs one
    NLopt instance per trajectory on the host.  Returns (free_values, times, objective history [iterations + 1][B],
    is_collision [B] at the returned state)."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, _, D = fixed_values.shape
    free_values = free_values.clone().contiguous()
    times = times.clone().contiguous()
    history = torch.empty((iterations + 1, B), dtype=torch.float64, device=times.device)
    hit = torch.empty((B,), dtype=torch.int32, device=times.device)
    host, margs = _collision_map(sdf, origin, resolution, min_bound, max_bound, dt, map_resolution, epsilon, robot_radius,
                                 coll_pot_multiplier, use_continuous_distance, oob_value)
    capi.check(_lib().minsnap_optimize_free_constraints(B, K, D, N, derivative, _hptr(mask),
                                                        _dptr(fixed_values, torch.float64), _dptr(free_values),
                                                        _dptr(times), int(bool(optimize_times)), float(w_d), float(w_c),
                                                        float(w_t), *margs, int(iterations), int(n_steps),
                                                        float(max_relative_step), float(min_time),
                                                        float(gradient_increment), _dptr(history), _dptr(hit), _stream()),
               "minsnap_optimize_free_constraints")
    return free_values, times, history, hit


def optimize_free_constraints_reference_glue(mask, fixed_values, free_values, times, sdf, origin, resolution, min_bound,
                                             max_bound, w_c, w_d=0.1, w_t=1.0, optimize_times=False, iterations=20,
                                             n_steps=8, max_relative_step=0.5, min_time=0.1, gradient_increment=1e-3,
                                             N=10, derivative=SNAP, **map_kw):
    """The descent of optimize_free_constraints with its glue written in elementwise torch operations around the
    C-ABI calls (derivative_gradient, collision_gradient, time_gradient, free_objective): kept as the checker of
    minsnap_optimize_free_constraints in the tests."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, n_fixed, D = fixed_values.shape
    dev = times.device
    col, counts = reorder(torch.from_numpy(mask.reshape(1, -1)).to(dev), N, K)
    n_free = int(counts[0, 1])
    free, times = free_values.clone(), times.clone()
    S = n_steps

    def objective(f, t):
        return free_objective(mask, fixed_values, f.contiguous(), t.contiguous(), sdf, origin, resolution, min_bound,
                              max_bound, w_c, w_d=w_d, w_t=w_t, N=N, derivative=derivative, want_terms=True, **map_kw)

    obj0, terms0 = objective(free[:, None], times[:, None])
    history, hit = [obj0[:, 0]], terms0["is_collision"][:, 0]
    ladder = 0.5 ** torch.arange(S, dtype=torch.float64, device=dev)
    rows = torch.arange(B, device=dev)
    for _ in range(iterations):
        dg = derivative_gradient(mask, fixed_values, free, times, N=N, derivative=derivative, want_coeffs=True,
                                 want_diag=True)
        cg = collision_gradient(dg["coeffs"], times, sdf, origin, resolution, min_bound, max_bound, col_of_row=col[0],
                                n_fixed=n_fixed, n_free=n_free, **map_kw)
        step = (w_d * dg["gradient"] + w_c * cg["gradient"]) / ((2.0 * w_d) * dg["diag"][:, :, None])
        cand_free = free[:, None] - ladder[None, :, None, None] * step[:, None]
        if optimize_times:
            g = time_gradient(dg["coeffs"], times, increment=gradient_increment, w_d=w_d, w_t=w_t, derivative=derivative)
            scale = (times / g.abs().clamp_min(1e-300)).min(1, keepdim=True).values
            cand_t = times[:, None, :] - ((max_relative_step * ladder)[None, :, None] * scale[:, :, None]) * g[:, None, :]
            cand_t = cand_t.clamp_min(min_time)
        else:
            cand_t = times[:, None, :].expand(B, S, K)
        obj, terms = objective(cand_free, cand_t)
        best, arg = torch.where(torch.isfinite(obj), obj, torch.full_like(obj, float("inf"))).min(1)
        improved = torch.isfinite(best) & (best < history[-1])
        free = torch.where(improved[:, None, None], cand_free[rows, arg], free)
        times = torch.where(improved[:, None], cand_t[rows, arg], times)
        hit = torch.where(improved, terms["is_collision"][rows, arg], hit)
        history.append(torch.where(improved, best, history[-1]))
    return free, times, torch.stack(history), hit


# ---- the soft limits in the free-derivative problem: J + w_sc soft ----------------------------------------------------
def soft_constraint_gradient(mask, coeffs, times, constraints, soft_constraint_weight=100.0, maximum_cost=1.0e12,
                             keep_small=False, want_times=True):
    """The soft cost of soft_constraint_cost and its closed-form gradient in the free derivatives and, with the
    end-point derivatives held fixed, in the segment times (minsnap_soft_constraint_gradient).  mask: host uint8
    [(K+1)][h]; coeffs [B][K][D][N], times [B][K] -> dict(cost [B], grad_free [B][n_free][D], grad_times [B][K] or
    None, max_value, max_time, max_segment [B][n_constraints]: the maximum and its time and segment)."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    B, K, D, N = coeffs.shape
    n_c = len(constraints)
    _, n_free = mask_counts(mask)
    dev = coeffs.device
    out = dict(cost=torch.empty((B,), dtype=torch.float64, device=dev),
               grad_free=torch.empty((B, n_free, D), dtype=torch.float64, device=dev),
               grad_times=torch.empty((B, K), dtype=torch.float64, device=dev) if want_times else None,
               max_value=torch.empty((B, n_c), dtype=torch.float64, device=dev),
               max_time=torch.empty((B, n_c), dtype=torch.float64, device=dev),
               max_segment=torch.empty((B, n_c), dtype=torch.int32, device=dev))
    host, sargs = _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small)
    capi.check(_lib().minsnap_soft_constraint_gradient(B, K, D, N, _hptr(mask), _dptr(coeffs, torch.float64),
                                                       _dptr(times, torch.float64), *sargs, _dptr(out["cost"]),
                                                       _dptr(out["grad_free"]), _dptr(out["grad_times"]),
                                                       _dptr(out["max_value"]), _dptr(out["max_time"]),
                                                       _dptr(out["max_segment"]), _stream()),
               "minsnap_soft_constraint_gradient")
    return out


def free_objective_soft(mask, fixed_values, free_values, times, sdf, origin, resolution, min_bound, max_bound, w_c,
                        constraints, w_sc, w_d=0.1, w_t=1.0, soft_constraint_weight=100.0, maximum_cost=1.0e12,
                        keep_small=False, dt=0.1, map_resolution=None, epsilon=0.5, robot_radius=0.5,
                        coll_pot_multiplier=1.0, use_continuous_distance=True, oob_value=0.0, N=10, derivative=SNAP,
                        want_terms=False):
    """free_objective plus w_sc times the soft cost of the recovered candidates, added last
    (minsnap_free_objective_soft).  Shapes as free_objective; with want_terms also dict(Jd, Jc, is_collision, soft),
    each [B][S]."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, S = times.shape[0], times.shape[1]
    D = fixed_values.shape[2]
    dev = times.device
    obj = torch.empty((B, S), dtype=torch.float64, device=dev)
    terms = dict(Jd=torch.empty((B, S), dtype=torch.float64, device=dev),
                 Jc=torch.empty((B, S), dtype=torch.float64, device=dev),
                 is_collision=torch.empty((B, S), dtype=torch.int32, device=dev),
                 soft=torch.empty((B, S), dtype=torch.float64, device=dev)) if want_terms else {}
    host, margs = _collision_map(sdf, origin, resolution, min_bound, max_bound, dt, map_resolution, epsilon, robot_radius,
                                 coll_pot_multiplier, use_continuous_distance, oob_value)
    shost, sargs = _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small)
    capi.check(_lib().minsnap_free_objective_soft(B, S, K, D, N, derivative, _hptr(mask),
                                                  _dptr(fixed_values, torch.float64), _dptr(free_values, torch.float64),
                                                  _dptr(times, torch.float64), float(w_d), float(w_c), float(w_t), *margs,
                                                  *sargs, float(w_sc), _dptr(obj), _dptr(terms.get("Jd")),
                                                  _dptr(terms.get("Jc")), _dptr(terms.get("is_collision")),
                                                  _dptr(terms.get("soft")), _stream()), "minsnap_free_objective_soft")
    return (obj, terms) if want_terms else obj


def optimize_free_constraints_soft(mask, fixed_values, free_values, times, sdf, origin, resolution, min_bound,
                                   max_bound, w_c, constraints, w_sc, w_d=0.1, w_t=1.0, optimize_times=False,
                                   iterations=20, n_steps=8, max_relative_step=0.5, min_time=0.1,
                                   gradient_increment=1e-3, soft_constraint_weight=100.0, maximum_cost=1.0e12,
                                   keep_small=False, dt=0.1, map_resolution=None, epsilon=0.5, robot_radius=0.5,
                                   coll_pot_multiplier=1.0, use_continuous_distance=True, oob_value=0.0, N=10,
                                   derivative=SNAP):
    """optimize_free_constraints on the objective of free_objective_soft: the soft term's closed-form gradient joins
    the step (and, with optimize_times, the time gradient).  One C-ABI call (minsnap_optimize_free_constraints_soft).
    Returns (free_values, times, objective history [iterations + 1][B], is_collision [B], max_value
    [B][n_constraints]), the last two at the returned state."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, _, D = fixed_values.shape
    free_values = free_values.clone().contiguous()
    times = times.clone().contiguous()
    dev = times.device
    history = torch.empty((iterations + 1, B), dtype=torch.float64, device=dev)
    hit = torch.empty((B,), dtype=torch.int32, device=dev)
    peak = torch.empty((B, len(constraints)), dtype=torch.float64, device=dev)
    host, margs = _collision_map(sdf, origin, resolution, min_bound, max_bound, dt, map_resolution, epsilon, robot_radius,
                                 coll_pot_multiplier, use_continuous_distance, oob_value)
    shost, sargs = _soft_args(constraints, soft_constraint_weight, maximum_cost, keep_small)
    capi.check(_lib().minsnap_optimize_free_constraints_soft(B, K, D, N, derivative, _hptr(mask),
                                                             _dptr(fixed_values, torch.float64), _dptr(free_values),
                                                             _dptr(times), int(bool(optimize_times)), float(w_d),
                                                             float(w_c), float(w_t), *margs, *sargs, float(w_sc),
                                                             int(iterations), int(n_steps), float(max_relative_step),
                                                             float(min_time), float(gradient_increment), _dptr(history),
                                                             _dptr(hit), _dptr(peak), _stream()),
               "minsnap_optimize_free_constraints_soft")
    return free_values, times, history, hit, peak


def optimize_free_constraints_soft_reference_glue(mask, fixed_values, free_values, times, sdf, origin, resolution,
                                                  min_bound, max_bound, w_c, constraints, w_sc, w_d=0.1, w_t=1.0,
                                                  optimize_times=False, iterations=20, n_steps=8, max_relative_step=0.5,
                                                  min_time=0.1, gradient_increment=1e-3, soft_constraint_weight=100.0,
                                                  maximum_cost=1.0e12, keep_small=False, N=10, derivative=SNAP,
                                                  **map_kw):
    """The descent of optimize_free_constraints_soft with its glue written in elementwise torch operations around the
    C-ABI calls (derivative_gradient, collision_gradient, time_gradient, soft_constraint_gradient,
    free_objective_soft): kept as the checker of minsnap_optimize_free_constraints_soft in the tests."""
    torch = _torch()
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    B, n_fixed, D = fixed_values.shape
    dev = times.device
    col, counts = reorder(torch.from_numpy(mask.reshape(1, -1)).to(dev), N, K)
    n_free = int(counts[0, 1])
    free, times = free_values.clone(), times.clone()
    S = n_steps
    soft_kw = dict(soft_constraint_weight=soft_constraint_weight, maximum_cost=maximum_cost, keep_small=keep_small)

    def objective(f, t):
        return free_objective_soft(mask, fixed_values, f.contiguous(), t.contiguous(), sdf, origin, resolution,
                                   min_bound, max_bound, w_c, constraints, w_sc, w_d=w_d, w_t=w_t, N=N,
                                   derivative=derivative, want_terms=True, **soft_kw, **map_kw)

    obj0, terms0 = objective(free[:, None], times[:, None])
    history, hit = [obj0[:, 0]], terms0["is_collision"][:, 0]
    ladder = 0.5 ** torch.arange(S, dtype=torch.float64, device=dev)
    rows = torch.arange(B, device=dev)
    for _ in range(iterations):
        dg = derivative_gradient(mask, fixed_values, free, times, N=N, derivative=derivative, want_coeffs=True,
                                 want_diag=True)
        cg = collision_gradient(dg["coeffs"], times, sdf, origin, resolution, min_bound, max_bound, col_of_row=col[0],
                                n_fixed=n_fixed, n_free=n_free, **map_kw)
        sg = soft_constraint_gradient(mask, dg["coeffs"], times, constraints, want_times=optimize_times, **soft_kw)
        step = (w_d * dg["gradient"] + w_c * cg["gradient"] + w_sc * sg["grad_free"]) / ((2.0 * w_d) * dg["diag"][:, :, None])
        cand_free = free[:, None] - ladder[None, :, None, None] * step[:, None]
        if optimize_times:
            g = time_gradient(dg["coeffs"], times, increment=gradient_increment, w_d=w_d, w_t=w_t, derivative=derivative)
            g = g + w_sc * sg["grad_times"]
            scale = (times / g.abs().clamp_min(1e-300)).min(1, keepdim=True).values
            cand_t = times[:, None, :] - ((max_relative_step * ladder)[None, :, None] * scale[:, :, None]) * g[:, None, :]
            cand_t = cand_t.clamp_min(min_time)
        else:
            cand_t = times[:, None, :].expand(B, S, K)
        obj, terms = objective(cand_free, cand_t)
        # the first minimum, as the select kernel takes it: a saturated soft term (maximum_cost) leaves the small
        # ladder steps tied, and min(1) does not say which index it returns at a tie
        obj = torch.where(torch.isfinite(obj), obj, torch.full_like(obj, float("inf")))
        best = obj.min(1).values
        arg = (obj == best[:, None]).to(torch.uint8).argmax(1)
        improved = torch.isfinite(best) & (best < history[-1])
        free = torch.where(improved[:, None, None], cand_free[rows, arg], free)
        times = torch.where(improved[:, None], cand_t[rows, arg], times)
        hit = torch.where(improved, terms["is_collision"][rows, arg], hit)
        history.append(torch.where(improved, best, history[-1]))
    return free, times, torch.stack(history), hit


EXTREMA_OPTIMIZATION = 0   # PolynomialOptimization::computeMaximumOfMagnitude (ref LIN.i:470-503)
EXTREMA_TRAJECTORY = 1     # Trajectory::computeMinMaxMagnitude (ref src/trajectory.cpp:181-217)
EXTREMA_KEEP_SMALL_COEFFICIENTS = 16   # OR into mode: do not truncate coefficients below 2.2e-16


def _dim_mask(D, dimensions):
    if dimensions is None:
        return (1 << D) - 1
    m = 0
    for d in dimensions:
        if not 0 <= int(d) < D:
            raise ValueError("dimension %r out of bounds [0..%d]" % (d, D - 1))
        m |= 1 << int(d)
    return m


def extrema_max_roots(N, derivative, n_dims):
    return _lib().minsnap_extrema_max_roots(N, derivative, n_dims)


def extrema(coeffs, times, derivative, mode=EXTREMA_OPTIMIZATION, dimensions=None, want_roots=False):
    """coeffs [B][K][D][N], times [B][K] (CUDA tensors) -> dict of [B] tensors: max_time, max_value,
    max_segment (and min_* in EXTREMA_TRAJECTORY mode); with want_roots also the per-segment
    candidate lists cand_times / cand_values [B][K][max_roots + 2] (start, end, roots ascending),
    root_count [B][K] and root_times (= cand_times[..., 2:]).  Times are local to the segment."""
    torch = _torch()
    B, K, D, N = coeffs.shape
    dev = coeffs.device
    mask = _dim_mask(D, dimensions)
    r = dict(max_time=torch.empty((B,), dtype=torch.float64, device=dev),
             max_value=torch.empty((B,), dtype=torch.float64, device=dev),
             max_segment=torch.empty((B,), dtype=torch.int32, device=dev))
    if mode & ~EXTREMA_KEEP_SMALL_COEFFICIENTS == EXTREMA_TRAJECTORY:
        r.update(min_time=torch.empty((B,), dtype=torch.float64, device=dev),
                 min_value=torch.empty((B,), dtype=torch.float64, device=dev),
                 min_segment=torch.empty((B,), dtype=torch.int32, device=dev))
    if want_roots:
        mr = extrema_max_roots(N, derivative, bin(mask).count("1"))
        r["cand_times"] = torch.zeros((B, K, mr + 2), dtype=torch.float64, device=dev)
        r["cand_values"] = torch.zeros((B, K, mr + 2), dtype=torch.float64, device=dev)
        r["root_count"] = torch.empty((B, K), dtype=torch.int32, device=dev)
    capi.check(_lib().minsnap_extrema(B, K, D, N, _dptr(coeffs, torch.float64), _dptr(times, torch.float64),
                                      derivative, mode, mask, _dptr(r["max_time"]), _dptr(r["max_value"]),
                                      _dptr(r["max_segment"]), _dptr(r.get("min_time")), _dptr(r.get("min_value")),
                                      _dptr(r.get("min_segment")), _dptr(r.get("cand_times")),
                                      _dptr(r.get("cand_values")), _dptr(r.get("root_count")), _stream()),
               "minsnap_extrema")
    if want_roots:
        r["root_times"] = r["cand_times"][:, :, 2:]
    return r


# ------------------------------------------------------------------------------------------
# host-buffer entry points (numpy arrays, synchronous, copies inside)
# ------------------------------------------------------------------------------------------
def extrema_host(coeffs, times, derivative, mode=EXTREMA_OPTIMIZATION, dimensions=None, want_roots=False):
    """numpy variant of extrema()."""
    coeffs = _np(coeffs, np.float64)
    times = _np(times, np.float64)
    B, K, D, N = coeffs.shape
    mask = _dim_mask(D, dimensions)
    r = dict(max_time=np.empty((B,), np.float64), max_value=np.empty((B,), np.float64),
             max_segment=np.empty((B,), np.int32))
    if mode & ~EXTREMA_KEEP_SMALL_COEFFICIENTS == EXTREMA_TRAJECTORY:
        r.update(min_time=np.empty((B,), np.float64), min_value=np.empty((B,), np.float64),
                 min_segment=np.empty((B,), np.int32))
    if want_roots:
        mr = extrema_max_roots(N, derivative, bin(mask).count("1"))
        r["cand_times"] = np.zeros((B, K, mr + 2), np.float64)
        r["cand_values"] = np.zeros((B, K, mr + 2), np.float64)
        r["root_count"] = np.empty((B, K), np.int32)
    capi.check(_lib().minsnap_extrema_host(B, K, D, N, _hptr(coeffs), _hptr(times), derivative, mode, mask,
                                           _hptr(r["max_time"]), _hptr(r["max_value"]), _hptr(r["max_segment"]),
                                           _hptr(r.get("min_time")), _hptr(r.get("min_value")),
                                           _hptr(r.get("min_segment")), _hptr(r.get("cand_times")),
                                           _hptr(r.get("cand_values")), _hptr(r.get("root_count"))),
               "minsnap_extrema_host")
    if want_roots:
        r["root_times"] = r["cand_times"][:, :, 2:]
    return r


def solve_host(mask, fixed_values, times, N=10, derivative=SNAP):
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    fixed_values = _np(fixed_values, np.float64)
    times = _np(times, np.float64)
    B, n_fixed, D = fixed_values.shape
    _, n_free = mask_counts(mask)
    coeffs = np.empty((B, K, D, N), np.float64)
    free = np.empty((B, n_free, D), np.float64)
    cost_a = np.empty((B,), np.float64)
    status = np.empty((B,), np.int32)
    col = np.empty((N * K,), np.int32)
    capi.check(_lib().minsnap_solve_host(B, K, D, N, derivative, _hptr(mask), _hptr(fixed_values), _hptr(times),
                                         _hptr(coeffs), _hptr(free), _hptr(cost_a), _hptr(status), _hptr(col)),
               "minsnap_solve_host")
    return dict(coeffs=coeffs, free_values=free, cost=cost_a, status=status, col_of_row=col)


def solve_standard_host(positions, times=None, end_derivatives=None, v_max=0.0, a_max=0.0, magic=6.5, N=10,
                        derivative=SNAP, coeffs=None, want_free=False, want_cost=False, want_status=False):
    """positions/times/coeffs may be numpy arrays or pinned CPU torch tensors (zero-copy)."""
    def host(a):
        if a is None:
            return None, None
        if isinstance(a, np.ndarray):
            a = np.ascontiguousarray(a, np.float64)
            return a, a.ctypes.data_as(C.c_void_p)
        assert not a.is_cuda and a.is_contiguous()
        return a, C.c_void_p(a.data_ptr())

    positions, p_pos = host(positions)
    times, p_t = host(times)
    end_derivatives, p_end = host(end_derivatives)
    B, K1, D = positions.shape
    K = K1 - 1
    h = N // 2
    if coeffs is None:
        coeffs = np.empty((B, K, D, N), np.float64)
    coeffs, p_c = host(coeffs)
    free = np.empty((B, (K - 1) * (h - 1), D), np.float64) if want_free else None
    cost_a = np.empty((B,), np.float64) if want_cost else None
    status = np.empty((B,), np.int32) if want_status else None
    times_out = np.empty((B, K), np.float64) if times is None else None
    capi.check(_lib().minsnap_solve_standard_host(B, K, D, N, derivative, p_pos, p_end, p_t, v_max, a_max, magic,
                                                  _hptr(times_out), p_c, _hptr(free), _hptr(cost_a), _hptr(status)),
               "minsnap_solve_standard_host")
    return dict(coeffs=coeffs, free_values=free, cost=cost_a, status=status,
                times=times if times is not None else times_out)


def sample_at_host(coeffs, times, t, n_deriv=5):
    coeffs = _np(coeffs, np.float64)
    times = _np(times, np.float64)
    t = _np(t, np.float64)
    B, K, D, N = coeffs.shape
    M = t.shape[-1]
    stride = 0 if t.ndim == 1 else M
    out = np.empty((B, M, n_deriv, D), np.float64)
    seg = np.empty((B, M), np.int32)
    capi.check(_lib().minsnap_sample_at_host(B, K, D, N, _hptr(coeffs), _hptr(times), M, _hptr(t), stride, n_deriv,
                                             _hptr(out), _hptr(seg)), "minsnap_sample_at_host")
    return out, seg


def evaluate_range_host(coeffs, times, t_start, t_end, dt, derivative, max_samples=1 << 16):
    coeffs = _np(coeffs, np.float64)
    times = _np(times, np.float64)
    K, D, N = coeffs.shape
    out = np.zeros((max_samples, D), np.float64)
    t_out = np.zeros((max_samples,), np.float64)
    count = C.c_int32()
    capi.check(_lib().minsnap_evaluate_range_host(K, D, N, _hptr(coeffs), _hptr(times), t_start, t_end, dt, derivative,
                                                  max_samples, _hptr(out), _hptr(t_out), C.byref(count)),
               "minsnap_evaluate_range_host")
    n = min(count.value, max_samples)
    return out[:n].copy(), t_out[:n].copy(), count.value


def segment_matrices_host(T, N=10, derivative=SNAP):
    T = _np(np.atleast_1d(T), np.float64)
    n = T.shape[0]
    out = {k: np.empty((n, N, N), np.float64) for k in ("A", "Ainv", "Q", "H")}
    capi.check(_lib().minsnap_segment_matrices_host(n, N, derivative, _hptr(T), _hptr(out["A"]), _hptr(out["Ainv"]),
                                                    _hptr(out["Q"]), _hptr(out["H"])), "minsnap_segment_matrices_host")
    return out


def estimate_segment_times_host(positions, v_max, a_max, magic=6.5):
    positions = _np(positions, np.float64)
    B, K1, D = positions.shape
    times = np.empty((B, K1 - 1), np.float64)
    capi.check(_lib().minsnap_estimate_segment_times_host(B, K1 - 1, D, _hptr(positions), v_max, a_max, magic,
                                                          _hptr(times)), "minsnap_estimate_segment_times_host")
    return times


def coeffs_from_constraints_host(mask, fixed_values, free_values, times, N=10):
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    fixed_values = _np(fixed_values, np.float64)
    free_values = _np(free_values, np.float64)
    times = _np(times, np.float64)
    B, _, D = fixed_values.shape
    coeffs = np.empty((B, K, D, N), np.float64)
    capi.check(_lib().minsnap_coeffs_from_constraints_host(B, K, D, N, _hptr(mask), _hptr(fixed_values),
                                                           _hptr(free_values), _hptr(times), _hptr(coeffs)),
               "minsnap_coeffs_from_constraints_host")
    return coeffs


def derivative_gradient_host(mask, fixed_values, free_values, times, N=10, derivative=SNAP):
    """numpy variant of derivative_gradient(): dict(Jd, gradient, diag, coeffs)."""
    mask = np.ascontiguousarray(mask, np.uint8)
    K = mask.shape[0] - 1
    fixed_values, free_values, times = _np(fixed_values, np.float64), _np(free_values, np.float64), _np(times, np.float64)
    B, _, D = fixed_values.shape
    _, n_free = mask_counts(mask)
    out = dict(Jd=np.empty((B,), np.float64), gradient=np.empty((B, n_free, D), np.float64),
               diag=np.empty((B, n_free), np.float64), coeffs=np.empty((B, K, D, N), np.float64))
    capi.check(_lib().minsnap_derivative_gradient_host(B, K, D, N, derivative, _hptr(mask), _hptr(fixed_values),
                                                       _hptr(free_values), _hptr(times), _hptr(out["coeffs"]),
                                                       _hptr(out["Jd"]), _hptr(out["gradient"]), _hptr(out["diag"])),
               "minsnap_derivative_gradient_host")
    return out


def cost_host(coeffs, times, derivative=SNAP):
    coeffs = _np(coeffs, np.float64)
    times = _np(times, np.float64)
    B, K, D, N = coeffs.shape
    out = np.empty((B,), np.float64)
    capi.check(_lib().minsnap_cost_host(B, K, D, N, derivative, _hptr(coeffs), _hptr(times), _hptr(out)),
               "minsnap_cost_host")
    return out


def sample_uniform_host(coeffs, times, M, n_deriv=5, want_times=False):
    coeffs, times = _np(coeffs, np.float64), _np(times, np.float64)
    B, K, D, N = coeffs.shape
    out = np.empty((B, M, n_deriv, D), np.float64)
    t_out = np.empty((B, M), np.float64) if want_times else None
    capi.check(_lib().minsnap_sample_uniform_host(B, K, D, N, _hptr(coeffs), _hptr(times), M, n_deriv, _hptr(out),
                                                  _hptr(t_out)), "minsnap_sample_uniform_host")
    return (out, t_out) if want_times else out


def cost_sweep_host(positions, times, end_derivatives=None, N=10, derivative=SNAP, want_status=False):
    """positions [B][K+1][D], times [B][S][K] (host) -> cost [B][S] (BASELINE configs[4] from host buffers)."""
    positions, times, end_derivatives = _np(positions, np.float64), _np(times, np.float64), _np(end_derivatives, np.float64)
    B, K1, D = positions.shape
    S = times.shape[1]
    out = np.empty((B, S), np.float64)
    status = np.empty((B, S), np.int32) if want_status else None
    capi.check(_lib().minsnap_cost_sweep_host(B, S, K1 - 1, D, N, derivative, _hptr(positions), _hptr(end_derivatives),
                                              _hptr(times), _hptr(out), _hptr(status)), "minsnap_cost_sweep_host")
    return (out, status) if want_status else out


def time_objective_host(positions, times, time_penalty, end_derivatives=None, N=10, derivative=SNAP, want_cost=False):
    positions, times, end_derivatives = _np(positions, np.float64), _np(times, np.float64), _np(end_derivatives, np.float64)
    B, K1, D = positions.shape
    S = times.shape[1]
    out = np.empty((B, S), np.float64)
    cost_a = np.empty((B, S), np.float64) if want_cost else None
    capi.check(_lib().minsnap_time_objective_host(B, S, K1 - 1, D, N, derivative, _hptr(positions), _hptr(end_derivatives),
                                                  _hptr(times), float(time_penalty), _hptr(out), _hptr(cost_a), None),
               "minsnap_time_objective_host")
    return (out, cost_a) if want_cost else out


def time_gradient_host(coeffs, times, increment=0.1, w_d=0.1, w_t=1.0, derivative=SNAP, want_segment_cost=False):
    coeffs, times = _np(coeffs, np.float64), _np(times, np.float64)
    B, K, D, N = coeffs.shape
    grad = np.empty((B, K), np.float64)
    seg = np.empty((B, K), np.float64) if want_segment_cost else None
    capi.check(_lib().minsnap_time_gradient_host(B, K, D, N, derivative, _hptr(coeffs), _hptr(times), float(increment),
                                                 float(w_d), float(w_t), _hptr(grad), _hptr(seg)), "minsnap_time_gradient_host")
    return (grad, seg) if want_segment_cost else grad


def collision_cost_host(coeffs, times, sdf, origin, resolution, min_bound, max_bound, dt=0.1, map_resolution=None,
                        epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.0, use_continuous_distance=True, oob_value=0.0):
    """numpy variant of collision_cost()."""
    coeffs, times, sdf = _np(coeffs, np.float64), _np(times, np.float64), _np(sdf, np.float64)
    B, K, D, N = coeffs.shape
    if map_resolution is None:
        map_resolution = resolution
    dims = np.asarray(sdf.shape, np.int32)
    org, lo, hi = _np(origin, np.float64), _np(min_bound, np.float64), _np(max_bound, np.float64)
    cost_a, hit, charged = np.empty((B,), np.float64), np.empty((B,), np.int32), np.empty((B,), np.int32)
    capi.check(_lib().minsnap_collision_cost_host(B, K, D, N, _hptr(coeffs), _hptr(times), _hptr(sdf), _hptr(dims), _hptr(org),
                                                  float(resolution), float(oob_value), _hptr(lo), _hptr(hi),
                                                  int(bool(use_continuous_distance)), float(dt), float(map_resolution),
                                                  float(epsilon), float(robot_radius), float(coll_pot_multiplier),
                                                  _hptr(cost_a), _hptr(hit), _hptr(charged)), "minsnap_collision_cost_host")
    return dict(cost=cost_a, is_collision=hit, charged=charged)


def collision_gradient_host(coeffs, times, sdf, origin, resolution, min_bound, max_bound, dt=0.1, map_resolution=None,
                            epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.0, use_continuous_distance=True,
                            oob_value=0.0, col_of_row=None, n_fixed=0, n_free=None):
    """numpy variant of collision_gradient()."""
    coeffs, times, sdf = _np(coeffs, np.float64), _np(times, np.float64), _np(sdf, np.float64)
    B, K, D, N = coeffs.shape
    if map_resolution is None:
        map_resolution = resolution
    if col_of_row is None:
        n_fixed, n_free = K + N - 1, (K - 1) * (N // 2 - 1)
        col = None
    else:
        col = _np(col_of_row, np.int32)
    dims = np.asarray(sdf.shape, np.int32)
    org, lo, hi = _np(origin, np.float64), _np(min_bound, np.float64), _np(max_bound, np.float64)
    cost_a, hit, charged = np.empty((B,), np.float64), np.empty((B,), np.int32), np.empty((B,), np.int32)
    grad = np.empty((B, n_free, 3), np.float64)
    capi.check(_lib().minsnap_collision_gradient_host(B, K, D, N, _hptr(coeffs), _hptr(times), _hptr(sdf), _hptr(dims),
                                                      _hptr(org), float(resolution), float(oob_value), _hptr(lo), _hptr(hi),
                                                      int(bool(use_continuous_distance)), float(dt), float(map_resolution),
                                                      float(epsilon), float(robot_radius), float(coll_pot_multiplier),
                                                      _hptr(col) if col is not None else None, int(n_fixed), int(n_free),
                                                      _hptr(cost_a), _hptr(grad), _hptr(hit), _hptr(charged)),
               "minsnap_collision_gradient_host")
    return dict(cost=cost_a, gradient=grad, is_collision=hit, charged=charged)


def save_npy(path, array):
    """float64 array -> .npy through the C ABI (minsnap_npy_write_f64); numpy.load reads it."""
    a = np.ascontiguousarray(array, np.float64)
    shape = np.asarray(a.shape, np.int64)
    capi.check(_lib().minsnap_npy_write_f64(str(path).encode(), _hptr(a), a.ndim, _hptr(shape)), "minsnap_npy_write_f64")


def load_npy(path):
    """.npy (little-endian float64, C order; e.g. written by numpy.save) -> array through the C ABI."""
    ndim = C.c_int()
    shape = np.zeros(8, np.int64)
    capi.check(_lib().minsnap_npy_read_f64(str(path).encode(), None, 0, C.byref(ndim), _hptr(shape)), "minsnap_npy_read_f64")
    out = np.empty(tuple(int(x) for x in shape[: ndim.value]), np.float64)
    capi.check(_lib().minsnap_npy_read_f64(str(path).encode(), _hptr(out), out.size, C.byref(ndim), _hptr(shape)),
               "minsnap_npy_read_f64")
    return out


def sampled_table_host(coeffs, times, dt=0.01, path=None):
    """The table of the reference's printMatlabSampledTrajectory (NL.i:2567-2662) for one trajectory:
    coeffs [K][D][N], times [K] (host) -> [rows][5 D + 2]; written as text when path is given."""
    coeffs = _np(coeffs, np.float64)
    times = _np(times, np.float64)
    K, D, N = coeffs.shape
    rows = _lib().minsnap_sampled_table_rows(K, _hptr(times), float(dt))
    table = np.empty((rows, 5 * D + 2), np.float64)
    r, c = C.c_int(), C.c_int()
    capi.check(_lib().minsnap_sampled_table_host(K, D, N, _hptr(coeffs), _hptr(times), float(dt), _hptr(table), rows,
                                                 C.byref(r), C.byref(c)), "minsnap_sampled_table_host")
    if path is not None:
        capi.check(_lib().minsnap_table_write_text(str(path).encode(), _hptr(table), rows, 5 * D + 2), "minsnap_table_write_text")
    return table


def random_positions_host(B, K, pos_min, pos_max, base_seed):
    """Batched createRandomVertices positions (host-only workload generator): [B][K+1][D]."""
    pos_min = _np(pos_min, np.float64)
    pos_max = _np(pos_max, np.float64)
    D = pos_min.shape[0]
    out = np.empty((B, K + 1, D), np.float64)
    capi.check(_lib().minsnap_random_positions_host(B, K, D, _hptr(pos_min), _hptr(pos_max), base_seed, _hptr(out)),
               "minsnap_random_positions_host")
    return out


# solve_standard runs the single-launch thread-pair kernel for N = 10, snap, K <= 24, D <= 3
# (csrc/minsnap_standard_fast.cuh); other shapes take the 4-launch generic route.
STANDARD_FAST_ROUTE = True


def reorder_host(masks, N, K):
    """masks uint8 [n_masks][(K+1)][h] (host) -> (col_of_row [n_masks][N*K], counts [n_masks][2])."""
    masks = np.ascontiguousarray(masks, np.uint8).reshape(-1, (K + 1) * (N // 2))
    n = masks.shape[0]
    col = np.empty((n, N * K), np.int32)
    counts = np.empty((n, 2), np.int32)
    capi.check(_lib().minsnap_reorder_host(N, K, n, _hptr(masks), _hptr(col), _hptr(counts)), "minsnap_reorder_host")
    return col, counts
