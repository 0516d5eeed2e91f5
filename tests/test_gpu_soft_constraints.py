"""GPU tests of the time-only objective with the reference's soft limits on max |p^(k)| (objectiveFunctionTime with
use_soft_constraints, NL.i:765-832; evaluateMaximumMagnitudeAsSoftConstraint, NL.i:2396-2426, over
evaluateMaximumMagnitudeConstraint, NL.i:2346-2392) and of the device-resident descent built on it.

The oracle side follows the reference with the oracle's own primitives: the objective of helpers.oracle_objective
plus, per constraint (k, limit), min(maximum_cost, exp((max - limit) / limit * weight)) with the maximum of
oracle.minmax_magnitude(..., k, 0) on the oracle's solve.  Tolerance 1e-6 relative, as the torch-glue objective's
test: the exponential multiplies the ~1e-9 relative error of the maximum by the weight of 100.
"""
import numpy as np
import pytest

from helpers import random_batch, standard_mask, vertex_values

pytestmark = pytest.mark.gpu

LIMITS = [(1, 4.0), (2, 2.0)]
WEIGHT, MAX_COST = 100.0, 1.0e12


def oracle_soft(oracle, pos, times, penalty, limits, weight=WEIGHT, maximum_cost=MAX_COST, end=None):
    """(objective, [term per constraint]) as the reference computes them for one trajectory."""
    K, D = times.shape[0], pos.shape[1]
    vals = vertex_values(pos)
    if end is not None:                      # [2][h-1][D]: derivatives 1..h-1 of the first and last vertex
        vals[0, 1:, :] = end[0]
        vals[-1, 1:, :] = end[1]
    r = oracle.solve(10, K, D, 4, standard_mask(K), vals, times)
    total = 0.0
    for t in times:
        total += t
    obj = float(r["cost"]) + total * total * penalty
    terms = []
    for k, limit in limits:
        peak = float(oracle.minmax_magnitude(np.asarray(r["coeffs"], np.float64), times, k, 0)["max"][1])
        terms.append(min(maximum_cost, float(np.exp((peak - limit) / limit * weight))))
    soft = 0.0
    for t in terms:
        soft += t
    return obj + soft, terms


def _cuda(torch, *arrays):
    return [torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in arrays]


# ---- 1. the evaluator -----------------------------------------------------------------------------------------------
def test_soft_constraint_cost_matches_oracle(ms, oracle, torch_cuda):
    torch = torch_cuda
    B, K = 8, 10
    pos, times = random_batch(oracle, B, K)
    rng = np.random.default_rng(11)
    times = times * rng.uniform(0.7, 1.5, (B, K))
    p, t = _cuda(torch, pos, times)
    coeffs = ms.solve_standard(p, t, want_status=False)["coeffs"]
    cost, parts = ms.soft_constraint_cost(coeffs, t, LIMITS, want_terms=True)
    cost, terms = cost.cpu().numpy(), parts["terms"].cpu().numpy()
    for b in range(B):
        _, want = oracle_soft(oracle, pos[b], times[b], 0.0, LIMITS)
        for j, term in enumerate(want):
            assert abs(terms[b, j] - term) <= 1e-6 * term, (b, j, terms[b, j], term)
        assert abs(cost[b] - sum(want)) <= 1e-6 * sum(want)
        assert cost[b] == terms[b, 0] + terms[b, 1]          # the sum from 0 in constraint order


@pytest.mark.parametrize("D", [1, 2, 3])
@pytest.mark.parametrize("keep_small", [False, True])
def test_maxima_equal_extrema_bit_for_bit(ms, oracle, torch_cuda, D, keep_small):
    """max_value of every constraint is minsnap_extrema's mode-0 max_value, the same bits, for k = 0..4 on a ragged
    batch (one not a multiple of the fold's 128 threads), one to four constraints per call."""
    torch = torch_cuda
    B, K = 203, 7
    pos, times = random_batch(oracle, B, K, D=D)
    times = times * np.random.default_rng(D).uniform(0.5, 3.0, (B, K))   # segments past 12 s: truncation matters
    p, t = _cuda(torch, pos, times)
    coeffs = ms.solve_standard(p, t, want_status=False)["coeffs"]
    mode = ms.EXTREMA_OPTIMIZATION | (ms.EXTREMA_KEEP_SMALL_COEFFICIENTS if keep_small else 0)
    want = {k: ms.extrema(coeffs, t, k, mode=mode)["max_value"] for k in range(5)}
    for ks in ([0, 1, 2, 3], [4], [2, 4, 1]):
        cons = [(k, 1.0 + k) for k in ks]
        _, parts = ms.soft_constraint_cost(coeffs, t, cons, keep_small=keep_small, want_terms=True)
        for j, k in enumerate(ks):
            assert torch.equal(parts["max_value"][:, j], want[k]), (D, keep_small, k)


def test_terms_saturate_at_maximum_cost(ms, oracle, torch_cuda):
    torch = torch_cuda
    pos, times = random_batch(oracle, 16, 10)
    p, t = _cuda(torch, pos, times)
    coeffs = ms.solve_standard(p, t, want_status=False)["coeffs"]
    cost, parts = ms.soft_constraint_cost(coeffs, t, [(1, 0.01), (2, 1e6)], maximum_cost=7.0, want_terms=True)
    assert bool((parts["terms"][:, 0] == 7.0).all())
    assert bool((parts["terms"][:, 1] < 1e-30).all())       # far below its limit: exp(-100)
    assert torch.equal(cost, parts["terms"][:, 0] + parts["terms"][:, 1])


# ---- 2. the objective -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("with_end", [False, True])
def test_time_objective_soft_matches_oracle_and_glue(ms, oracle, torch_cuda, with_end):
    torch = torch_cuda
    B, S, K, penalty = 6, 4, 10, 500.0
    pos, times = random_batch(oracle, B, K)
    rng = np.random.default_rng(9)
    cand = times[:, None, :] * rng.uniform(0.7, 1.5, (B, S, K))
    end = rng.uniform(-0.5, 0.5, (B, 2, 4, 3)) if with_end else None
    p, c = _cuda(torch, pos, cand)
    e = _cuda(torch, end)[0] if with_end else None
    obj, parts = ms.time_objective_soft(p, c, penalty, LIMITS, end_derivatives=e, want_terms=True)
    glue, glue_parts = ms.time_objective_with_soft_constraints(p, c, penalty, LIMITS, end_derivatives=e,
                                                               want_terms=True)
    # the same solve and extrema; only the time sum, the order of the additions and torch's rounding of the
    # exponent (a division by a scalar may become a multiplication by its reciprocal) differ
    assert float(((obj - glue).abs() / glue.abs()).max()) <= 1e-12
    assert torch.equal(parts["cost_trajectory"], glue_parts["cost_trajectory"])
    for j in range(len(LIMITS)):
        got, ref = parts["cost_constraints"][j], glue_parts["cost_constraints"][j]
        assert float(((got - ref).abs() / ref.abs()).max()) <= 1e-12
    obj = obj.cpu().numpy()
    for b in range(B):
        for s in range(S):
            want, terms = oracle_soft(oracle, pos[b], cand[b, s], penalty, LIMITS, end=None if end is None else end[b])
            assert abs(obj[b, s] - want) <= 1e-6 * want, (b, s, obj[b, s], want)
            for j, term in enumerate(terms):
                got = float(parts["cost_constraints"][j][b, s])
                assert abs(got - term) <= 1e-6 * term


def test_failed_solve_gives_a_non_finite_objective(ms, oracle, torch_cuda):
    torch = torch_cuda
    B, S, K = 5, 3, 6
    pos, times = random_batch(oracle, B, K)
    cand = np.repeat(times[:, None, :], S, 1)
    cand[1, 2, 3] = 0.0
    cand[4, 0, 0] = -1.0
    p, c = _cuda(torch, pos, cand)
    obj = ms.time_objective_soft(p, c, 500.0, LIMITS).cpu().numpy()
    bad = np.zeros((B, S), bool)
    bad[1, 2] = bad[4, 0] = True
    assert not np.isfinite(obj[bad]).any()
    assert np.isfinite(obj[~bad]).all()


# ---- 3. the driver --------------------------------------------------------------------------------------------------
def test_soft_descent(ms, oracle, torch_cuda):
    torch = torch_cuda
    B, K, penalty = 128, 10, 0.05
    pos, times = random_batch(oracle, B, K)
    p, t0 = _cuda(torch, pos, times)
    t1, hist, peak = ms.optimize_segment_times_soft(p, t0, LIMITS, iterations=12, time_penalty=penalty)
    h = hist.cpu().numpy()
    assert np.all(np.diff(h, axis=0) <= 0)                     # never accepts a worse allocation
    assert np.mean(h[-1] / h[0]) < 0.9
    assert float(t1.min()) >= 0.1
    t1h = t1.cpu().numpy()
    for b in (0, 17, 127):
        want, _ = oracle_soft(oracle, pos[b], t1h[b], penalty, LIMITS)
        assert abs(h[-1, b] - want) <= 1e-6 * want
    coeffs = ms.solve_standard(p, t1, want_status=False)["coeffs"]
    for j, (k, _) in enumerate(LIMITS):
        assert torch.equal(peak[:, j], ms.extrema(coeffs, t1, k, mode=ms.EXTREMA_OPTIMIZATION)["max_value"])


# ---- 4. against the torch glue --------------------------------------------------------------------------------------
def test_device_resident_soft_descent_matches_the_glue_version(ms, oracle, torch_cuda):
    """The same allocations go through the same C-ABI solves and soft costs at the same batch sizes, so the two
    agree to rounding after one iteration (the glue sums the times pairwise and adds the gradient's penalty part
    in torch).  Over ten iterations the central differences amplify last-bit differences of the times, as in
    test_device_resident_descent_matches_the_glue_version, so the histories agree to 1e-4."""
    torch = torch_cuda
    B, K, penalty = 96, 10, 0.05
    pos, times = random_batch(oracle, B, K)
    p, t0 = _cuda(torch, pos, times)
    end = _cuda(torch, np.random.default_rng(3).uniform(-0.5, 0.5, (B, 2, 4, 3)))[0]
    for e in (None, end):
        t_dev, h_dev, _ = ms.optimize_segment_times_soft(p, t0, LIMITS, iterations=1, time_penalty=penalty,
                                                         end_derivatives=e)
        t_ref, h_ref = ms.api.optimize_segment_times_soft_reference_glue(p, t0, LIMITS, iterations=1,
                                                                         time_penalty=penalty, end_derivatives=e)
        assert h_dev.shape == h_ref.shape == (2, B)
        assert float(((h_dev - h_ref).abs() / h_ref.abs()).max()) <= 1e-10
        assert float(((t_dev - t_ref).abs() / t_ref.abs()).max()) <= 1e-10
        t_dev, h_dev, _ = ms.optimize_segment_times_soft(p, t0, LIMITS, iterations=10, time_penalty=penalty,
                                                         end_derivatives=e)
        t_ref, h_ref = ms.api.optimize_segment_times_soft_reference_glue(p, t0, LIMITS, iterations=10,
                                                                         time_penalty=penalty, end_derivatives=e)
        assert float(((h_dev - h_ref).abs() / h_ref.abs()).max()) <= 1e-4
        assert bool((h_dev[1:] <= h_dev[:-1]).all())


# ---- 5. graph capture -----------------------------------------------------------------------------------------------
def test_soft_descent_replays_from_a_cuda_graph(ms, oracle, torch_cuda):
    torch = torch_cuda
    B, K, iterations = 64, 10, 4
    pos, times = random_batch(oracle, B, K)
    p, t0 = _cuda(torch, pos, times)
    t_buf = t0.clone()
    hist = torch.empty((iterations + 1, B), dtype=torch.float64, device="cuda")
    peak = torch.empty((B, 2), dtype=torch.float64, device="cuda")
    ks = np.array([k for k, _ in LIMITS], np.int32)
    lim = np.array([v for _, v in LIMITS], np.float64)
    lib = ms.capi.load()
    api = ms.api

    def enqueue():
        ms.capi.check(lib.minsnap_optimize_segment_times_soft(B, K, 3, 10, 4, api._dptr(p), None, api._dptr(t_buf),
                                                              iterations, 0.05, 16, 0.5, 0.1, 1e-3, 2, api._hptr(ks),
                                                              api._hptr(lim), WEIGHT, MAX_COST, 0, api._dptr(hist),
                                                              api._dptr(peak), api._stream()),
                      "minsnap_optimize_segment_times_soft")
    enqueue()
    torch.cuda.synchronize()
    first_h, first_t, first_p = hist.clone(), t_buf.clone(), peak.clone()
    t_buf.copy_(t0)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        enqueue()
    hist.zero_()
    peak.zero_()
    t_buf.copy_(t0)
    g.replay()
    torch.cuda.synchronize()
    assert torch.equal(hist, first_h) and torch.equal(t_buf, first_t) and torch.equal(peak, first_p)


# ---- 6. it does its job ---------------------------------------------------------------------------------------------
def test_soft_descent_brings_trajectories_within_the_limits(ms, oracle, torch_cuda):
    """256 trajectories whose maxima mostly exceed the limits: the limits are set to 0.9 of the batch's median
    maximum speed and acceleration at the heuristic times, and the time penalty is small (0.05), so the limits
    bind.  The share of trajectories within 1.05x of both limits must rise over 30 iterations to at least 0.6.
    Measured on one NVIDIA B200 at a 1,000 W power limit: 0.297 at the start, 0.715 after 30 iterations."""
    torch = torch_cuda
    B, K = 256, 10
    pos, times = random_batch(oracle, B, K)
    p, t0 = _cuda(torch, pos, times)
    coeffs = ms.solve_standard(p, t0, want_status=False)["coeffs"]
    v0 = ms.extrema(coeffs, t0, 1, mode=ms.EXTREMA_OPTIMIZATION)["max_value"]
    a0 = ms.extrema(coeffs, t0, 2, mode=ms.EXTREMA_OPTIMIZATION)["max_value"]
    limits = [(1, 0.9 * float(v0.median())), (2, 0.9 * float(a0.median()))]

    def share(peak):
        ok = (peak[:, 0] <= 1.05 * limits[0][1]) & (peak[:, 1] <= 1.05 * limits[1][1])
        return float(ok.double().mean())

    start = share(torch.stack([v0, a0], 1))
    t1, hist, peak = ms.optimize_segment_times_soft(p, t0, limits, iterations=30, time_penalty=0.05)
    end = share(peak)
    print("share within 1.05x of both limits: start %.4f, after 30 iterations %.4f" % (start, end))
    assert start < 0.5
    assert end >= 0.6
