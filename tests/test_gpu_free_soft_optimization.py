"""GPU tests of the soft limits in the free-derivative problem: the closed-form gradient of the soft cost
(minsnap_soft_constraint_gradient), the objective J + w_sc soft (minsnap_free_objective_soft) and the descent on it
(minsnap_optimize_free_constraints_soft).

The gradient is checked against the long-double restatement of test_free_soft_cpu.py, evaluated at the (segment,
time) the device reports, and against central differences of minsnap_soft_constraint_cost.  The driver has no
reference counterpart (NLopt is absent); it is checked against the collision-only driver at w_sc = 0, for monotone
descent, against the same descent written as torch glue, for CUDA-graph replay, and for what it does to the limits.
"""
import numpy as np
import pytest

from helpers import compact_fixed, random_batch, standard_mask, vertex_values
from test_collision_cost import field
from test_free_soft_cpu import general_mask, restated_gradient
from test_gpu_free_constraint_optimization import MAP, colliding_problem

pytestmark = pytest.mark.gpu


def recovered(ms, oracle, torch, mask, B, K, D, N, seed, spread=0.5):
    """Random vertices, their fixed values, free values away from the optimum, times and the recovered
    coefficients."""
    pos, times = random_batch(oracle, B, K, D=D, seed=seed)
    fixed = torch.from_numpy(np.stack([compact_fixed(mask, vertex_values(p, N)) for p in pos])).cuda()
    t = torch.from_numpy(times).cuda()
    _, n_free = ms.mask_counts(mask)
    rng = np.random.default_rng(seed)
    free = torch.from_numpy(rng.normal(size=(B, n_free, D)) * spread).cuda()
    coeffs = ms.coeffs_from_constraints(mask, fixed, free, t, N=N)
    return fixed, free, t, coeffs


def limits_below(ms, coeffs, t, ks, frac=0.9):
    """Limits at frac of the batch's median maxima: most terms live, none saturated."""
    peak = ms.soft_constraint_cost(coeffs, t, [(k, 1.0) for k in ks], want_terms=True)[1]["max_value"]
    return [(k, frac * float(peak[:, j].median())) for j, k in enumerate(ks)]


@pytest.mark.parametrize("N", [6, 8, 10, 12])
@pytest.mark.parametrize("D", [1, 2, 3])
@pytest.mark.parametrize("mask_kind", ["standard", "general"])
@pytest.mark.parametrize("keep_small", [False, True])
def test_gradient_matches_the_restatement(ms, oracle, torch_cuda, N, D, mask_kind, keep_small):
    """Every derivative k = 0..min(4, N-2) (k >= N/2 at N = 6): the argmax segment equals the oracle's, its time
    agrees within 1e-6 T (a root of g next to a flat maximum: 3.0e-7 T measured at N = 10, D = 2), and both
    gradients agree with the long-double restatement at the device's (segment, time) within 1e-9 of their largest
    component, plus 64 eps times the restatement's bound on the rounding of each entry
    (entries that vanish in exact arithmetic, at a fixed vertex for instance, come out of a double evaluation as
    cancellation noise of that size); cost and maxima are minsnap_soft_constraint_cost's bits."""
    torch = torch_cuda
    B, K = 13, 5                                  # ragged: not a multiple of the warps per block
    mask = standard_mask(K, N) if mask_kind == "standard" else general_mask(K, N)
    col, n_fixed, n_free = oracle.reorder(N, K, mask)
    fixed, free, t, coeffs = recovered(ms, oracle, torch, mask, B, K, D, N, 500 + 10 * N + D)
    for ks in [[k] for k in range(min(4, N - 2) + 1)] + [[1, 2]]:
        cons = limits_below(ms, coeffs, t, ks)
        out = ms.soft_constraint_gradient(mask, coeffs, t, cons, soft_constraint_weight=10.0, keep_small=keep_small)
        cost, terms = ms.soft_constraint_cost(coeffs, t, cons, soft_constraint_weight=10.0, keep_small=keep_small,
                                              want_terms=True)
        assert torch.equal(out["cost"], cost) and torch.equal(out["max_value"], terms["max_value"])
        c_h, t_h = coeffs.cpu().numpy(), t.cpu().numpy()
        seg, tim = out["max_segment"].cpu().numpy(), out["max_time"].cpu().numpy()
        gf, gt = out["grad_free"].cpu().numpy(), out["grad_times"].cpu().numpy()
        for b in range(B):
            for j, (k, _) in enumerate(cons):
                ot, _, os_ = oracle.minmax_magnitude(c_h[b], t_h[b], k, 0, keep_small=keep_small)["max"]
                assert seg[b, j] == os_
                assert abs(tim[b, j] - float(ot)) <= 1e-6 * t_h[b, seg[b, j]]
            where = [(int(seg[b, j]), float(tim[b, j])) for j in range(len(cons))]
            _, rf, rt, bf, bt = restated_gradient(c_h[b], t_h[b], col, n_fixed, n_free, cons, 10.0, 1e12, where,
                                                  want_bound=True)
            rf, rt, bf, bt = (a.astype(np.float64) for a in (rf, rt, bf, bt))
            scale = max(np.abs(rf).max(initial=0.0), np.abs(rt).max())
            eps = np.finfo(np.float64).eps
            assert (np.abs(gf[b] - rf) <= 1e-9 * scale + 64 * eps * bf).all()
            assert (np.abs(gt[b] - rt) <= 1e-9 * scale + 64 * eps * bt).all()


@pytest.mark.parametrize("N,D", [(10, 3), (6, 2), (12, 1)])
def test_gradient_matches_finite_differences(ms, oracle, torch_cuda, N, D):
    """Central differences of minsnap_soft_constraint_cost over minsnap_coeffs_from_constraints at d_p +/- h and at
    T +/- h with d fixed, within 1e-5 relative, on the entries whose argmax does not move."""
    torch = torch_cuda
    B, K = 6, 4
    mask = standard_mask(K, N)
    fixed, free, t, coeffs = recovered(ms, oracle, torch, mask, B, K, D, N, 77 + N)
    cons = limits_below(ms, coeffs, t, [1, 2])
    out = ms.soft_constraint_gradient(mask, coeffs, t, cons, soft_constraint_weight=10.0)
    _, n_free = ms.mask_counts(mask)

    def soft(f, tt):   # the fixed and free values are d: recovering at moved times holds d fixed
        c = ms.coeffs_from_constraints(mask, fixed, f, tt, N=N)
        r = ms.soft_constraint_gradient(mask, c, tt, cons, soft_constraint_weight=10.0, want_times=False)
        return r["cost"], r["max_segment"]
    base_seg = out["max_segment"]
    h = 1e-6
    n_checked = 0
    for j in range(n_free):
        for d in range(D):
            fp, fm = free.clone(), free.clone()
            fp[:, j, d] += h
            fm[:, j, d] -= h
            (sp, segp), (sm, segm) = soft(fp, t), soft(fm, t)
            ok = (segp == base_seg).all(1) & (segm == base_seg).all(1)
            fd = (sp - sm) / (2 * h)
            g = out["grad_free"][:, j, d]
            scale = out["grad_free"].abs().flatten(1).max(1).values.clamp_min(1e-300)
            assert bool(((g - fd).abs()[ok] <= 1e-5 * scale[ok] + 1e-9 * fd.abs()[ok]).all())
            n_checked += int(ok.sum())
    assert n_checked > 0
    for s in range(K):
        hs = 1e-6 * t[:, s]
        tp, tm = t.clone(), t.clone()
        tp[:, s] += hs
        tm[:, s] -= hs
        (sp, segp), (sm, segm) = soft(free, tp), soft(free, tm)
        ok = (segp == base_seg).all(1) & (segm == base_seg).all(1)
        fd = (sp - sm) / (2 * hs)
        scale = out["grad_times"].abs().max(1).values.clamp_min(1e-300)
        assert bool(((out["grad_times"][:, s] - fd).abs()[ok] <= 1e-5 * scale[ok]).all())


def test_gradient_edge_cases(ms, oracle, torch_cuda):
    """A saturated term and a zero magnitude give a zero gradient; a maximum at the end of the last segment with
    k < N/2 gives a time gradient of zero up to rounding; two calls give the same bits."""
    torch = torch_cuda
    B, K, D, N = 16, 4, 3, 10
    mask = standard_mask(K, N)
    fixed, free, t, coeffs = recovered(ms, oracle, torch, mask, B, K, D, N, 31)
    # saturated: a tiny limit makes exp(...) exceed maximum_cost
    sat = ms.soft_constraint_gradient(mask, coeffs, t, [(1, 1e-3)], maximum_cost=10.0)
    assert bool((sat["cost"] == 10.0).all())
    assert bool((sat["grad_free"] == 0).all()) and bool((sat["grad_times"] == 0).all())
    # zero magnitude: the position of an all-zero trajectory
    zero = ms.soft_constraint_gradient(mask, torch.zeros_like(coeffs), t, [(0, 1.0)])
    assert bool((zero["grad_free"] == 0).all()) and bool((zero["grad_times"] == 0).all())
    # the position's maximum at the end of the last segment: a trajectory moving away from the origin
    c = torch.zeros((1, K, D, N), dtype=torch.float64, device="cuda")
    c[0, :, 0, 1] = 1.0                             # x(t) = t in each segment, offset so x is continuous
    tt = torch.ones((1, K), dtype=torch.float64, device="cuda")
    for s in range(K):
        c[0, s, 0, 0] = float(s)
    end = ms.soft_constraint_gradient(mask, c, tt, [(0, 0.9 * K)], soft_constraint_weight=1.0)
    assert int(end["max_segment"][0, 0]) == K - 1 and float(end["max_time"][0, 0]) == 1.0
    g = end["grad_times"][0]
    assert float(g[:K - 1].abs().max()) == 0.0 and abs(float(g[K - 1])) <= 1e-12 * max(1.0, float(end["cost"][0]))
    # repeatability
    cons = limits_below(ms, coeffs, t, [1, 2])
    a = ms.soft_constraint_gradient(mask, coeffs, t, cons)
    b = ms.soft_constraint_gradient(mask, coeffs, t, cons)
    for key in a:
        assert torch.equal(a[key], b[key])


# ---- the objective and the driver -----------------------------------------------------------------------------------
CONS = [(1, 3.0), (2, 5.0)]


def test_objective_with_and_without_the_soft_term(ms, oracle, torch_cuda):
    """w_sc = 0 gives free_objective's bits; w_sc > 0 adds w_sc soft last, soft being soft_constraint_cost of the
    recovered candidates."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 24, g)
    B, S = 24, 3
    rng = np.random.default_rng(5)
    cand = (opt[:, None] + torch.from_numpy(rng.normal(size=(B, S) + tuple(opt.shape[1:])) * 0.3).cuda()).contiguous()
    ct = (t[:, None, :] * torch.from_numpy(1.0 + 0.1 * rng.random((B, S, 1))).cuda()).contiguous()
    base, bt = ms.free_objective(mask, fixed, cand, ct, g, w_c=10.0, want_terms=True, **MAP)
    zero, zt = ms.free_objective_soft(mask, fixed, cand, ct, g, w_c=10.0, constraints=CONS, w_sc=0.0, want_terms=True,
                                      **MAP)
    assert torch.equal(zero, base) and torch.equal(zt["Jc"], bt["Jc"]) and torch.equal(zt["Jd"], bt["Jd"])
    obj, terms = ms.free_objective_soft(mask, fixed, cand, ct, g, w_c=10.0, constraints=CONS, w_sc=2.5, want_terms=True,
                                        **MAP)
    assert torch.equal(obj, base + 2.5 * terms["soft"])
    coeffs = ms.coeffs_from_constraints(mask, fixed.repeat_interleave(S, 0), cand.flatten(0, 1), ct.flatten(0, 1))
    assert torch.equal(terms["soft"].flatten(), ms.soft_constraint_cost(coeffs, ct.flatten(0, 1), CONS))


@pytest.mark.parametrize("optimize_times", [False, True])
def test_driver_at_zero_weight_is_the_collision_driver(ms, oracle, torch_cuda, optimize_times):
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 64, g)
    kw = dict(w_c=10.0, optimize_times=optimize_times, iterations=5, **MAP)
    f0, t0, h0, c0 = ms.optimize_free_constraints(mask, fixed, opt, t, g, **kw)
    f1, t1, h1, c1, _ = ms.optimize_free_constraints_soft(mask, fixed, opt, t, g, constraints=CONS, w_sc=0.0, **kw)
    assert torch.equal(f0, f1) and torch.equal(t0, t1) and torch.equal(h0, h1) and torch.equal(c0, c1)


@pytest.mark.parametrize("optimize_times", [False, True])
def test_driver_is_monotone_and_matches_its_glue(ms, oracle, torch_cuda, optimize_times):
    """The history never increases; the torch-glue descent agrees after one iteration (history 1e-12, the same
    accepted steps) and after six (1e-9 relative), as the collision-only driver agrees with its glue; the returned
    maxima are soft_constraint_cost's at the returned state."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 48, g)
    map_kw = {k: v for k, v in MAP.items() if k not in ("origin", "resolution", "min_bound", "max_bound")}
    for iterations in (1, 6):
        kw = dict(w_c=10.0, optimize_times=optimize_times, iterations=iterations)
        f, tt, h, hit, peak = ms.optimize_free_constraints_soft(mask, fixed, opt, t, g, constraints=CONS, w_sc=1.0,
                                                                **kw, **MAP)
        assert bool((h[1:] <= h[:-1]).all()) and bool((h[-1] < h[0]).any())
        gf, gtt, gh, ghit = ms.optimize_free_constraints_soft_reference_glue(mask, fixed, opt, t, g, MAP["origin"],
                                                                             MAP["resolution"], MAP["min_bound"],
                                                                             MAP["max_bound"], constraints=CONS,
                                                                             w_sc=1.0, **kw, **map_kw)
        rel = float(((h - gh).abs() / gh.abs()).max())
        print("glue vs device after %d iterations (optimize_times=%s): %.3e" % (iterations, optimize_times, rel))
        if iterations == 1:
            assert rel <= 1e-12 and torch.equal(hit, ghit)
            assert float((f - gf).abs().max()) <= 1e-14 * float(gf.abs().max())
            assert float((tt - gtt).abs().max()) <= 1e-14 * float(gtt.abs().max())
        else:
            assert rel <= 1e-9
        coeffs = ms.coeffs_from_constraints(mask, fixed, f, tt)
        assert torch.equal(peak, ms.soft_constraint_cost(coeffs, tt, CONS, want_terms=True)[1]["max_value"])


def test_driver_replays_from_a_cuda_graph(ms, oracle, torch_cuda):
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 64, g)
    B, K = 64, 10
    f_buf, t_buf = opt.clone(), t.clone()
    hist = torch.empty((5, B), dtype=torch.float64, device="cuda")
    hit = torch.empty((B,), dtype=torch.int32, device="cuda")
    peak = torch.empty((B, 2), dtype=torch.float64, device="cuda")
    lib = ms.capi.load()
    host, margs = ms.api._collision_map(g, MAP["origin"], MAP["resolution"], MAP["min_bound"], MAP["max_bound"],
                                        MAP["dt"], MAP["map_resolution"], MAP["epsilon"], MAP["robot_radius"],
                                        MAP["coll_pot_multiplier"], True, MAP["oob_value"])
    shost, sargs = ms.api._soft_args(CONS, 100.0, 1e12, False)
    m = np.ascontiguousarray(mask, np.uint8)

    def enqueue():
        ms.capi.check(lib.minsnap_optimize_free_constraints_soft(B, K, 3, 10, 4, ms.api._hptr(m), ms.api._dptr(fixed),
                                                                 ms.api._dptr(f_buf), ms.api._dptr(t_buf), 1, 0.1, 10.0,
                                                                 1.0, *margs, *sargs, 1.0, 4, 8, 0.5, 0.1, 1e-3,
                                                                 ms.api._dptr(hist), ms.api._dptr(hit),
                                                                 ms.api._dptr(peak), ms.api._stream()),
                      "minsnap_optimize_free_constraints_soft")
    enqueue()
    torch.cuda.synchronize()
    first, first_free, first_peak = hist.clone(), f_buf.clone(), peak.clone()
    f_buf.copy_(opt)
    t_buf.copy_(t)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        enqueue()
    f_buf.copy_(opt)
    t_buf.copy_(t)
    hist.zero_()
    peak.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(hist, first) and torch.equal(f_buf, first_free) and torch.equal(peak, first_peak)
    assert bool((first[-1] < first[0]).any())


def test_driver_brings_more_trajectories_within_the_limits(ms, oracle, torch_cuda):
    """256 trajectories crossing the sphere, limits at 0.9 of the batch's median maxima, 20 iterations: more end within
    1.05x of both limits than with the collision-only driver at the same settings."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 256, g)
    coeffs = ms.coeffs_from_constraints(mask, fixed, opt, t)
    cons = limits_below(ms, coeffs, t, [1, 2])
    lim = torch.tensor([v for _, v in cons], dtype=torch.float64, device="cuda")
    kw = dict(w_c=10.0, iterations=20, **MAP)
    f0, t0, _, hit0 = ms.optimize_free_constraints(mask, fixed, opt, t, g, **kw)
    peak0 = ms.soft_constraint_cost(ms.coeffs_from_constraints(mask, fixed, f0, t0), t0, cons,
                                    want_terms=True)[1]["max_value"]
    f1, t1, _, hit1, peak1 = ms.optimize_free_constraints_soft(mask, fixed, opt, t, g, constraints=cons, w_sc=1.0, **kw)
    within0 = float((peak0 <= 1.05 * lim).all(1).double().mean())
    within1 = float((peak1 <= 1.05 * lim).all(1).double().mean())
    free0, free1 = float((hit0 == 0).double().mean()), float((hit1 == 0).double().mean())
    print("within 1.05x: collision-only %.3f, with soft term %.3f; collision-free %.3f / %.3f"
          % (within0, within1, free0, free1))
    assert within1 > within0
