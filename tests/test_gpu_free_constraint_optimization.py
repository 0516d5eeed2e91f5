"""GPU tests of the free-constraint problem: J = w_d J_d + w_c J_c + w_t sum(T) over the free derivatives d_p (and
the segment times), the objective of the reference's nonlinear optimiser.

Parity is claimed for the objective and every gradient it is built from, against the oracle's restatement:
  J_d = sum_dim d^T R d and dJ_d/dd_p = 2 (R_pf d_f + R_pp d_p)  with R from Oracle.solve(..., want_R=True)
        (ref getCostAndGradientDerivative, NL.i:1452-1521);
  J_c = oracle_py.collision_cost (ref getCostAndGradientCollision, NL.i:1523-1709).
The driver (minsnap_optimize_free_constraints) has no reference counterpart (NLopt is absent); it is checked for
monotone descent, for its fixed point on the convex problem, for what it does near an obstacle, and against the same
descent written as torch glue around the C-ABI calls.
"""
import numpy as np
import pytest

from helpers import COST_TOL, compact_fixed, random_batch, standard_mask, vertex_values
from test_collision_cost import ORIGIN, RES, field

pytestmark = pytest.mark.gpu

MAP = dict(origin=ORIGIN, resolution=RES, min_bound=[-10.0, -20.0, -10.0], max_bound=[10.0, 20.0, 10.0], dt=0.1,
           map_resolution=RES, epsilon=0.5, robot_radius=0.5, coll_pot_multiplier=1.5, oob_value=10.0)   # outside: free space


def general_mask(K, N):
    """A velocity-constrained interior vertex, a constrained higher derivative at another, and free derivatives at
    both ends."""
    h = N // 2
    m = standard_mask(K, N).copy()
    m[2, 1] = 1
    m[3, h - 1] = 1
    m[K, h - 1] = 0
    m[0, 1] = 0
    return m


def problem(oracle, oracle_ld, B, K, D, N, mask, seed):
    """Vertex values (non-zero fixed higher derivatives), times and the oracle's solve with R for every b.  R comes
    from the long-double oracle: in double, its A^-T Q A^-1 loses about 1e-8 of J_d to cancellation at N = 12."""
    h = N // 2
    deriv = min(4, h - 1)
    lo, hi = (-10.0 * np.ones(D), 10.0 * np.ones(D))
    rng = np.random.default_rng(seed)
    out = []
    for b in range(B):
        pos = oracle.create_random_positions(K, lo, hi, seed + b)
        times = oracle.estimate_segment_times(pos, 3.0, 5.0)
        vv = vertex_values(pos, N)
        vv = vv + mask[:, :, None] * (np.arange(h) > 0)[None, :, None] * rng.normal(size=vv.shape) * 0.3
        sol = oracle_ld.solve(N, K, D, deriv, mask, vv, np.asarray(times, np.float64), want_R=True)
        out.append((np.asarray(times, np.float64), np.asarray(compact_fixed(mask, vv), np.float64), sol))
    return deriv, out


@pytest.mark.parametrize("N", [6, 8, 10, 12])
@pytest.mark.parametrize("D", [1, 2, 3])
@pytest.mark.parametrize("mask_kind", ["standard", "general"])
def test_derivative_gradient_matches_oracle(ms, oracle, oracle_ld, torch_cuda, N, D, mask_kind):
    """J_d within COST_TOL of 2 computeCost and of d^T R d; the gradient within 1e-9 of its largest component and
    diag(R_pp) entry by entry within 1e-9 relative, against the long-double oracle (measured at most 1.0e-11 and
    3.5e-11, both at N = 12; 6e-14 and 8e-14 at N = 10) -- tighter than the 1e-6 of the time gradient, whose bar
    comes from the double oracle's A^-T Q A^-1; the coefficients bit-identical to minsnap_coeffs_from_constraints."""
    torch = torch_cuda
    B, K = 37, 6                      # a ragged batch: not a multiple of the warps per block
    mask = standard_mask(K, N) if mask_kind == "standard" else general_mask(K, N)
    deriv, rows = problem(oracle, oracle_ld, B, K, D, N, mask, 400 + N + D)
    rng = np.random.default_rng(N * 10 + D)
    times = np.stack([r[0] for r in rows])
    fixed = np.stack([r[1] for r in rows])
    free = np.stack([np.asarray(r[2]["d_free"], np.float64).T for r in rows])     # [B][n_free][D]
    free = free + rng.normal(size=free.shape) * 0.2 * (np.abs(free).max() + 1.0)   # away from the optimum
    t, f, p = (torch.from_numpy(a).cuda() for a in (times, fixed, free))
    out = ms.derivative_gradient(mask, f, p, t, N=N, derivative=deriv, want_coeffs=True, want_diag=True)
    ref_coeffs = ms.coeffs_from_constraints(mask, f, p, t, N=N)
    assert torch.equal(out["coeffs"], ref_coeffs)
    jd, grad, diag = out["Jd"].cpu().numpy(), out["gradient"].cpu().numpy(), out["diag"].cpu().numpy()
    col, n_fixed, n_free = oracle.reorder(N, K, mask)
    worst_g = worst_diag = 0.0
    for b in range(B):
        R = np.asarray(rows[b][2]["R"], np.longdouble)
        d_all = np.concatenate([fixed[b].T, free[b].T], axis=1)                     # [D][n_all]
        dl = d_all.astype(np.longdouble)
        want_g = np.stack([2.0 * (R[n_fixed:] @ dl[k]) for k in range(D)], axis=1).astype(np.float64)
        worst_g = max(worst_g, float(np.abs(grad[b] - want_g).max() / np.abs(want_g).max()))
        assert np.abs(grad[b] - want_g).max() <= 1e-9 * np.abs(want_g).max(), (b, np.abs(grad[b] - want_g).max())
        want_jd = float(sum(dl[k] @ R @ dl[k] for k in range(D)))
        assert abs(jd[b] - want_jd) <= COST_TOL * want_jd
        coeffs = oracle_ld.coeffs_from_constraints(N, K, D, col, d_all, times[b])
        cost = float(oracle_ld.compute_cost(N, K, D, deriv, coeffs, times[b]))
        assert abs(jd[b] - 2.0 * cost) <= COST_TOL * 2.0 * cost
        want_diag = np.diag(R)[n_fixed:].astype(np.float64)
        worst_diag = max(worst_diag, float((np.abs(diag[b] - want_diag) / np.abs(want_diag)).max()))
        assert np.all(np.abs(diag[b] - want_diag) <= 1e-9 * np.abs(want_diag)), (b, diag[b], want_diag)
    print("N=%d D=%d %s: gradient err %.3e of max, diag err %.3e relative" % (N, D, mask_kind, worst_g, worst_diag))
    # the host entry point returns the same bits
    host = ms.derivative_gradient_host(mask, fixed, free, times, N=N, derivative=deriv)
    assert np.array_equal(host["gradient"], grad) and np.array_equal(host["Jd"], jd)
    assert np.array_equal(host["diag"], diag)


def test_derivative_gradient_is_the_derivative_of_jd(ms, oracle, torch_cuda):
    """J_d is quadratic in d_p: a central difference of J_d in every free component equals the gradient up to
    rounding (measured 6.3e-13 of the largest component; bound 1e-10).  At the QP optimum the gradient is rounding
    (measured 4.7e-16 of 2 |R_pf d_f|, the gradient at d_p = 0; bound 1e-12)."""
    torch = torch_cuda
    K, N, D = 10, 10, 3
    mask = standard_mask(K)
    pos, times = random_batch(oracle, 8, K)
    fixed = np.stack([compact_fixed(mask, vertex_values(p)) for p in pos])
    t, f = torch.from_numpy(times).cuda(), torch.from_numpy(fixed).cuda()
    opt = ms.solve(mask, f, t)["free_values"]
    g_opt = ms.derivative_gradient(mask, f, opt, t)["gradient"]
    g_zero = ms.derivative_gradient(mask, f, torch.zeros_like(opt), t)["gradient"]   # 2 R_pf d_f
    ratio = (g_opt.abs().amax((1, 2)) / g_zero.abs().amax((1, 2))).max().item()
    print("free-constraint gradient at the QP optimum / 2|R_pf d_f|: %.3e" % ratio)
    assert ratio <= 1e-12
    # central differences for one perturbed trajectory, every component at once
    b, h = 3, 1e-3
    base = opt[b] + torch.from_numpy(np.random.default_rng(4).normal(size=tuple(opt[b].shape))).cuda() * 0.5
    n = base.numel()
    eye = torch.eye(n, dtype=torch.float64, device="cuda").reshape(n, *base.shape)
    pert = torch.cat([base[None] + h * eye, base[None] - h * eye]).contiguous()
    rep = lambda a: a[b:b + 1].expand(2 * n, *a.shape[1:]).contiguous()
    jd = ms.derivative_gradient(mask, rep(f), pert, rep(t))["Jd"]
    fd = ((jd[:n] - jd[n:]) / (2 * h)).reshape(base.shape)
    g = ms.derivative_gradient(mask, f[b:b + 1], base[None].contiguous(), t[b:b + 1])["gradient"][0]
    err = ((fd - g).abs().max() / g.abs().max()).item()
    print("central difference vs gradient: %.3e" % err)
    assert err <= 1e-10


@pytest.mark.parametrize("name", ["sphere", "box"])
@pytest.mark.parametrize("continuous", [True, False])
def test_free_objective_matches_oracle(ms, oracle, torch_cuda, name, continuous):
    """w_d 2 computeCost + w_c collision_cost + w_t sum(T) from the oracle, within 1e-8 relative; the terms and the
    collision flags as well."""
    from oracle import oracle_py
    torch = torch_cuda
    B, S, K, N, D = 16, 3, 10, 10, 3
    w_d, w_c, w_t = 0.1, 10.0, 1.0
    mask = standard_mask(K)
    pos, times = random_batch(oracle, B, K, seed=31)
    fixed = np.stack([compact_fixed(mask, vertex_values(p)) for p in pos])
    rng = np.random.default_rng(2)
    opt = ms.solve(mask, torch.from_numpy(fixed).cuda(), torch.from_numpy(times).cuda())["free_values"].cpu().numpy()
    free = opt[:, None] + rng.normal(size=(B, S) + opt.shape[1:]) * np.array([0.0, 0.3, 0.6])[None, :, None, None]
    cand_t = times[:, None, :] * np.array([1.0, 0.9, 1.2])[None, :, None]
    g = field(name)
    kw = dict(MAP, use_continuous_distance=continuous)
    obj, terms = ms.free_objective(mask, torch.from_numpy(fixed).cuda(), torch.from_numpy(free).cuda(),
                                   torch.from_numpy(cand_t).cuda(), torch.from_numpy(g).cuda(), w_c=w_c, w_d=w_d, w_t=w_t,
                                   want_terms=True, **kw)
    obj, jd, jc, hit = (a.cpu().numpy() for a in (obj, terms["Jd"], terms["Jc"], terms["is_collision"]))
    col, n_fixed, _ = oracle.reorder(N, K, mask)
    n_hit = 0
    for b in range(B):
        for s in range(S):
            d_all = np.concatenate([fixed[b].T, free[b, s].T], axis=1)
            coeffs = np.asarray(oracle.coeffs_from_constraints(N, K, D, col, d_all, cand_t[b, s]), np.float64)
            want_jd = 2.0 * float(oracle.compute_cost(N, K, D, 4, coeffs, cand_t[b, s]))
            want_jc, want_hit, _ = oracle_py.collision_cost(coeffs, cand_t[b, s], g, **kw)
            total = 0.0
            for x in cand_t[b, s]:
                total += x
            want = w_d * want_jd + w_c * want_jc + w_t * total
            assert abs(obj[b, s] - want) <= 1e-8 * abs(want), (b, s, obj[b, s], want)
            assert abs(jd[b, s] - want_jd) <= COST_TOL * want_jd
            assert abs(jc[b, s] - want_jc) <= 1e-8 * max(abs(want_jc), 1e-3)
            assert hit[b, s] == want_hit
            n_hit += want_hit
    assert n_hit > 0


# ---- the driver ------------------------------------------------------------------------------------------------
def standard_problem(ms, oracle, torch, B, K=10, seed=12345):
    mask = standard_mask(K)
    pos, times = random_batch(oracle, B, K, seed=seed)
    fixed = torch.from_numpy(np.stack([compact_fixed(mask, vertex_values(p)) for p in pos])).cuda()
    t = torch.from_numpy(times).cuda()
    opt = ms.solve(mask, fixed, t)["free_values"]
    return mask, fixed, t, opt


def colliding_problem(ms, oracle, torch, B, g):
    """B trajectories whose min-snap path crosses the obstacle of the field g."""
    mask = standard_mask(10)
    pos, times = random_batch(oracle, 8 * B, 10, seed=777)
    p, t = torch.from_numpy(pos).cuda(), torch.from_numpy(times).cuda()
    coeffs = ms.solve_standard(p, t, want_status=False)["coeffs"]
    hit = ms.collision_cost(coeffs, t, g, **MAP)["is_collision"].bool()
    idx = torch.nonzero(hit).flatten()[:B]
    assert idx.numel() == B
    fixed = torch.from_numpy(np.stack([compact_fixed(mask, vertex_values(x)) for x in pos])).cuda()[idx].contiguous()
    t = t[idx].contiguous()
    return mask, fixed, t, ms.solve(mask, fixed, t)["free_values"]


def test_descent_is_monotone_and_reports_the_objective(ms, oracle, torch_cuda):
    """The history never increases, and its last row is free_objective at the returned (d_p, T)."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 64, g)
    for optimize_times in (False, True):
        free, times, hist, hit = ms.optimize_free_constraints(mask, fixed, opt, t, g, w_c=10.0, iterations=12,
                                                              optimize_times=optimize_times, **MAP)
        assert bool((hist[1:] <= hist[:-1]).all())
        obj, terms = ms.free_objective(mask, fixed, free[:, None].contiguous(), times[:, None].contiguous(), g, w_c=10.0,
                                       want_terms=True, **MAP)
        assert float(((obj[:, 0] - hist[-1]).abs() / hist[-1].abs()).max()) <= 1e-12
        assert torch.equal(terms["is_collision"][:, 0], hit)
        if not optimize_times:
            assert torch.equal(times, t)
        assert float(times.min()) >= 0.1


def test_convex_case_fixed_point_and_contraction(ms, oracle, torch_cuda):
    """w_c = 0, fixed times and a field that is everywhere farther than robot_radius + epsilon (J_c = 0 exactly):
    the problem is the QP.  Started at its optimum, the history stays constant to rounding (measured 7.8e-15
    relative; bound 1e-13) and d_p moves by rounding only (measured 5.4e-15 of |d_p|; bound 1e-12).  Started away
    from it, J_d decreases and d_p approaches the solve's in the metric of the problem: the distance
    |d_p - d_p*|_R = sqrt(J_d(d_p) - J_d(d_p*)) shrinks for every trajectory (measured median ratio of the squares
    2.8e-3 after 20 iterations).  The Euclidean distance mixes the units of velocity, acceleration, jerk and snap,
    which the Jacobi-scaled step does not: it shrinks for the batch (summed), not for every trajectory (measured
    median ratio 0.56, largest 1.18)."""
    torch = torch_cuda
    B = 128
    mask, fixed, t, opt = standard_problem(ms, oracle, torch, B)
    far = torch.full((48, 88, 48), 5.0, dtype=torch.float64, device="cuda")
    kw = dict(MAP, oob_value=5.0)
    free, times, hist, hit = ms.optimize_free_constraints(mask, fixed, opt, t, far, w_c=0.0, iterations=10, **kw)
    assert int(hit.sum()) == 0
    drift = ((hist - hist[0]).abs() / hist[0]).max().item()
    move = ((free - opt).abs().amax((1, 2)) / opt.abs().amax((1, 2))).max().item()
    print("at the optimum: history drift %.3e, d_p move %.3e" % (drift, move))
    assert drift <= 1e-13 and move <= 1e-12
    rng = np.random.default_rng(11)
    start = opt + torch.from_numpy(rng.normal(size=tuple(opt.shape))).cuda() * 0.5
    free, _, hist, _ = ms.optimize_free_constraints(mask, fixed, start, t, far, w_c=0.0, iterations=20, **kw)
    jd0 = ms.derivative_gradient(mask, fixed, start, t)["Jd"]
    jd1 = ms.derivative_gradient(mask, fixed, free, t)["Jd"]
    jd_opt = ms.derivative_gradient(mask, fixed, opt, t)["Jd"]
    assert bool((jd1 < jd0).all())
    excess = (jd1 - jd_opt) / (jd0 - jd_opt)          # squared R-metric distance to the optimum, after / before
    d0 = (start - opt).flatten(1).norm(dim=1)
    d1 = (free - opt).flatten(1).norm(dim=1)
    print("convex: excess J_d ratio median %.3e max %.3e, Euclidean distance ratio median %.3e max %.3e, summed %.3e"
          % (excess.median().item(), excess.max().item(), (d1 / d0).median().item(), (d1 / d0).max().item(),
             (d1.sum() / d0.sum()).item()))
    assert bool((excess < 1.0).all())
    assert float(d1.sum()) < float(d0.sum())
    # the objective is w_d J_d + w_t sum(T) here: the history is 0.1 J_d + sum(T)
    assert float(((hist[-1] - (0.1 * jd1 + t.sum(1))).abs() / hist[-1]).max()) <= 1e-12


@pytest.mark.parametrize("optimize_times", [False, True])
def test_obstacle_case_moves_trajectories_out_of_collision(ms, oracle, torch_cuda, optimize_times):
    """256 trajectories whose min-snap path crosses the sphere: the mean collision cost and the number of
    trajectories in collision both drop.  Measured on a B200 (20 iterations, 8 steps, w_d = 0.1, w_c = 10,
    w_t = 1): mean J_c 10.03 -> 3.15 and 152 of the 256 (59.4 %) end collision-free with the times fixed;
    10.03 -> 3.17 and 155 (60.5 %) with the times optimised too."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 256, g)
    free, times, hist, hit = ms.optimize_free_constraints(mask, fixed, opt, t, g, w_c=10.0, iterations=20,
                                                          optimize_times=optimize_times, **MAP)
    before = ms.free_objective(mask, fixed, opt[:, None].contiguous(), t[:, None].contiguous(), g, w_c=10.0,
                               want_terms=True, **MAP)[1]
    after = ms.free_objective(mask, fixed, free[:, None].contiguous(), times[:, None].contiguous(), g, w_c=10.0,
                              want_terms=True, **MAP)[1]
    jc0, jc1 = before["Jc"].mean().item(), after["Jc"].mean().item()
    n0, n1 = int(before["is_collision"].sum()), int(after["is_collision"].sum())
    print("obstacle (optimize_times=%s): mean J_c %.4g -> %.4g, in collision %d -> %d of 256 (%.1f%% collision-free)"
          % (optimize_times, jc0, jc1, n0, n1, 100.0 * (256 - n1) / 256))
    assert n0 >= 230 and torch.equal(after["is_collision"][:, 0], hit)
    assert jc1 < jc0 and n1 < n0
    assert bool((hist[1:] <= hist[:-1]).all())


@pytest.mark.parametrize("optimize_times", [False, True])
def test_device_resident_descent_matches_the_glue_version(ms, oracle, torch_cuda, optimize_times):
    """minsnap_optimize_free_constraints against the same descent in torch glue around the C-ABI calls: after one
    iteration the same history (1e-12) and the same accepted steps; after ten, agreement to 1e-9 relative (measured
    1.2e-12 with the times fixed, 3.9e-11 with them optimised: the time ladder's last bits differ, as in the
    time-only driver)."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 96, g)
    kw = dict(w_c=10.0, optimize_times=optimize_times, **MAP)
    f_dev, t_dev, h_dev, c_dev = ms.optimize_free_constraints(mask, fixed, opt, t, g, iterations=1, **kw)
    f_ref, t_ref, h_ref, c_ref = ms.api.optimize_free_constraints_reference_glue(mask, fixed, opt, t, g, iterations=1, **kw)
    assert h_dev.shape == h_ref.shape == (2, 96)
    assert float(((h_dev - h_ref).abs() / h_ref.abs()).max()) <= 1e-12
    assert bool((h_dev[1] < h_dev[0]).any())                     # steps were taken
    assert float((f_dev - f_ref).abs().max()) <= 1e-14 * float(f_ref.abs().max())
    assert float((t_dev - t_ref).abs().max()) <= 1e-14 * float(t_ref.abs().max())
    assert torch.equal(c_dev, c_ref)
    f_dev, t_dev, h_dev, _ = ms.optimize_free_constraints(mask, fixed, opt, t, g, iterations=10, **kw)
    f_ref, t_ref, h_ref, _ = ms.api.optimize_free_constraints_reference_glue(mask, fixed, opt, t, g, iterations=10, **kw)
    rel = float(((h_dev - h_ref).abs() / h_ref.abs()).max())
    print("glue vs device after 10 iterations (optimize_times=%s): %.3e" % (optimize_times, rel))
    assert rel <= 1e-9


def test_driver_replays_from_a_cuda_graph(ms, oracle, torch_cuda):
    """The loop holds no host-side decision and the mask travels by value: the driver captured into a CUDA graph and
    replayed gives the history of a direct run, bit for bit."""
    torch = torch_cuda
    g = torch.from_numpy(field("sphere")).cuda()
    mask, fixed, t, opt = colliding_problem(ms, oracle, torch, 64, g)
    B, K = 64, 10
    f_buf, t_buf = opt.clone(), t.clone()
    hist = torch.empty((5, B), dtype=torch.float64, device="cuda")
    hit = torch.empty((B,), dtype=torch.int32, device="cuda")
    lib = ms.capi.load()
    host, margs = ms.api._collision_map(g, MAP["origin"], MAP["resolution"], MAP["min_bound"], MAP["max_bound"],
                                        MAP["dt"], MAP["map_resolution"], MAP["epsilon"], MAP["robot_radius"],
                                        MAP["coll_pot_multiplier"], True, MAP["oob_value"])
    m = np.ascontiguousarray(mask, np.uint8)

    def enqueue():
        ms.capi.check(lib.minsnap_optimize_free_constraints(B, K, 3, 10, 4, ms.api._hptr(m), ms.api._dptr(fixed),
                                                            ms.api._dptr(f_buf), ms.api._dptr(t_buf), 1, 0.1, 10.0, 1.0,
                                                            *margs, 4, 8, 0.5, 0.1, 1e-3, ms.api._dptr(hist),
                                                            ms.api._dptr(hit), ms.api._stream()),
                      "minsnap_optimize_free_constraints")
    enqueue()
    torch.cuda.synchronize()
    first, first_free, first_hit = hist.clone(), f_buf.clone(), hit.clone()
    f_buf.copy_(opt)
    t_buf.copy_(t)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        enqueue()
    f_buf.copy_(opt)
    t_buf.copy_(t)
    hist.zero_()
    graph.replay()
    torch.cuda.synchronize()
    assert torch.equal(hist, first) and torch.equal(f_buf, first_free) and torch.equal(hit, first_hit)
    assert bool((first[-1] < first[0]).any())
