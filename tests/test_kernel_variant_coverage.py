"""Every launch variant of the sampling, evaluate_range, cost and cost-sweep launchers has a case in
tests/test_gpu_kernel_variants.py.  The variant of each case comes from that file's restatement of the launcher's
choice, so a threshold moved in a .cu file (and mirrored there) that leaves some variant without a case fails here,
on a machine without a GPU.  The same holds for the collision walk and the gradient instantiation of the general
kernel in tests/test_gpu_collision_walk.py, whose hand-built and map cases are also checked here to reach the edges
they are built for, and for the kernels behind minsnap_solve_standard in tests/test_gpu_standard_variants.py."""
import numpy as np

import test_gpu_collision_walk as W
import test_gpu_kernel_variants as V
import test_gpu_standard_variants as S
from oracle import oracle_py
from test_collision_cost import field

SMS = V.B200_SMS


def test_every_sampling_variant_has_a_case():
    have = {(args[0], tag) for args, tag in V.SAMPLE_CASES}
    kernels = {tag[0] for _, tag in have}
    assert kernels == {"fast", "staged", "unstaged"}
    for N in V.ORDERS:
        for nd in range(1, 6):
            assert any(n == N and tag[:2] == ("fast", nd) for n, tag in have), ("fast", N, nd)
        for kernel in ("staged", "unstaged"):
            assert any(n == N and tag[0] == kernel for n, tag in have), (kernel, N)
    for kernel in kernels:
        for grid in ("chunked", "per_trajectory"):
            assert any(tag[0] == kernel and tag[2] == grid for _, tag in have), (kernel, grid)
    assert {tag[3] for _, tag in have if tag[0] == "fast"} == {"vector", "mixed", "scalar"}
    # rows k >= N on the fast and the staged kernel; find_segment's linear scan and its binary search (K > 16)
    cases = [(args, tag) for args, tag in V.SAMPLE_CASES]
    assert any(a[3] > a[0] and t[0] == "fast" for a, t in cases)
    assert {a[0] for a, t in cases if a[3] > a[0] and t[0] == "staged"} >= {10, 12}
    assert any(a[1] <= 16 for a, _ in cases) and any(a[1] > 16 for a, _ in cases)
    assert {a[2] for a, _ in cases} >= {1, 2, 3, 4}
    assert {a[5] for a, _ in cases} >= {1, 31, 32, 33, 1000}


def test_every_sweep_variant_has_a_case():
    tags = {(tag, args[4]) for args, tag in V.SWEEP_CASES}
    assert tags == {(v, ends) for v in ("direct", "global_slots") for ends in (False, True)}
    direct = [args for args, tag in V.SWEEP_CASES if tag == "direct"]
    assert {K for K, _, _, _, ends in direct if ends} >= {1, 2, 3}    # the boundary-coupling paths
    assert {D for _, D, _, _, _ in direct} == {1, 2, 3}
    problems = {S * B for _, _, S, B, _ in direct}
    assert any(n % 16 for n in problems) and any(n % 16 == 0 for n in problems) and min(problems) < 16
    assert all(V.sweep_variant(5, D, N, delta) == "generic" for N, delta, D in V.SWEEP_GENERIC_CASES)
    for D in (1, 2, 3):
        K = V.sweep_k_limit(D)
        assert V.sweep_variant(K, D) == "global_slots" and V.sweep_variant(K + 1, D) == "generic"
    # the input-staging limit the long-chain tests rely on: ~440 at D = 3, beyond 513 at D < 3
    assert 440 <= V.sweep_k_limit(3) < 513 and V.sweep_k_limit(2) > 513 and V.sweep_k_limit(1) > 513


def test_grid_stride_cases_loop():
    assert V.evaluate_range_loops(V.EVALUATE_RANGE_LOOP_B, SMS)
    assert V.cost_loops(V.COST_LOOP_B, SMS)
    assert V.sweep_variant(V.SWEEP_LOOP_K, V.SWEEP_LOOP_D) == "direct"
    assert V.sweep_loops(V.SWEEP_LOOP_B * V.SWEEP_LOOP_S, V.SWEEP_LOOP_K, V.SWEEP_LOOP_D, SMS)
    assert not V.evaluate_range_loops(64 * SMS, SMS) and not V.cost_loops(128 * SMS, SMS)


# ---- the collision walk and the gradient kernel (tests/test_gpu_collision_walk.py) ----------------------------------
def test_gradient_kernel_warp_steps_have_cases():
    """Every warps-per-CTA step of the general kernel's gradient instantiation has a case at its first and its last
    K for both masks, the first refused K has a case, and D = 1 has one past its last step."""
    steps, refused = W.warp_steps(3, "standard")
    assert steps == {8: (1, 21), 4: (22, 42), 2: (43, 82), 1: (83, 365)} and refused == 366
    steps_d1, refused_d1 = W.warp_steps(1, "standard")
    assert [steps_d1[w][0] for w in (4, 2, 1)] == [25, 49, 96] and refused_d1 == 419
    for kind in ("standard", "general"):
        steps, refused = W.warp_steps(3, kind)
        have = {args[0]: tag for args, tag in W.GRADIENT_CASES if args[1:] == (3, kind)}
        assert set(steps) == {8, 4, 2, 1}
        for warps, (first, last) in steps.items():
            assert have.get(first) == warps and have.get(last) == warps, (kind, warps, first, last)
        assert (refused, 3, kind) in W.ERROR_CASES
    for K, D, kind in W.ERROR_CASES:
        assert W.gradient_variant(K, D, kind) is None and W.gradient_variant(K - 1, D, kind) == 1
    assert any(args[1] == 1 and args[0] > steps_d1[1][0] and tag == 1 for args, tag in W.GRADIENT_CASES)
    assert any(args[0] == 1 for args, _ in W.GRADIENT_CASES) and 1 in W.WALK_K_CASES


def test_collision_walk_and_gradient_loop_cases_loop():
    """The batch of every grid-stride case loops on 148 SMs, and the chunks it is compared with do not."""
    assert W.walk_loops(W.WALK_LOOP_B, SMS) and not W.walk_loops(W.WALK_CHUNK, SMS)
    looped = set()
    for K, B, chunk in W.GRADIENT_LOOP_CASES:
        warps = W.gradient_variant(K, 3, "standard")
        assert W.general_loops(B, warps, SMS) and not W.general_loops(chunk, warps, SMS)
        looped.add(warps)
    assert looped == {8, 1}
    n, warps = W.FREE_B * W.FREE_S, W.gradient_variant(W.FREE_K, 3, "standard")
    assert W.general_loops(n, warps, SMS) and W.walk_loops(n, SMS)
    chunk = W.FREE_CHUNK * W.FREE_S
    assert not W.general_loops(chunk, warps, SMS) and not W.walk_loops(chunk, SMS)


def test_walk_boundary_cases_reach_their_edges():
    """The hand-built walks do what they are built for, on a Python replay of the walk that agrees with the oracle
    on the number of charged samples."""
    g = field("sphere")
    for name, (rows, row_times, dt, limit, _) in W.BOUNDARY_CASES.items():
        kw = dict(W.MAP1, dt=dt, map_resolution=limit, use_continuous_distance=True)
        for c, times in zip(rows, row_times):
            charged, entry, counts, margin = W.replay_walk(c, times, dt, limit)
            assert oracle_py.collision_cost(c, times, g, **kw)[2] == len(charged), name
            assert margin > 1e-6 and max(counts) < 1e5, (name, margin)
        charged, entry, counts, margin = W.replay_walk(rows[0], row_times[0], dt, limit)
        times = row_times[0]
        cost, hit, _ = oracle_py.collision_cost(rows[0], times, g, **kw)
        assert cost > 0.1 and hit, name                        # the walk crosses the obstacle
        if name == "lane31":     # on and one ulp below 32 dt: a full chunk, then one with no valid sample; one ulp
            assert times[0] == W.repeated(dt, 32) and times[1] < times[0] < times[2]     # above: a 33rd sample
            assert counts == [32, 32, 33, 64]
        elif name == "short_and_zero":
            assert counts[1] == 0 and counts[3] == 1 and times[3] < dt
            assert 0.0 <= entry[1] < dt and entry[2] < 0.0     # the zero-length segment leaves time_sum negative
        elif name == "many_chunks":
            assert counts[0] > 60 * 32
        else:
            slow = [s for s in charged if s[0] == 1 and s[1] == 0.0]
            assert len(slow) == 1 and np.linalg.norm(slow[0][4]) < 1e-6 and slow[0][2] > 0.5
            cost, _, hit = oracle_py.collision_potential(slow[0][3], g, **W.potential_kw(kw))
            assert hit and cost > 1.0


def test_walk_map_cases_reach_their_edges(oracle):
    """The charged samples of the map cases reach all three branches of cost_potential and cells outside the grid,
    and in continuous mode a centre whose eight-cell stencil falls off the grid (the discrete fallback)."""
    g = W.grid2_field()
    assert g.shape == W.GRID2_DIMS and len(set(W.GRID2_DIMS)) == 3 and len(set(W.GRID2_ORIGIN)) == 3
    for case in W.MAP_CASES:
        for continuous in (True, False):
            coeffs, times, kw = W.map_case(oracle, case, continuous)
            seen = W.map_edges(coeffs, times, g, kw)
            assert min(seen["collision"], seen["band"], seen["free"], seen["outside"]) > 0, (case, seen)
            assert seen["stencil_off"] > 0 or not continuous, (case, seen)
    mr = {W.walk_kw(dict(resolution=W.GRID2_RES, **kw))["map_resolution"] for kw in W.MAP_CASES.values()}
    assert min(mr) < W.GRID2_RES < max(mr)
    assert {kw.get("robot_radius", 0.5) for kw in W.MAP_CASES.values()} >= {0.0}
    assert {kw["oob_value"] < 0.5 for kw in W.MAP_CASES.values()} == {True, False}


def test_walk_chain_cases_reach_the_last_free_vertex(oracle):
    """At every K > 1 the oracle's gradient is non-zero in the columns of vertex K - 1, the last free one."""
    g = field(W.CHAIN_FIELD)
    kw = W.chain_kw()
    for K in W.WALK_K_CASES:
        if K == 1:
            continue
        coeffs, times = W.chain_case(oracle, K)
        col, n_fixed, n_free = oracle.reorder(10, K, W.standard_mask(K))
        last = max(np.abs(oracle_py.collision_cost_gradient(coeffs[b], times[b], col, n_fixed, n_free, sdf=g, **kw)[1]
                          [-4:]).max() for b in range(len(times)))
        assert last > 0, K


# ---- minsnap_solve_standard (tests/test_gpu_standard_variants.py) ------------------------------------------------
def _standard_variants():
    routes = S.routes_of(S.STD_CASES)
    return [(c, r, S.variant(c, r)) for c, r in zip(S.STD_CASES, routes)]


def test_every_standard_route_variant_has_a_case():
    """Each case reaches the route it is written for (the route binary), and every variant has a case: the 24 tm
    instantiations through solve_standard, every tm grid mode for each D, pair (D, kCost) and its grid-stride loop,
    both pair_long scratch branches, every bcr thread step at D = 3 and a looping bcr case for each D, every chunk
    length for each D on one and on two ranges, and the general route at N != 10, derivative != 4 and D >= 4."""
    cases = _standard_variants()
    for c, r, _ in cases:
        assert r == (c.forced or r) and r != "unsupported", (c, r)
    tags = {}
    for c, r, v in cases:
        tags.setdefault(r, set()).add(v)
    assert all(r == "tm" for c, r, _ in cases if c in S.TM_CASES)
    assert {v[:4] for v in tags["tm"]} == {(D, cost, ex, odd) for D in (1, 2, 3) for cost in (False, True)
                                           for ex in (False, True) for odd in (False, True)}
    for inst in {v[:4] for v in tags["tm"]}:     # two time modes for every instantiation
        assert len({c.times for c, r, v in cases if r == "tm" and v[:4] == inst}) >= 2, inst
    modes = ("one batch per warp", "two batches, even waves", "two batches, odd waves")
    assert {(v[0], v[4]) for v in tags["tm"]} == {(D, m) for D in (1, 2, 3) for m in modes}
    assert any(r == "tm" and v[0] == 1 and v[4] != modes[0] and S.tm_ctas(c.K, 1, False, False) == 3
               for c, r, v in cases)
    assert {v[:2] for v in tags["pair"]} == {(D, cost) for D in (1, 2, 3) for cost in (False, True)}
    assert any(v[2] for v in tags["pair"])
    assert {v[1:] for v in tags["pair_long"]} >= {(f, t) for f in ("free scratch", "free out")
                                                  for t in ("given", "times scratch", "est_out")}
    assert {v[1] for v in tags["bcr"] if v[0] == 3} == {64, 96, 128, 160, 192, 224, 256}
    assert {v[0] for v in tags["bcr"] if v[3]} == {1, 2, 3} and any(v[4] for v in tags["bcr"])
    assert {(v[0], v[2]) for v in tags["bcr"]} == {(D, n) for D in (1, 2, 3) for n in (1, 2)}
    assert {v for v in tags["chunked"]} == {(D, m, n) for D in (1, 2, 3) for m in (4, 6, 8, 10, 12) for n in (1, 2)}
    general = tags["general"]
    assert {v[0] for v in general} >= {4, 6, 8, 12} and {v[1] for v in general if v[0] == 10} >= {2, 3}
    assert {v[2] for v in general} >= {4, 5}


def test_standard_loop_and_edge_cases():
    """Grid-stride and capacity cases are where they are meant to be at 148 SMs."""
    assert S.pair_loops(S.PAIR_LOOP.B, 3, 1, SMS) and not S.pair_loops(S.PAIR_LOOP.B // 2, 3, 1, SMS)
    for c in S.BCR_CASES:
        if c.K == 40:
            assert c.B > SMS * S.bcr_resident(40, c.D)
    for D, K in ((1, 907), (2, 604), (3, 453)):
        c = S.Case(K, D, 3, "given", False, False, False, "pair_long")
        assert c in [x._replace(times="given", ends=False, free=False, cost=False) for x in S.PAIR_LONG_CASES]
        assert S.routes_of([c, c._replace(K=K + 1)]) == ["pair_long", "unsupported"]
    N, K, D, B = S.SOLVE_LOOP
    assert W.general_loops(B, S.general_solve_warps(N, K, D), SMS)
    steps, refused = S.general_solve_steps(10, 3)
    assert (steps, refused) == W.warp_steps(3, "standard")
    assert {K for N, K, _, _ in S.SOLVE_CASES if N == 10} >= {k for lo_hi in steps.values() for k in lo_hi}
    steps12, _ = S.general_solve_steps(12, 3)
    assert {S.general_solve_warps(12, K, 3) for N, K, _, _ in S.SOLVE_CASES if N == 12} == set(steps12)
    # past the standard-mask kernels (K = 513 / 604 / 907 at D = 3 / 2 / 1) the general route refuses every K, and
    # each first refused K has a case
    for D, K in S.REFUSED.items():
        c = S.Case(K, D, 2, "given", False, False, False)
        assert S.routes_of([c, c._replace(K=K - 1)]) == ["general", "bcr" if D == 3 else "pair_long"]
        assert S.general_solve_warps(10, K, D) is None
    assert S.REFUSED == {3: 514, 2: 605, 1: 908}
