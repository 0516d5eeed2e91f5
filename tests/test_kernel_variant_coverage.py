"""Every launch variant of the sampling, evaluate_range, cost and cost-sweep launchers has a case in
tests/test_gpu_kernel_variants.py.  The variant of each case comes from that file's restatement of the launcher's
choice, so a threshold moved in a .cu file (and mirrored there) that leaves some variant without a case fails here,
on a machine without a GPU."""
import test_gpu_kernel_variants as V

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
