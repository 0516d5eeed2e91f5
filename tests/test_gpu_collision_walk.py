"""The collision walk (collision_cost_kernel, minsnap_collision.cu) and the gradient instantiation of the general
recovery kernel (solve_general_kernel<N, false, true>, minsnap_general.cu) against the oracle across their launch
shapes and the edges of the map (pytest -m gpu).  Together they are the whole of an iteration of
minsnap_optimize_free_constraints.

As in test_gpu_kernel_variants.py, the launchers' choices are restated in Python with the lines they restate
(`walk_loops`, `general_warps`, `general_loops`), every case carries the variant it is meant to reach, a GPU test
checks the restatement against the device's SM count, and tests/test_kernel_variant_coverage.py (CPU) fails when a
variant has no case.

Truth and bars:
  * walk: oracle_py.collision_cost / collision_cost_gradient (ref getCostAndGradientCollision, NL.i:1523-1709).
    Cost within 1e-8 relative (floor 1e-3), gradient within 1e-8 of its largest component (floor 1e-6), the
    collision flag and the number of charged samples exactly.
  * gradient kernel: R of the long-double oracle (K <= 100), else a per-segment long-double restatement
    (R d)_c = sum over the rows (segment i, row r) that map to column c of (H_i d_i)_r.  Gradient 2 (R d)_p within
    1e-9 of its largest component, diag(R_pp) entry by entry within 1e-9 relative, J_d within COST_TOL of d^T R d
    and of 2 computeCost.
  * batches large enough for the grid-stride loop: every output bit for bit equal to the same trajectories sent in
    chunks too small to loop (one warp computes a trajectory whatever its index, and the general kernel's warps per
    CTA depend on (N, K, D, n_fixed, n_free) only), then a strided sample of 64 against the oracle.

A `charged` mismatch on random trajectories may be a threshold tie (the oracle evaluates positions as sum t^n c_n,
the kernel by Horner's rule): the assertion message carries the walk's smallest |dist_sum - map_resolution|.
No case passes an infinite segment time or more than about 1e5 samples per segment: such a walk does not end."""
import ctypes as C
import math

import numpy as np
import pytest

from helpers import COST_TOL, random_batch, standard_mask, vertex_values
from oracle import oracle_py
from test_collision_cost import ORIGIN, RES, field
from test_gpu_kernel_variants import dev, offset_view

pytestmark = pytest.mark.gpu

B200_SMS = 148
MAX_DYNAMIC_SMEM = 227 * 1024                  # minsnap_launch.h: kMaxDynamicSmem
N = 10
SNAP = 4
BOX_LO, BOX_HI = [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0]


# ------------------------------------------------------------------------------------------
# Restatements of the launchers' choices
# ------------------------------------------------------------------------------------------
def walk_loops(B, sms=B200_SMS):
    """launch_collision_cost, minsnap_collision.cu:303-307: CTAs of 128 threads (4 warps, a warp per trajectory),
    at most 32 CTAs per SM, so warps loop over the grid stride once B > SMs x 32 x 4."""
    return B > sms * 32 * 4


def general_per_warp_doubles(K, D, n_fixed, n_free, N=N):
    """GeneralLayout<N>::per_warp_doubles, minsnap_general.cu:194-196."""
    return K * (2 * N - 1) + n_free * N + n_free * D + n_fixed * D + N


def general_cta_bytes(warps, K, D, n_fixed, n_free, N=N):
    """GeneralLayout<N>::cta_bytes, minsnap_general.cu:197-200."""
    return (2 * N * N + warps * general_per_warp_doubles(K, D, n_fixed, n_free, N)) * 8 + 4 * N * K


def general_warps(K, D, n_fixed, n_free, N=N):
    """launch_general_n, minsnap_general.cu:441-444: warps per CTA halved from 8 while the CTA needs more than
    100 KiB, None (cudaErrorInvalidConfiguration, MINSNAP_ERR_UNSUPPORTED) above kMaxDynamicSmem."""
    warps = 8
    while warps > 1 and general_cta_bytes(warps, K, D, n_fixed, n_free, N) > 100 * 1024:
        warps >>= 1
    return warps if general_cta_bytes(warps, K, D, n_fixed, n_free, N) <= MAX_DYNAMIC_SMEM else None


def general_loops(B, warps, sms=B200_SMS):
    """minsnap_general.cu:456-458: at most 32 CTAs per SM, a warp per trajectory."""
    return B > sms * 32 * warps


def general_mask(K):
    """Free velocity at the first vertex and free snap at the last; the velocity fixed at vertex 1 when it is
    interior."""
    m = standard_mask(K).copy()
    m[0, 1] = 0
    m[K, N // 2 - 1] = 0
    if K >= 2:
        m[1, 1] = 1
    return m


MASKS = {"standard": standard_mask, "general": general_mask}


def mask_counts(mask):
    n_fixed = int(np.asarray(mask).sum())
    return n_fixed, np.asarray(mask).size - n_fixed


def gradient_variant(K, D, kind):
    return general_warps(K, D, *mask_counts(MASKS[kind](K)))


def warp_steps(D, kind, k_max=1000):
    """{warps: (first K, last K)} of the rule, and the first K it refuses."""
    steps = {}
    for K in range(1, k_max):
        w = gradient_variant(K, D, kind)
        if w is None:
            return steps, K
        lo, _ = steps.get(w, (K, K))
        steps[w] = (lo, K)
    raise AssertionError("no refused K below %d" % k_max)


# ------------------------------------------------------------------------------------------
# Case tables
# ------------------------------------------------------------------------------------------
# The walk's grid-stride loop: twice the warps of the capped grid and a ragged rest; chunks that do not loop.
WALK_LOOP_B = 2 * (B200_SMS * 128) + 37
WALK_CHUNK = 4096
# K on the walk: no free column (K = 1), the last vertex's column at every K
WALK_K_CASES = (1, 2, 3, 33, 100)

# (K, D, mask kind) -> warps per CTA; K = 2 and the first and last K of every step of the rule, for both masks
GRADIENT_CASES = []
ERROR_CASES = []                               # (K, D, mask kind): the first K the launcher refuses
for _kind in ("standard", "general"):
    _steps, _refused = warp_steps(3, _kind)
    for _K in sorted({2, *(k for lo_hi in _steps.values() for k in lo_hi)}):
        GRADIENT_CASES.append(((_K, 3, _kind), gradient_variant(_K, 3, _kind)))
    ERROR_CASES.append((_refused, 3, _kind))
GRADIENT_CASES.append(((100, 1, "standard"), gradient_variant(100, 1, "standard")))   # D = 1 past its K = 96 step

# (K, B, chunk) of the gradient kernel's grid-stride cases: 8 warps per CTA at K = 10, 1 warp at K = 100
GRADIENT_LOOP_CASES = [(10, 2 * B200_SMS * 32 * 8 + 37, 8192), (100, 2 * B200_SMS * 32 * 1 + 37, 2048)]
# free_objective: B x S candidates go through coeffs_from_constraints (the same launcher, 8 warps at K = 10) and the
# walk; chunks of FREE_CHUNK trajectories loop in neither
FREE_K, FREE_B, FREE_S, FREE_CHUNK = 10, 5000, 8, 500

# Map geometry: three sizes, three origins, a grid smaller than [min_bound, max_bound] in x and y
GRID2_DIMS = (40, 72, 56)
GRID2_ORIGIN = np.array([-10.75, -17.5, -13.25])
GRID2_RES = 0.5
MAP_CASES = {
    "oob_collides": dict(oob_value=0.0),                           # outside the grid: d = 0 < robot_radius
    "oob_free": dict(oob_value=2.0),                               # outside the grid: d > robot_radius + epsilon
    "fine_threshold": dict(oob_value=0.0, map_resolution=0.35),
    "coarse_threshold": dict(oob_value=2.0, map_resolution=1.3),
    "zero_radius": dict(oob_value=0.0, robot_radius=0.0),
}


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
WORST = {}


def record(key, value):
    WORST[key] = max(WORST.get(key, 0.0), float(value))


def report(*keys):
    print(" ".join("%s %.3e" % (k, WORST.get(k, 0.0)) for k in keys))


def sample_rows(B, n=64):
    return sorted({0, B - 1, *np.linspace(0, B - 1, n).astype(int).tolist()})


def horner(c, t):
    x = c[-1]
    for a in c[-2::-1]:
        x = x * t + a
    return x


def replay_walk(coeffs, times, dt, limit):
    """The walk of minsnap_collision.cu:142-239 (ref NL.i:1560-1698) in Python.  -> (charged samples as
    (segment, t, time_sum, position, velocity), time_sum on entering each segment, number of samples of each
    segment, smallest |dist_sum - limit| met)."""
    charged, entry, counts, margin = [], [], [], np.inf
    time_sum, dist_sum, prev = -1.0, 0.0, None
    for i, T in enumerate(times):
        entry.append(time_sum)
        c = coeffs[i]
        dc = c[:, 1:] * np.arange(1, c.shape[1])
        t, n = 0.0, 0
        while t < T:
            n += 1
            p = np.array([horner(c[k], t) for k in range(3)])
            if time_sum < 0:
                time_sum, prev = 0.0, p
                t += dt
                continue
            time_sum += dt
            dist_sum += math.sqrt(((p - prev) ** 2).sum())
            prev = p
            margin = min(margin, abs(dist_sum - limit))
            if dist_sum >= limit:
                charged.append((i, t, time_sum, p, np.array([horner(dc[k], t) for k in range(3)])))
                dist_sum = time_sum = 0.0
            t += dt
        counts.append(n)
        time_sum += -dt + (T - t)
    return charged, entry, counts, margin


def walk_kw(kw):
    return dict(kw, map_resolution=kw.get("map_resolution", kw["resolution"]))


def check_walk(coeffs, times, g, kw, cost, hit, charged, grad=None, col=None, n_fixed=0, n_free=0, rows=None,
               key="walk"):
    """Rows of the kernel's outputs against the oracle; the gradient when `grad` is given."""
    kw = walk_kw(kw)
    for b in range(len(times)) if rows is None else rows:
        if grad is None:
            want_cost, want_hit, want_charged = oracle_py.collision_cost(coeffs[b], times[b], g, **kw)
        else:
            want_cost, want_g, want_hit, want_charged = oracle_py.collision_cost_gradient(coeffs[b], times[b], col,
                                                                                         n_fixed, n_free, sdf=g, **kw)
        if charged[b] != want_charged:
            margin = replay_walk(coeffs[b], times[b], kw["dt"], kw["map_resolution"])[3]
            raise AssertionError("row %d: %d charged samples, oracle %d; smallest |dist_sum - map_resolution| %.3e"
                                 % (b, charged[b], want_charged, margin))
        assert hit[b] == want_hit, (b, hit[b], want_hit)
        rel = abs(cost[b] - want_cost) / max(abs(want_cost), 1e-3)
        record(key + "_cost_rel", rel)
        assert rel <= 1e-8, (b, cost[b], want_cost)
        if grad is not None and n_free > 0:
            scale = max(np.abs(want_g).max(), 1e-6)
            err = np.abs(grad[b] - want_g).max() / scale
            record(key + "_grad_rel", err)
            assert err <= 1e-8, (b, err, scale)


def walk_on_device(ms, torch, coeffs_d, times_d, sdf_d, kw, col=None, n_fixed=0, n_free=None):
    """collision_cost with the charged counts and collision_gradient in the standard mask's closed form (or through
    `col`); the cost, flag and count of both calls must agree bit for bit."""
    plain = ms.collision_cost(coeffs_d, times_d, sdf_d, want_charged=True, **kw)
    if col is None:
        out = ms.collision_gradient(coeffs_d, times_d, sdf_d, **kw)
    else:
        out = ms.collision_gradient(coeffs_d, times_d, sdf_d, col_of_row=dev(torch, col), n_fixed=n_fixed,
                                    n_free=n_free, **kw)
    for k in ("cost", "is_collision", "charged"):
        assert torch.equal(out[k], plain[k]), k
    return out


def solved_standard(ms, torch, B, K, seed, lo=BOX_LO, hi=BOX_HI):
    """Trajectories of the reference's generator solved on the device: (coeffs, times) as CUDA tensors."""
    pos = dev(torch, ms.random_positions_host(B, K, lo, hi, seed))
    times = ms.estimate_segment_times(pos, 3.0, 5.0)
    return ms.solve_standard(pos, times, want_status=False)["coeffs"], times


def oracle_trajectories(oracle, B, K, seed, lo=BOX_LO, hi=BOX_HI):
    """Trajectories of the reference's generator solved by the oracle (standard mask): (coeffs, times)."""
    pos = [oracle.create_random_positions(K, lo, hi, seed + b) for b in range(B)]
    times = np.stack([oracle.estimate_segment_times(x, 3.0, 5.0) for x in pos]).astype(np.float64)
    coeffs = np.stack([oracle.solve(N, K, 3, SNAP, standard_mask(K), vertex_values(x), t)["coeffs"]
                       for x, t in zip(pos, times)]).astype(np.float64)
    return coeffs, times


CHAIN_B, CHAIN_SEED, CHAIN_FIELD = 6, 700, "box"
MAP_B, MAP_K, MAP_SEED = 24, 6, 4100
MAP_LO, MAP_HI = [-12.0, -22.0, -12.0], [12.0, 22.0, 12.0]     # beyond the grid in x and y, beyond the bounds in z


def chain_case(oracle, K):
    return oracle_trajectories(oracle, CHAIN_B, K, CHAIN_SEED + K)


def chain_kw():
    return dict(MAP1, map_resolution=RES, use_continuous_distance=True)


def map_case(oracle, case, continuous):
    coeffs, times = oracle_trajectories(oracle, MAP_B, MAP_K, MAP_SEED, MAP_LO, MAP_HI)
    kw = dict(origin=GRID2_ORIGIN, resolution=GRID2_RES, min_bound=BOX_LO, max_bound=BOX_HI, dt=0.1, epsilon=0.5,
              robot_radius=0.5, coll_pot_multiplier=1.5, use_continuous_distance=continuous)
    kw.update(MAP_CASES[case])
    return coeffs, times, kw


def host(t, rows=None):
    return (t if rows is None else t[rows]).cpu().numpy()


# The map of test_collision_cost.py (48 x 88 x 48, sphere field) with a threshold and weights the tests vary
MAP1 = dict(origin=ORIGIN, resolution=RES, min_bound=BOX_LO, max_bound=BOX_HI, dt=0.1, epsilon=0.5, robot_radius=0.5,
            coll_pot_multiplier=1.5, oob_value=0.0)


def grid2_field():
    """Asymmetric in every axis, with values in all three branches of cost_potential."""
    ax = [GRID2_ORIGIN[k] + (np.arange(GRID2_DIMS[k]) + 0.5) * GRID2_RES for k in range(3)]
    X, Y, Z = np.meshgrid(*ax, indexing="ij")
    return (0.75 + 0.5 * np.sin(0.6 * X + 0.3) * np.cos(0.35 * Y - 0.2) + 0.3 * np.sin(0.5 * Z + 0.9) + 0.02 * X
            - 0.015 * Y + 0.01 * Z + 0.004 * X * Y)


# ------------------------------------------------------------------------------------------
# The restatements on this device
# ------------------------------------------------------------------------------------------
def test_restatements_hold_on_this_device(ms, torch_cuda):
    """The grid caps are restated for the SM count of the device, and the warps-per-CTA steps are the ones the
    launcher takes: the first refused K of each mask is refused and the K below it is taken."""
    torch = torch_cuda
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    assert sms == ms.device_info()["sm_count"] == B200_SMS, "the loop cases' batch sizes are set for %d SMs" % B200_SMS
    print("walk: %d trajectories loop over %d warps; chunks of %d do not"
          % (WALK_LOOP_B, B200_SMS * 128, WALK_CHUNK))
    assert walk_loops(WALK_LOOP_B, sms) and not walk_loops(WALK_CHUNK, sms)
    for K, B, chunk in GRADIENT_LOOP_CASES:
        w = gradient_variant(K, 3, "standard")
        print("gradient kernel K=%d: %d warps per CTA, %d trajectories loop over %d warps; chunks of %d do not"
              % (K, w, B, sms * 32 * w, chunk))
        assert general_loops(B, w, sms) and not general_loops(chunk, w, sms)
    for K, D, kind in ERROR_CASES:
        for k in (K - 1, K):
            m = MASKS[kind](k)
            n_fixed, n_free = mask_counts(m)
            args = (m, torch.zeros((2, n_fixed, D), dtype=torch.float64, device="cuda"),
                    torch.zeros((2, n_free, D), dtype=torch.float64, device="cuda"),
                    torch.ones((2, k), dtype=torch.float64, device="cuda"))
            if k < K:
                ms.derivative_gradient(*args)
            else:
                with pytest.raises(ms.MinsnapError):
                    ms.derivative_gradient(*args)


# ------------------------------------------------------------------------------------------
# The walk: grid-stride loop, chain lengths, segment boundaries, map geometry, call paths
# ------------------------------------------------------------------------------------------
def test_walk_grid_stride(ms, oracle, torch_cuda):
    """More trajectories than the capped grid has warps: every output equals chunked calls that do not loop, bit for
    bit, for the cost, the flag, the charged count and the gradient (closed form and index map); 64 rows against the
    oracle."""
    torch = torch_cuda
    B, K = WALK_LOOP_B, 10
    assert walk_loops(B) and not walk_loops(WALK_CHUNK)
    print("walk grid stride: B = %d > %d warps of the capped grid" % (B, B200_SMS * 128))
    coeffs_d, times_d = solved_standard(ms, torch, B, K, 9001)
    g = field("sphere")
    g_d = dev(torch, g)
    kw = dict(MAP1, map_resolution=RES, use_continuous_distance=True)
    col, n_fixed, n_free = oracle.reorder(N, K, standard_mask(K))
    out = walk_on_device(ms, torch, coeffs_d, times_d, g_d, kw)
    out_map = ms.collision_gradient(coeffs_d, times_d, g_d, col_of_row=dev(torch, col), n_fixed=n_fixed, n_free=n_free,
                                    **kw)
    assert torch.equal(out["gradient"], out_map["gradient"]) and torch.equal(out["cost"], out_map["cost"])
    for s in range(0, B, WALK_CHUNK):
        e = min(s + WALK_CHUNK, B)
        part = walk_on_device(ms, torch, coeffs_d[s:e], times_d[s:e], g_d, kw)
        for k in ("cost", "is_collision", "charged", "gradient"):
            assert torch.equal(part[k], out[k][s:e]), (k, s)
    rows = sample_rows(B)
    idx = torch.tensor(rows, device="cuda")
    coeffs, times = host(coeffs_d, idx), host(times_d, idx)
    r = range(len(rows))
    check_walk(coeffs, times, g, kw, host(out["cost"], idx), host(out["is_collision"], idx), host(out["charged"], idx),
               host(out["gradient"], idx), col, n_fixed, n_free, rows=r, key="walk_loop")
    assert int(out["is_collision"].sum()) > 0 and float(out["gradient"].abs().max()) > 0
    report("walk_loop_cost_rel", "walk_loop_grad_rel")


@pytest.mark.parametrize("K", WALK_K_CASES)
def test_walk_chain_lengths(ms, oracle, torch_cuda, K):
    """The closed form of the standard mask's columns (minsnap_collision.cu:263-265) equals the index map bit for bit
    at every K, the last vertex's column (row r >= N/2 of segment K-1) included; K = 1 has no free column and returns
    a [B, 0, 3] gradient.  An all-fixed general mask (n_free = 0) gives the cost alone.  The host entry points
    return the device's bits at K = 1 and K = 100."""
    torch = torch_cuda
    B = CHAIN_B
    coeffs, times = chain_case(oracle, K)
    coeffs_d, times_d = dev(torch, coeffs), dev(torch, times)
    g = field(CHAIN_FIELD)
    g_d = dev(torch, g)
    kw = chain_kw()
    col, n_fixed, n_free = oracle.reorder(N, K, standard_mask(K))
    assert n_free == 4 * (K - 1)
    out = walk_on_device(ms, torch, coeffs_d, times_d, g_d, kw)
    out_map = walk_on_device(ms, torch, coeffs_d, times_d, g_d, kw, col, n_fixed, n_free)
    assert out["gradient"].shape == (B, n_free, 3)
    assert torch.equal(out["gradient"], out_map["gradient"])
    check_walk(coeffs, times, g, kw, host(out["cost"]), host(out["is_collision"]), host(out["charged"]),
               host(out["gradient"]), col, n_fixed, n_free, key="walk_chain")
    ones = np.ones((K + 1, N // 2), np.uint8)
    col1, nf1, np1 = oracle.reorder(N, K, ones)
    assert np1 == 0
    fixed_only = walk_on_device(ms, torch, coeffs_d, times_d, g_d, kw, col1, nf1, np1)
    assert fixed_only["gradient"].shape == (B, 0, 3) and torch.equal(fixed_only["cost"], out["cost"])
    if K in (1, 100):
        hc = ms.collision_cost_host(coeffs, times, g, **kw)
        hg = ms.collision_gradient_host(coeffs, times, g, **kw)
        for k in ("cost", "is_collision", "charged"):
            assert np.array_equal(hc[k], host(out[k])) and np.array_equal(hg[k], host(out[k])), k
        assert np.array_equal(hg["gradient"], host(out["gradient"]))
    report("walk_chain_cost_rel", "walk_chain_grad_rel")


def line_coeffs(starts, velocities, accelerations=None):
    """Segment i: start_i + v_i t (+ a_i t^2 / 2) -> coeffs [K][3][N]."""
    K = len(starts)
    c = np.zeros((K, 3, N))
    c[:, :, 0] = starts
    c[:, :, 1] = velocities
    if accelerations is not None:
        c[:, :, 2] = 0.5 * np.asarray(accelerations)
    return c


def chained(start, velocities, times):
    """Continuous piecewise-linear: each segment starts where the previous one ends."""
    starts = [np.asarray(start, float)]
    for v, T in zip(velocities[:-1], times[:-1]):
        starts.append(starts[-1] + np.asarray(v) * T)
    return line_coeffs(starts, velocities)


def repeated(dt, n):
    t = 0.0
    for _ in range(n):
        t += dt
    return t


def boundary_cases():
    """Hand-built walks through the obstacle of field("sphere"), with what each must exercise (checked on the Python
    replay by test_kernel_variant_coverage.py).  Speeds near 1 and thresholds half a step away from a multiple of
    the step length keep every charge clear of a tie."""
    dt = 0.1
    T32, T64 = repeated(dt, 32), repeated(dt, 64)
    v = [[0.6, -0.7, 0.38], [-0.5, 0.55, 0.62], [0.7, 0.45, -0.52], [-0.66, -0.6, 0.41]]
    cases = {}
    # a chunk ends exactly at lane 31 (the next chunk has no valid sample) with T on, one ulp below and above 32 dt
    times = np.array([T32, np.nextafter(T32, 0.0), np.nextafter(T32, np.inf), T64])
    cases["lane31"] = (chained([-2.0, 1.5, -1.0], v, times), times, dt, 0.45, True)
    # a segment shorter than dt, and an interior T = 0 that turns time_sum negative (the next first sample is skipped)
    times = np.array([0.75, 0.0, 1.2, 0.05, 0.9])
    cases["short_and_zero"] = (chained([-2.0, -1.0, 0.0], v + [v[0]], times), times, dt, 0.45, False)
    # more than 60 chunks in one segment
    times = np.array([2.0, 1.1])
    cases["many_chunks"] = (chained([-1.0, -3.0, -1.5], v[:2], times), times, 0.001, 0.0505, True)
    # a jump into the obstacle onto a sample with |v| < 1e-6: charged, kept by the cost, dropped by the gradient
    T = np.array([1.0, 1.5, 1.0])
    jump = np.array([1.5, -1.0, 0.0])                  # inside the sphere of field("sphere")
    v1, a1 = np.array([3e-7, -2e-7, 4e-7]), np.array([1.2, 0.8, -0.6])
    end1 = jump + v1 * T[1] + 0.5 * a1 * T[1] ** 2
    c = line_coeffs([[-6.0, -8.0, 2.0], jump, end1], [[0.01, 0.005, 0.0], v1, v1 + a1 * T[1]],
                    [np.zeros(3), a1, np.zeros(3)])
    cases["slow_jump"] = (c, T, dt, 0.45, True)
    # two rows (two warps): the walk and the same walk translated, which charges the same samples elsewhere
    shift = np.zeros((3, N))
    shift[:, 0] = [0.3, -0.2, 0.1]
    return {k: (np.stack([c, c + shift]), np.stack([t, t]), dt, limit, grad)
            for k, (c, t, dt, limit, grad) in cases.items()}


BOUNDARY_CASES = boundary_cases()


@pytest.mark.parametrize("name", list(BOUNDARY_CASES))
def test_walk_segment_boundaries(ms, oracle, torch_cuda, name):
    """Hand-built walks against the oracle.  The case with a zero-length segment is checked for the cost only: its
    mapping matrix is singular, so neither the reference nor the kernel has a gradient there."""
    torch = torch_cuda
    c3, t3, dt, limit, with_gradient = BOUNDARY_CASES[name]
    K = t3.shape[1]
    g = field("sphere")
    kw = dict(MAP1, dt=dt, map_resolution=limit, use_continuous_distance=True)
    c_d, t_d, g_d = dev(torch, c3), dev(torch, t3), dev(torch, g)
    if with_gradient:
        col, n_fixed, n_free = oracle.reorder(N, K, standard_mask(K))
        out = walk_on_device(ms, torch, c_d, t_d, g_d, kw)
        out_map = walk_on_device(ms, torch, c_d, t_d, g_d, kw, col, n_fixed, n_free)
        assert torch.equal(out["gradient"], out_map["gradient"])
        check_walk(c3, t3, g, kw, host(out["cost"]), host(out["is_collision"]), host(out["charged"]),
                   host(out["gradient"]), col, n_fixed, n_free, key="walk_boundary")
    else:
        out = ms.collision_cost(c_d, t_d, g_d, want_charged=True, **kw)
        check_walk(c3, t3, g, kw, host(out["cost"]), host(out["is_collision"]), host(out["charged"]),
                   key="walk_boundary")
    report("walk_boundary_cost_rel", "walk_boundary_grad_rel")


def potential_kw(kw):
    return {k: kw[k] for k in ("origin", "resolution", "min_bound", "max_bound", "map_resolution", "epsilon",
                               "robot_radius", "coll_pot_multiplier", "use_continuous_distance", "oob_value")}


def map_edges(coeffs, times, g, kw):
    """What the charged samples of these walks reach: the three branches of cost_potential, samples outside the
    grid, and (continuous mode) centres whose eight-cell stencil falls off the grid inside the valid bounds."""
    kw = walk_kw(kw)
    dims, org, res, mr = np.array(g.shape), np.asarray(kw["origin"]), kw["resolution"], kw["map_resolution"]
    lo, hi = np.asarray(kw["min_bound"]), np.asarray(kw["max_bound"])
    seen = dict(collision=0, band=0, free=0, outside=0, stencil_off=0)
    for b in range(len(times)):
        for _, _, _, p, _ in replay_walk(coeffs[b], times[b], kw["dt"], mr)[0]:
            cost, _, hit = oracle_py.collision_potential(p, g, **potential_kw(kw))
            seen["collision" if hit else ("band" if cost > 0 else "free")] += 1
            idx = np.floor((p - org) / res).astype(int)
            seen["outside"] += bool(((idx < 0) | (idx >= dims)).any())
            valid_state = bool(((p >= lo + mr) & (p <= hi - mr)).all())
            seen["stencil_off"] += valid_state and bool(((idx - 1 < 0) | (idx + 1 >= dims)).any())
    return seen


@pytest.mark.parametrize("continuous", [True, False])
@pytest.mark.parametrize("case", list(MAP_CASES))
def test_walk_map_geometry(ms, oracle, torch_cuda, case, continuous):
    """A 40 x 72 x 56 grid with three different origins, smaller than [min_bound, max_bound] in x and y, an
    asymmetric field, trajectories that leave the grid; oob_value below robot_radius and above robot_radius +
    epsilon, map_resolution smaller and larger than the grid's, robot_radius = 0.  That the charged samples reach
    the three branches of cost_potential, cells outside the grid and (continuous mode) the discrete fallback of a
    stencil that falls off the grid is checked on the CPU (test_kernel_variant_coverage.py)."""
    torch = torch_cuda
    coeffs, times, kw = map_case(oracle, case, continuous)
    g = grid2_field()
    col, n_fixed, n_free = oracle.reorder(N, MAP_K, standard_mask(MAP_K))
    out = walk_on_device(ms, torch, dev(torch, coeffs), dev(torch, times), dev(torch, g), kw)
    check_walk(coeffs, times, g, kw, host(out["cost"]), host(out["is_collision"]), host(out["charged"]),
               host(out["gradient"]), col, n_fixed, n_free, key="walk_map")
    assert int(host(out["is_collision"]).sum()) > 0
    report("walk_map_cost_rel", "walk_map_grad_rel")


def test_walk_call_paths(ms, oracle, torch_cuda):
    """Null is_collision and charged pointers through the C ABI (as minsnap_free_objective and the descent call the
    walk) and coefficients, times and field read through 8-byte-offset views: the same bits."""
    torch = torch_cuda
    B, K = 40, 10
    coeffs_d, times_d = solved_standard(ms, torch, B, K, 5150)
    g = field("smooth")
    g_d = dev(torch, g)
    kw = dict(MAP1, map_resolution=RES, use_continuous_distance=True)
    out = walk_on_device(ms, torch, coeffs_d, times_d, g_d, kw)
    lib = ms.capi.load()
    # held: the host arrays margs points into, alive until the calls below have returned
    held, margs = ms.api._collision_map(g_d, kw["origin"], kw["resolution"], kw["min_bound"], kw["max_bound"],
                                        kw["dt"], kw["map_resolution"], kw["epsilon"], kw["robot_radius"],
                                        kw["coll_pot_multiplier"], True, kw["oob_value"])
    p = lambda t: C.c_void_p(t.data_ptr())
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    cost = torch.full((B,), -1.0, dtype=torch.float64, device="cuda")
    ms.capi.check(lib.minsnap_collision_cost(B, K, 3, N, p(coeffs_d), p(times_d), *margs, p(cost), None, None, stream),
                  "minsnap_collision_cost")
    assert torch.equal(cost, out["cost"])
    cost.fill_(-1.0)
    grad = torch.full_like(out["gradient"], 7.0)
    ms.capi.check(lib.minsnap_collision_gradient(B, K, 3, N, p(coeffs_d), p(times_d), *margs, None, 0,
                                                 4 * (K - 1), p(cost), p(grad), None, None, stream),
                  "minsnap_collision_gradient")
    assert torch.equal(cost, out["cost"]) and torch.equal(grad, out["gradient"])
    c_o, t_o, g_o = offset_view(torch, host(coeffs_d)), offset_view(torch, host(times_d)), offset_view(torch, g)
    off = walk_on_device(ms, torch, c_o, t_o, g_o, kw)
    for k in ("cost", "is_collision", "charged", "gradient"):
        assert torch.equal(off[k], out[k]), k
    check_walk(host(coeffs_d), host(times_d), g, kw, host(out["cost"]), host(out["is_collision"]), host(out["charged"]),
               host(out["gradient"]), *oracle.reorder(N, K, standard_mask(K)), rows=range(0, B, 5), key="walk_paths")


# ------------------------------------------------------------------------------------------
# The gradient kernel: every warps-per-CTA step, the refused K, the grid-stride loop, free_objective
# ------------------------------------------------------------------------------------------
def gradient_problem(oracle, B, K, D, mask, seed):
    """Times of the reference's generator, fixed values with non-zero higher derivatives, random free values."""
    pos, times = random_batch(oracle, B, K, D, seed=seed)
    rng = np.random.default_rng(seed)
    h = N // 2
    vv = np.stack([vertex_values(p) for p in pos])
    vv = vv + mask[None, :, :, None] * (np.arange(h) > 0)[None, None, :, None] * rng.normal(size=vv.shape) * 0.3
    fixed = np.ascontiguousarray(vv[:, mask.astype(bool)])
    free = rng.normal(size=(B, mask_counts(mask)[1], D)) * 2.0
    return times, fixed, free


def per_segment_truth(oracle_ld, col, n_fixed, d_all, times):
    """(R d [D][n_all], diag(R) [n_all]) in long double from the segments' Hessians, R = sum_i M_i^T H_i M_i
    (orc_solve_linear's assembly): row r of segment i holds column col[i N + r]."""
    d = d_all.astype(np.longdouble)
    Rd = np.zeros(d.shape, np.longdouble)
    diag = np.zeros(d.shape[1], np.longdouble)
    for i, T in enumerate(times):
        H = oracle_ld.segment_hessian(N, SNAP, T)
        cols = col[i * N:(i + 1) * N]
        Rd[:, cols] += d[:, cols] @ H.T
        diag[cols] += np.diag(H)
    return Rd, diag


def check_gradient_rows(oracle, oracle_ld, mask, fixed, free, times, jd, grad, diag, rows, use_R, key):
    K = mask.shape[0] - 1
    D = fixed.shape[2]
    col, n_fixed, n_free = oracle.reorder(N, K, mask)
    for j, b in enumerate(rows):
        d_all = np.concatenate([fixed[b].T, free[b].T], axis=1)          # [D][n_all]
        Rd, want_diag = per_segment_truth(oracle_ld, col, n_fixed, d_all, times[b])
        if use_R:
            vv = np.zeros((K + 1, N // 2, D))
            vv[mask.astype(bool)] = fixed[b]
            R = np.asarray(oracle_ld.solve(N, K, D, SNAP, mask, vv, times[b], want_R=True)["R"], np.longdouble)
            Rd_R = d_all.astype(np.longdouble) @ R.T
            # the restatement used where R is too dear agrees with R
            assert np.abs(Rd_R - Rd).max() <= 1e-12 * np.abs(Rd_R).max()
            assert np.abs(np.diag(R) - want_diag).max() <= 1e-12 * np.abs(want_diag).max()
            Rd, want_diag = Rd_R, np.diag(R)
        want_jd = float((d_all.astype(np.longdouble) * Rd).sum())
        rel = abs(jd[j] - want_jd) / want_jd
        record(key + "_jd_rel", rel)
        assert rel <= COST_TOL, (b, jd[j], want_jd)
        coeffs = oracle_ld.coeffs_from_constraints(N, K, D, col, d_all, times[b])
        cost2 = 2.0 * float(oracle_ld.compute_cost(N, K, D, SNAP, coeffs, times[b]))
        assert abs(jd[j] - cost2) <= COST_TOL * cost2, (b, jd[j], cost2)
        if n_free == 0:
            continue
        want_g = (2.0 * Rd[:, n_fixed:]).T.astype(np.float64)             # [n_free][D]
        err = np.abs(grad[j] - want_g).max() / np.abs(want_g).max()
        record(key + "_grad_rel", err)
        assert err <= 1e-9, (b, err)
        wd = want_diag[n_fixed:].astype(np.float64)
        derr = (np.abs(diag[j] - wd) / np.abs(wd)).max()
        record(key + "_diag_rel", derr)
        assert derr <= 1e-9, (b, derr)


@pytest.mark.parametrize("case", GRADIENT_CASES, ids=lambda c: "K%d-D%d-%s-w%d" % (*c[0], c[1]))
def test_derivative_gradient_warp_steps(ms, oracle, oracle_ld, torch_cuda, case):
    """One case on each side of every warps-per-CTA step; ragged batches (2 warps + 1 trajectories: a third CTA with
    one).  Truth: the long-double oracle's R up to K = 100, the per-segment restatement (checked against R there) above."""
    torch = torch_cuda
    (K, D, kind), warps = case
    mask = MASKS[kind](K)
    B = 2 * warps + 1
    times, fixed, free = gradient_problem(oracle, B, K, D, mask, 50 + K + 7 * D)
    t, f, p = dev(torch, times), dev(torch, fixed), dev(torch, free)
    out = ms.derivative_gradient(mask, f, p, t, want_coeffs=True, want_diag=True)
    assert torch.equal(out["coeffs"], ms.coeffs_from_constraints(mask, f, p, t))
    assert out["gradient"].shape == (B, mask_counts(mask)[1], D)
    check_gradient_rows(oracle, oracle_ld, mask, fixed, free, times, host(out["Jd"]), host(out["gradient"]),
                        host(out["diag"]), range(B), use_R=K <= 100, key="gradient_steps")
    report("gradient_steps_jd_rel", "gradient_steps_grad_rel", "gradient_steps_diag_rel")


@pytest.mark.parametrize("case", ERROR_CASES, ids=lambda c: "K%d-D%d-%s" % c)
def test_derivative_gradient_refused_shape(ms, oracle, torch_cuda, case):
    """The first K whose CTA exceeds kMaxDynamicSmem at one warp: MINSNAP_ERR_UNSUPPORTED (MinsnapError in Python)
    and not one output written."""
    torch = torch_cuda
    K, D, kind = case
    assert gradient_variant(K, D, kind) is None and gradient_variant(K - 1, D, kind) == 1
    mask = MASKS[kind](K)
    n_fixed, n_free = mask_counts(mask)
    B = 3
    times, fixed, free = gradient_problem(oracle, B, K, D, mask, 66)
    t, f, pf = dev(torch, times), dev(torch, fixed), dev(torch, free)
    with pytest.raises(ms.MinsnapError):
        ms.derivative_gradient(mask, f, pf, t, want_coeffs=True, want_diag=True)
    coeffs = torch.full((B, K, D, N), -7.5, dtype=torch.float64, device="cuda")
    jd = torch.full((B,), -7.5, dtype=torch.float64, device="cuda")
    grad = torch.full((B, n_free, D), -7.5, dtype=torch.float64, device="cuda")
    diag = torch.full((B, n_free), -7.5, dtype=torch.float64, device="cuda")
    lib = ms.capi.load()
    ws_bytes = lib.minsnap_solve_workspace_bytes(N, K)
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device="cuda")
    m = np.ascontiguousarray(mask, np.uint8)
    p = lambda x: C.c_void_p(x.data_ptr())
    rc = lib.minsnap_derivative_gradient(B, K, D, N, SNAP, m.ctypes.data_as(C.c_void_p), p(f), p(pf), p(t), p(coeffs),
                                         p(jd), p(grad), p(diag), p(ws), ws_bytes,
                                         C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert rc == ms.capi.ERR_UNSUPPORTED
    for x in (coeffs, jd, grad, diag):
        assert bool((x == -7.5).all())


def vectorised_fixed(positions, mask):
    vv = np.zeros(positions.shape[:2] + (N // 2, positions.shape[2]))
    vv[:, :, 0] = positions
    return np.ascontiguousarray(vv[:, mask.astype(bool)])


@pytest.mark.parametrize("K,B,chunk", GRADIENT_LOOP_CASES)
def test_derivative_gradient_grid_stride(ms, oracle, oracle_ld, torch_cuda, K, B, chunk):
    """More trajectories than the capped grid has warps, at 8 and at 1 warp per CTA: J_d, the gradient, diag(R_pp)
    and the coefficients equal chunked calls bit for bit; 64 rows against the per-segment long-double truth."""
    torch = torch_cuda
    mask = standard_mask(K)
    warps = gradient_variant(K, 3, "standard")
    assert general_loops(B, warps) and not general_loops(chunk, warps)
    print("gradient kernel grid stride: K = %d, B = %d > %d warps of the capped grid (%d per CTA)"
          % (K, B, B200_SMS * 32 * warps, warps))
    pos = ms.random_positions_host(B, K, BOX_LO, BOX_HI, 777 + K)
    f = dev(torch, vectorised_fixed(pos, mask))
    t = ms.estimate_segment_times(dev(torch, pos), 3.0, 5.0)
    gen = torch.Generator(device="cuda").manual_seed(K)
    p = 2.0 * torch.randn((B, mask_counts(mask)[1], 3), generator=gen, device="cuda", dtype=torch.float64)
    out = ms.derivative_gradient(mask, f, p, t, want_coeffs=True, want_diag=True)
    for s in range(0, B, chunk):
        e = min(s + chunk, B)
        part = ms.derivative_gradient(mask, f[s:e], p[s:e], t[s:e], want_coeffs=True, want_diag=True)
        for k in ("Jd", "gradient", "diag", "coeffs"):
            assert torch.equal(part[k], out[k][s:e]), (k, s)
    rows = sample_rows(B)
    idx = torch.tensor(rows, device="cuda")
    check_gradient_rows(oracle, oracle_ld, mask, host(f), host(p), host(t), host(out["Jd"], idx),
                        host(out["gradient"], idx), host(out["diag"], idx), rows, use_R=False, key="gradient_loop")
    report("gradient_loop_jd_rel", "gradient_loop_grad_rel", "gradient_loop_diag_rel")


def test_free_objective_grid_stride(ms, oracle, torch_cuda):
    """B x S candidates beyond both capped grids (the recovery at 8 warps per CTA and the walk): J_c equals
    collision_cost on coeffs_from_constraints of the flattened candidates bit for bit, J_d, J_c, the flags and the
    objective equal chunked calls bit for bit, and 64 candidates are within 1e-8 of the oracle's objective."""
    torch = torch_cuda
    K, B, S = FREE_K, FREE_B, FREE_S
    mask = standard_mask(K)
    n = B * S
    warps = gradient_variant(K, 3, "standard")
    assert general_loops(n, warps) and walk_loops(n)
    assert not general_loops(FREE_CHUNK * S, warps) and not walk_loops(FREE_CHUNK * S)
    print("free_objective grid stride: %d candidates > %d warps of the recovery grid and > %d of the walk's"
          % (n, B200_SMS * 32 * warps, B200_SMS * 128))
    pos = ms.random_positions_host(B, K, BOX_LO, BOX_HI, 2024)
    f = dev(torch, vectorised_fixed(pos, mask))
    base = ms.estimate_segment_times(dev(torch, pos), 3.0, 5.0)
    opt = ms.solve(mask, f, base)["free_values"]
    gen = torch.Generator(device="cuda").manual_seed(5)
    free = (opt[:, None] + 0.4 * torch.randn((B, S) + tuple(opt.shape[1:]), generator=gen, device="cuda",
                                             dtype=torch.float64)).contiguous()
    times = (base[:, None, :] * (0.8 + 0.45 * torch.rand((B, S, K), generator=gen, device="cuda",
                                                          dtype=torch.float64))).contiguous()
    g = field("sphere")
    g_d = dev(torch, g)
    kw = dict(MAP1, map_resolution=RES, use_continuous_distance=True, oob_value=10.0)
    w = dict(w_c=10.0, w_d=0.1, w_t=1.0)
    obj, terms = ms.free_objective(mask, f, free, times, g_d, want_terms=True, **w, **kw)
    flat_t = times.reshape(n, K)
    coeffs = ms.coeffs_from_constraints(mask, f.repeat_interleave(S, 0), free.reshape(n, -1, 3), flat_t)
    jc = ms.collision_cost(coeffs, flat_t, g_d, **kw)
    assert torch.equal(terms["Jc"].reshape(-1), jc["cost"])
    assert torch.equal(terms["is_collision"].reshape(-1), jc["is_collision"])
    for s in range(0, B, FREE_CHUNK):
        e = min(s + FREE_CHUNK, B)
        o, tm = ms.free_objective(mask, f[s:e], free[s:e], times[s:e], g_d, want_terms=True, **w, **kw)
        assert torch.equal(o, obj[s:e])
        for k in ("Jd", "Jc", "is_collision"):
            assert torch.equal(tm[k], terms[k][s:e]), (k, s)
    assert int(terms["is_collision"].sum()) > 0
    col, n_fixed, _ = oracle.reorder(N, K, mask)
    fixed_h, free_h, times_h, obj_h = host(f), host(free), host(times), host(obj)
    for r in sample_rows(n):
        b, s = divmod(r, S)
        d_all = np.concatenate([fixed_h[b].T, free_h[b, s].T], axis=1)
        c = np.asarray(oracle.coeffs_from_constraints(N, K, 3, col, d_all, times_h[b, s]), np.float64)
        want_jd = 2.0 * float(oracle.compute_cost(N, K, 3, SNAP, c, times_h[b, s]))
        want_jc = oracle_py.collision_cost(c, times_h[b, s], g, **kw)[0]
        total = 0.0
        for x in times_h[b, s]:
            total += x
        want = w["w_d"] * want_jd + w["w_c"] * want_jc + w["w_t"] * total
        rel = abs(obj_h[b, s] - want) / abs(want)
        record("free_objective_rel", rel)
        assert rel <= 1e-8, (b, s, obj_h[b, s], want)
    report("free_objective_rel")
