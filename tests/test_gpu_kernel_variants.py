"""The kernels that run after a solve -- sampling, evaluate_range, cost, the time gradient and the cost sweep --
against the oracle on every compiled variant their launchers pick (pytest -m gpu).

Each launcher chooses a kernel from the shape, the batch size, the SM count and pointer alignment.  The functions
`sample_variant`, `sweep_variant` and the `*_loops` predicates below restate those choices in Python, citing the
lines they restate; every case of the tables carries the variant it is meant to reach, a GPU test asserts that the
restatement on the device at hand agrees with the tag, and tests/test_kernel_variant_coverage.py (CPU) fails when
some variant has no case.  A threshold moved in a .cu file without the matching edit here therefore fails a test
instead of silently moving cases to another kernel.

Tolerances are those of helpers.py: samples SAMPLE_TOL absolute and 1e-11 relative to each derivative's scale,
sample instants and segment indices bit-exact, cost COST_TOL relative.  Where the f64 oracle's reference-order
arithmetic is itself off (N = 12, high derivatives, orders other than snap) the long-double oracle is the truth and
the allowance against the f64 oracle is widened by that oracle's distance from the truth."""
import ctypes as C

import numpy as np
import pytest

from helpers import COST_TOL, SAMPLE_TOL, random_batch, standard_mask, vertex_values

pytestmark = pytest.mark.gpu

ORDERS = (4, 6, 8, 10, 12)
B200_SMS = 148
MAX_DYNAMIC_SMEM = 227 * 1024                  # minsnap_launch.h: kMaxDynamicSmem
MEASURED = {}                                  # worst error per check, for the record


def record(key, value):
    MEASURED[key] = max(MEASURED.get(key, 0.0), float(value))


# ------------------------------------------------------------------------------------------
# Restatements of the launchers' choices
# ------------------------------------------------------------------------------------------
def sample_variant(N, K, D, n_deriv, B, offset8=False, sms=B200_SMS):
    """launch_sample_n, minsnap_sample.cu:239-314 -> (kernel, ND, grid, store).

    fast:     n_deriv <= 5 and 8 (2K + KDN + 1 + 4 (32 n_deriv D + 1)) bytes <= 96 KB       (:243-247)
    staged:   else 8 (2K + 4 32 n_deriv D) + 8 n_deriv KDN bytes <= 64 KB                    (:278-280)
    unstaged: else                                                                            (:281)
    grid:     M cut into chunks when B < 8 SMs, else one trajectory per CTA                 (:251, :287)
    store (fast kernel only, :226): 16-byte stores when the output is 16-byte aligned and a warp's run starts and
    ends on an even double; an odd row (n_deriv D odd) mixes the two paths, an 8-byte-offset output is all scalar."""
    per = n_deriv * D
    grid = "chunked" if B < 8 * sms else "per_trajectory"
    fast_bytes = 8 * (2 * K + K * D * N + 1 + 4 * (32 * per + 1))
    if n_deriv <= 5 and fast_bytes <= 96 * 1024:
        store = "scalar" if offset8 else ("vector" if per % 2 == 0 else "mixed")
        return ("fast", n_deriv, grid, store)
    base = 8 * (2 * K + 4 * 32 * per)
    staged = base + 8 * n_deriv * K * D * N
    if staged <= 64 * 1024:
        return ("staged", None, grid, None)
    assert base <= MAX_DYNAMIC_SMEM
    return ("unstaged", None, grid, None)


def _lane_slots(K, D):
    """fast::lane_slots, minsnap_standard_fast.cuh:204-214."""
    mA = (K - 1) // 2
    stored = mA - 1 if mA > 0 else 0
    return max((16 + 4 * D) * stored, 4 * D * stored + 12 * D)


def _warp_smem_doubles(K, D, global_slots, direct):
    """fast::warp_smem_doubles, minsnap_standard_fast.cuh:216-226."""
    slots = 0 if global_slots else (_lane_slots(K, D) * 32 + 1) & ~1
    if direct:
        return slots
    return slots + ((16 * (K + 1) * D + 1) & ~1) + ((16 * K + 1) & ~1)


def sweep_k_limit(D):
    """Largest K fast::inputs_fit admits (minsnap_standard_fast.cuh:852-859): the inputs of 16 problems staged."""
    K = 25
    while _warp_smem_doubles(K + 1, D, True, False) * 8 <= MAX_DYNAMIC_SMEM:
        K += 1
    return K


def sweep_variant(K, D, N=10, derivative=4):
    """launch_cost_sweep (minsnap_standard.cu:164-174) with fast::supported (minsnap_standard_fast.cuh:855-859) and
    fast::launch_d (:910-918): the two-lane kernel reading its inputs straight from global memory for K <= 24, the
    same kernel with its block storage in global memory up to the input-staging limit, else generic_route with
    fixed_div = S."""
    if N == 10 and derivative == 4 and 1 <= D <= 3 and K <= 24:
        return "direct"
    if N == 10 and derivative == 4 and 1 <= D <= 3 and K <= sweep_k_limit(D):
        return "global_slots"
    return "generic"


def sweep_warps_per_cta(K, D):
    """fast::launch_mode (minsnap_standard_fast.cuh:861-875): warps per CTA, direct mode."""
    per_warp = _warp_smem_doubles(K, D, False, True) * 8
    warps, best = 1, 0
    for w in range(1, 5):
        if per_warp * w > MAX_DYNAMIC_SMEM:
            break
        resident = min((228 * 1024) // (per_warp * w + 1024) * w, 8)
        if resident > best:
            best, warps = resident, w
    return warps


def sweep_loops(n_problems, K, D, sms=B200_SMS):
    """Grid capped at 256 CTAs per SM (minsnap_standard_fast.cuh:889-890): warps loop over the grid stride once
    there are more than SMs x 256 x warps x 16 problems."""
    return n_problems > sms * 256 * sweep_warps_per_cta(K, D) * 16


def evaluate_range_loops(B, sms=B200_SMS):
    """launch_evaluate_range (minsnap_sample.cu:407-408): 16 CTAs of 4 warps per SM at most, one warp a trajectory."""
    return B > sms * 16 * 4


def cost_loops(B, sms=B200_SMS):
    """launch_cost (minsnap_general.cu:541-543): 16 CTAs of 8 warps per SM at most, one warp a trajectory."""
    return B > sms * 16 * 8


# ------------------------------------------------------------------------------------------
# Case tables
# ------------------------------------------------------------------------------------------
# (N, K, D, n_deriv, B, M, offset8) -> the variant of sample_variant it is meant to reach
SAMPLE_CASES = []


def _sample_case(N, K, D, nd, B, M, offset8=False):
    SAMPLE_CASES.append(((N, K, D, nd, B, M, offset8), sample_variant(N, K, D, nd, B, offset8)))


for _N in ORDERS:
    for _nd in range(1, 6):
        _sample_case(_N, 5, 3, _nd, 4, 100)                        # fast, every (N, ND); ND > N at N = 4
for _N, _nd in ((4, 6), (6, 8), (8, 12), (10, 6), (10, 12), (12, 8), (12, 14)):
    _sample_case(_N, 3, 2, _nd, 3, 300)                            # staged; rows k >= N at N = 4, 10, 12
for _N in ORDERS:
    _sample_case(_N, 200, 3, 6, 2, 300)                            # unstaged at every N
_sample_case(10, 50, 3, 6, 3, 500)                                 # unstaged: staged tables ~91 KB
_sample_case(10, 400, 3, 5, 2, 700)                                # unstaged: fast tables > 96 KB
for _D in (1, 2, 3, 4):
    for _K in (16, 17, 40):
        _sample_case(10, _K, _D, 5, 3, 777)                        # linear scan / binary search of find_segment
for _M in (1, 31, 32, 33, 1000):
    _sample_case(8, 7, 3, 4, 3, _M)
_sample_case(10, 10, 3, 5, 8 * B200_SMS - 1, 64)                   # largest chunked batch
_sample_case(10, 10, 3, 5, 8 * B200_SMS, 64)                       # one trajectory per CTA
_sample_case(6, 20, 3, 4, 8 * B200_SMS + 50, 100)                  # one trajectory per CTA, binary search
_sample_case(12, 3, 2, 7, 8 * B200_SMS + 3, 200)                   # staged, one trajectory per CTA
_sample_case(4, 200, 3, 6, 8 * B200_SMS + 1, 40)                   # unstaged, one trajectory per CTA
_sample_case(10, 10, 3, 5, 5, 333, True)                           # odd row, 8-byte-offset output
_sample_case(10, 10, 2, 5, 5, 333, True)                           # even row, 8-byte-offset output

# (K, D, S, B, with end derivatives) -> sweep_variant, N = 10 snap
SWEEP_CASES = []
for _D in (1, 2, 3):
    for _K in (1, 2, 3, 4, 10, 24, 25, 64, 200):
        # B S ragged (< 16 too) and a multiple of 16; fewer problems at K = 200, where an oracle solve takes 0.3 s
        for _S, _B in ((1, 5), (7, 3), (16, 2), (1, 48)) if _K < 200 else ((7, 2), (16, 1)):
            for _ends in (False, True):
                SWEEP_CASES.append(((_K, _D, _S, _B, _ends), sweep_variant(_K, _D)))
# (N, derivative, D) on generic_route
SWEEP_GENERIC_CASES = [(6, 2, 3), (8, 3, 3), (12, 5, 3), (10, 2, 3), (10, 3, 3), (10, 4, 4), (10, 4, 5)]

# batch sizes that make warps loop over the grid stride on a B200 (checked on the device and by the coverage test)
EVALUATE_RANGE_LOOP_B = 2 * 64 * B200_SMS + 37
COST_LOOP_B = 20000
SWEEP_LOOP_K, SWEEP_LOOP_D, SWEEP_LOOP_S = 10, 3, 64
SWEEP_LOOP_B = 2 * B200_SMS * 256 * sweep_warps_per_cta(SWEEP_LOOP_K, SWEEP_LOOP_D) * 16 // SWEEP_LOOP_S + 7


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def offset_view(torch, a):
    """A device copy of `a` whose data pointer is 8 bytes past a 16-byte boundary."""
    a = np.ascontiguousarray(a, np.float64)
    buf = torch.empty(a.size + 1, dtype=torch.float64, device="cuda")
    v = buf[1:].view(a.shape)
    v.copy_(torch.from_numpy(a))
    assert v.data_ptr() % 16 == 8
    return v


def random_times(rng, B, K, lo=0.5, hi=1.5):
    return rng.uniform(lo, hi, (B, K))


def random_coeffs(rng, times, D, N):
    """c_j ~ N(0, 1) / (j! T^j): derivative k stays O(T^-k) over the segment.  Without the j! the high derivatives
    at N = 12 reach 1e8, where the f64 oracle's own Horner is 4e-6 off the long-double truth."""
    B, K = times.shape
    fact = np.cumprod(np.concatenate([[1.0], np.arange(1.0, N)]))
    return rng.normal(size=(B, K, D, N)) / (fact * times[:, :, None, None] ** np.arange(N))


def solved_coeffs(oracle, pos, times, N, derivative, ends=None):
    """The f64 oracle's solve of the standard mask (rest-to-rest, or the given end derivatives [B][2][h-1][D])."""
    B, K1, D = pos.shape
    K = K1 - 1
    mask = standard_mask(K, N)
    out = np.empty((B, K, D, N))
    for b in range(B):
        out[b] = oracle.solve(N, K, D, derivative, mask, end_values(pos[b], N, None if ends is None else ends[b]),
                              times[b])["coeffs"]
    return out


def end_values(pos, N, ends=None):
    v = vertex_values(pos, N)
    if ends is not None:
        v[0, 1:] = ends[0]
        v[-1, 1:] = ends[1]
    return v


def seq_total(t):
    total = 0.0
    for x in t:
        total += x
    return total


def check_samples(got, want, truth=None, key="sample"):
    """got / want / truth [M][n_deriv][D]: SAMPLE_TOL absolute and 1e-11 relative to each derivative's scale."""
    def errs(a, ref):
        ref = np.asarray(ref, np.float64)
        err = np.abs(a - ref)
        scale = np.abs(ref).max(axis=(0, 2))
        rel = np.where(scale > 0, err.max(axis=(0, 2)) / np.where(scale > 0, scale, 1.0), 0.0)
        return float(err.max(initial=0.0)), float(rel.max(initial=0.0))
    slack_a, slack_r = 0.0, 0.0
    if truth is not None:
        a, r = errs(got, truth)
        record(key + "_abs_vs_ld", a)
        record(key + "_rel_vs_ld", r)
        assert a <= SAMPLE_TOL and r <= 1e-11, (a, r)
        slack_a, slack_r = errs(want, truth)
    a, r = errs(got, want)
    record(key + "_abs", a)
    record(key + "_rel", r)
    assert a <= SAMPLE_TOL + slack_a and r <= 1e-11 + slack_r, (a, r, slack_a, slack_r)


def rows_to_check(B, n=8):
    return sorted({0, B - 1, *np.linspace(0, B - 1, n).astype(int).tolist()})


# ------------------------------------------------------------------------------------------
# sampling
# ------------------------------------------------------------------------------------------
def test_variant_tags_hold_on_this_device(torch_cuda):
    sms = torch_cuda.cuda.get_device_properties(0).multi_processor_count
    for args, tag in SAMPLE_CASES:
        N, K, D, nd, B, M, off = args
        assert sample_variant(N, K, D, nd, B, off, sms) == tag, (args, sms)
    for args, tag in SWEEP_CASES:
        assert sweep_variant(args[0], args[1]) == tag
    assert sms == B200_SMS, "the batch sizes of the grid-stride cases are set for %d SMs" % B200_SMS


@pytest.mark.parametrize("case", SAMPLE_CASES, ids=lambda c: "N%d-K%d-D%d-nd%d-B%d-M%d%s" % (*c[0][:6], "-off8" * c[0][6]))
def test_sample_uniform_variants(ms, oracle, oracle_ld, torch_cuda, case):
    torch = torch_cuda
    (N, K, D, nd, B, M, offset8), tag = case
    rng = np.random.default_rng(hash((N, K, D, nd, B, M)) % 2**32)
    times = random_times(rng, B, K)
    if K >= 16 and D == 2:
        times[:, K // 2] = 0.0                                     # a zero-length segment is never chosen
    if K == 7 and D == 3 and B == 3:
        times[1, 3] = 0.0
    coeffs = random_coeffs(rng, times, D, N)
    c_d, t_d = dev(torch, coeffs), dev(torch, times)
    out = offset_view(torch, np.zeros((B, M, nd, D))) if offset8 else None
    out, t = ms.sample_uniform(c_d, t_d, M, nd, out=out, want_times=True)
    out, t = out.cpu().numpy(), t.cpu().numpy()
    # N = 12, high derivatives: the f64 oracle's reference-order Horner is itself off; long double is the truth
    use_truth = N == 12 or nd > 5
    for b in rows_to_check(B) if B > 16 else range(B):
        assert np.array_equal(t[b], np.arange(M) * (seq_total(times[b]) / M))
        want = oracle.trajectory_sample(coeffs[b], times[b], t[b], nd)
        truth = oracle_ld.trajectory_sample(coeffs[b], times[b], t[b], nd) if use_truth else None
        check_samples(out[b], want, truth, "sample_" + tag[0])
        if nd > N:
            assert (out[b, :, N:] == 0).all()


def sample_at_instants(times):
    ends = np.cumsum(times, axis=1)                                # left-to-right, as the kernels accumulate
    B = times.shape[0]
    return np.concatenate([np.zeros((B, 1)), ends, np.nextafter(ends, -np.inf), np.nextafter(ends, np.inf),
                           np.full((B, 1), -0.25), ends[:, -1:] + 1.0, np.full((B, 1), np.inf),
                           np.full((B, 1), np.nan), np.linspace(0.0, ends[:, -1], 40).T], axis=1)


@pytest.mark.parametrize("N,K,nd", [(4, 5, 5), (10, 12, 5), (10, 20, 5), (12, 33, 3), (8, 20, 7), (10, 17, 12)])
def test_sample_at_variants(ms, oracle, torch_cuda, N, K, nd):
    """Per-trajectory rows and a shared row (stride 0) at instants on every vertex, one ulp either side of it, at 0,
    negative, past the end, +inf and NaN; the segment index bit-exact against the oracle's (find_segment's linear
    scan for K <= 16, its binary search above).  The f64 oracle is the reference here: the long-double build
    accumulates the segment ends in long double and so picks other segments one ulp from a vertex."""
    torch = torch_cuda
    D, B = 3, 5
    rng = np.random.default_rng(N * 100 + K)
    times = random_times(rng, B, K)
    times[2, K // 2] = 0.0
    coeffs = random_coeffs(rng, times, D, N)
    c_d, t_d = dev(torch, coeffs), dev(torch, times)
    t = sample_at_instants(times)
    out, seg = ms.sample_at(c_d, t_d, dev(torch, t), nd, want_segment=True)
    out, seg = out.cpu().numpy(), seg.cpu().numpy()
    shared = t[2]
    out_s, seg_s = ms.sample_at(c_d, t_d, dev(torch, shared), nd, want_segment=True)
    out_s, seg_s = out_s.cpu().numpy(), seg_s.cpu().numpy()
    for b in range(B):
        for tt, o, sg in ((t[b], out[b], seg[b]), (shared, out_s[b], seg_s[b])):
            want_seg = np.array([oracle.trajectory_evaluate(coeffs[b], times[b], x, 0)[1] for x in tt])
            assert np.array_equal(sg, want_seg)
            want = oracle.trajectory_sample(coeffs[b], times[b], tt, nd)
            assert (o[want_seg < 0] == 0).all()
            check_samples(o, want, key="sample_at")


@pytest.mark.parametrize("N", ORDERS)
def test_sample_solved_trajectories(ms, oracle, oracle_ld, torch_cuda, N):
    """One solved batch per order (the general solve of the standard mask, minimum derivative h - 1)."""
    torch = torch_cuda
    K, B, M = 9, 6, 500
    pos, times = random_batch(oracle, B, K, seed=31 + N)
    coeffs = solved_coeffs(oracle, pos, times, N, N // 2 - 1)
    out = ms.sample_uniform(dev(torch, coeffs), dev(torch, times), M, 5).cpu().numpy()
    for b in range(B):
        t = np.arange(M) * (seq_total(times[b]) / M)
        want = oracle.trajectory_sample(coeffs[b], times[b], t, 5)
        truth = oracle_ld.trajectory_sample(coeffs[b], times[b], t, 5) if N == 12 else None
        check_samples(out[b], want, truth, "sample_solved")


# ------------------------------------------------------------------------------------------
# evaluate_range
# ------------------------------------------------------------------------------------------
def evaluate_range_raw(ms, torch, coeffs_d, times_d, t_start, t_end, dt, derivative, max_samples, sentinel=-7.5):
    """minsnap_evaluate_range through the C ABI into buffers pre-filled with a sentinel (the wrapper zero-fills)."""
    B, K, D, N = coeffs_d.shape
    out = torch.full((B, max_samples, D), sentinel, dtype=torch.float64, device="cuda")
    t_out = torch.full((B, max_samples), sentinel, dtype=torch.float64, device="cuda")
    count = torch.full((B,), -1, dtype=torch.int32, device="cuda")
    p = lambda x: C.c_void_p(x.data_ptr())
    rc = ms.load().minsnap_evaluate_range(B, K, D, N, p(coeffs_d), p(times_d), t_start, t_end, dt, derivative,
                                          max_samples, p(out), p(t_out), p(count),
                                          C.c_void_p(torch.cuda.current_stream().cuda_stream))
    ms.capi.check(rc, "minsnap_evaluate_range")
    return out.cpu().numpy(), t_out.cpu().numpy(), count.cpu().numpy()


def check_range(oracle, coeffs, times, t_start, t_end, dt, derivative, max_samples, out, t_out, count, rows,
                sentinel=-7.5):
    for b in rows:
        want, want_t = oracle.trajectory_evaluate_range(coeffs[b], times[b], t_start, t_end, dt, derivative, 1 << 14)
        n = len(want_t)
        assert n < 1 << 14
        assert count[b] == n, (b, count[b], n)
        m = min(n, max_samples)
        assert np.array_equal(t_out[b, :m], want_t[:m])              # sequential accumulation, bit-exact
        err = np.abs(out[b, :m] - want[:m]).max(initial=0.0)
        record("evaluate_range_abs", err)
        assert err <= SAMPLE_TOL
        assert (out[b, m:] == sentinel).all() and (t_out[b, m:] == sentinel).all()


@pytest.mark.parametrize("D", [1, 3])
@pytest.mark.parametrize("N", ORDERS)
def test_evaluate_range_variants(ms, oracle, torch_cuda, N, D):
    """Derivatives 0 .. N + 1; t_start at 0, inside, exactly on a segment's end, at and past the total; t_end past
    the end; dt longer than some segments (the walker skips them) and short enough for several 32-sample batches;
    max_samples below the reference's count (count still reports the reference's count, nothing is written past
    max_samples)."""
    torch = torch_cuda
    K, B = 6, 4
    rng = np.random.default_rng(7 * N + D)
    times = random_times(rng, B, K, 0.2, 1.5)
    times[:, 2] = 0.05                                             # shorter than every dt below but the first
    coeffs = random_coeffs(rng, times, D, N)
    c_d, t_d = dev(torch, coeffs), dev(torch, times)
    ends = np.cumsum(times[0])
    total = ends[-1]
    for derivative in sorted({0, 1, N // 2, N - 1, N, N + 1}):
        for t_start in (0.0, 0.37 * total, ends[1], ends[2], total, total + 0.5):
            for dt, t_end in ((0.013, total + 0.5), (0.3, 0.8 * total), (1.1, total + 3.0)):
                n_ref = len(oracle.trajectory_evaluate_range(coeffs[0], times[0], t_start, t_end, dt, derivative,
                                                             1 << 14)[1])
                for max_samples in sorted({n_ref + 3, max(n_ref // 2, 1)}):
                    out, t_out, count = evaluate_range_raw(ms, torch, c_d, t_d, t_start, t_end, dt, derivative,
                                                           max_samples)
                    check_range(oracle, coeffs, times, t_start, t_end, dt, derivative, max_samples, out, t_out,
                                count, range(B))


def test_evaluate_range_grid_stride(ms, oracle, torch_cuda):
    """More trajectories than warps in the capped grid: warps loop over the grid stride."""
    torch = torch_cuda
    B, K, N, D = EVALUATE_RANGE_LOOP_B, 5, 10, 3
    assert evaluate_range_loops(B)
    rng = np.random.default_rng(3)
    times = random_times(rng, B, K)
    coeffs = random_coeffs(rng, times, D, N)
    dt, t_end = 0.021, 3.0
    out, t_out, count = evaluate_range_raw(ms, torch, dev(torch, coeffs), dev(torch, times), 0.25, t_end, dt, 2, 200)
    check_range(oracle, coeffs, times, 0.25, t_end, dt, 2, 200, out, t_out, count, rows_to_check(B, 300))


# ------------------------------------------------------------------------------------------
# cost and time gradient at every (N, derivative)
# ------------------------------------------------------------------------------------------
ORDER_DERIVATIVES = [(N, delta) for N in ORDERS for delta in range(N // 2)]


def solved_set(oracle, N, delta, D, K, B, seed):
    pos, times = random_batch(oracle, B, K, D, seed=seed)
    return solved_coeffs(oracle, pos, times, N, delta), times


def cost_terms(oracle_ld, N, delta, coeffs, times):
    """0.5 sum_seg sum_dim |c|^T |Q(T)| |c|: the scale of the rounding error of computeCost."""
    return float(sum(0.5 * np.abs(c) @ np.abs(oracle_ld.cost_matrix(N, delta, T)) @ np.abs(c)
                     for seg, T in zip(coeffs, times) for c in seg))


@pytest.mark.parametrize("N,delta", ORDER_DERIVATIVES)
def test_cost_every_order(ms, oracle, oracle_ld, torch_cuda, N, delta):
    torch = torch_cuda
    for D in (1, 3, 5):
        for K in (1, 7, 33):
            coeffs, times = solved_set(oracle, N, delta, D, K, 3, seed=1000 * N + 100 * delta + 10 * D + K)
            got = ms.cost(dev(torch, coeffs), dev(torch, times), delta).cpu().numpy()
            want = np.array([float(oracle.compute_cost(N, K, D, delta, c, t)) for c, t in zip(coeffs, times)])
            truth = np.array([oracle_ld.compute_cost(N, K, D, delta, c, t) for c, t in zip(coeffs, times)])
            terms = np.array([cost_terms(oracle_ld, N, delta, c, t) for c, t in zip(coeffs, times)])
            # c^T Q c of a minimum-derivative solution cancels (at N = 12, derivative 0 the f64 oracle is 7.8e-5 off
            # the long-double truth): the bar is COST_TOL relative or 1e-12 of the magnitudes of the terms (measured on
            # a B200: 8.7e-17 of them at worst, 1.5e-5 relative at N = 12, derivative 0)
            bar = np.maximum(COST_TOL * np.abs(truth), 1e-12 * terms)
            record("cost_rel_vs_ld", np.abs(got / truth - 1.0).max())
            record("cost_err_rel_to_terms", (np.abs(got - truth) / terms).max())
            assert (np.abs(got - truth) <= bar).all(), (D, K, got, truth, terms)
            assert (np.abs(got - want) <= bar + np.abs(want - truth)).all()


def test_cost_random_coefficients_and_grid_stride(ms, oracle, torch_cuda):
    """Random (non-optimal) coefficients make c^T Q c a sum of large cancelling terms: the two summation orders agree
    to ~1e-10 (test_coeffs_from_constraints_and_cost), so the bar is 1e-9.  B = 20,000 is more trajectories than
    warps in the capped grid."""
    torch = torch_cuda
    B, K, D, N = COST_LOOP_B, 7, 3, 10
    assert cost_loops(B)
    rng = np.random.default_rng(17)
    times = random_times(rng, B, K)
    coeffs = random_coeffs(rng, times, D, N)
    got = ms.cost(dev(torch, coeffs), dev(torch, times), 4).cpu().numpy()
    for b in rows_to_check(B, 300):
        want = float(oracle.compute_cost(N, K, D, 4, coeffs[b], times[b]))
        record("cost_random_rel", abs(got[b] / want - 1.0))
        assert abs(got[b] / want - 1.0) <= 1e-9


def gradient_reference(oracle_ld, coeffs, times, delta, increment, w_d, w_t):
    """getCostAndGradientTime restated in long double for one trajectory: d_seg holds derivatives 0..h-1 at both
    ends of the segment, q(T') = sum_dim d_seg^T H(T') d_seg, gradient = w_d (q(T+) - q(T-)) / (2 inc) + w_t, with
    the reference's clamp T <= 0.1 -> T+- = 0.1.  Returns (gradient, q(T), and the scales of their rounding errors:
    w_d (a(T+) + a(T-)) / (2 inc) and a(T), with a(T') = sum_dim |d_seg|^T |H(T')| |d_seg| the sum of the
    magnitudes of the terms the kernel adds)."""
    K, D, N = coeffs.shape
    h = N // 2
    grad, q0, g_scale, q_scale = np.zeros(K), np.zeros(K), np.zeros(K), np.zeros(K)
    for i in range(K):
        T = float(times[i])
        Tm, Tp = (0.1, 0.1) if T <= 0.1 else (T - increment, T + increment)
        H = [oracle_ld.segment_hessian(N, delta, x) for x in (T, Tm, Tp)]
        q = [np.longdouble(0)] * 3
        a = [np.longdouble(0)] * 3
        for dim in range(D):
            c = coeffs[i, dim]
            d = np.array([oracle_ld.polynomial_evaluate(c, 0.0, k) for k in range(h)] +
                         [oracle_ld.polynomial_evaluate(c, T, k) for k in range(h)], np.longdouble)
            q = [qq + d @ Hx @ d for qq, Hx in zip(q, H)]
            a = [aa + np.abs(d) @ np.abs(Hx) @ np.abs(d) for aa, Hx in zip(a, H)]
        inc2 = np.longdouble(2.0) * np.longdouble(increment)
        grad[i] = float(np.longdouble(w_d) * ((q[2] - q[1]) / inc2) + np.longdouble(w_t))
        q0[i] = float(q[0])
        g_scale[i] = float(np.longdouble(w_d) * (a[2] + a[1]) / inc2)
        q_scale[i] = float(a[0])
    return grad, q0, g_scale, q_scale


@pytest.mark.parametrize("N,delta", ORDER_DERIVATIVES)
def test_time_gradient_every_order(ms, oracle, oracle_ld, torch_cuda, N, delta):
    """The kernel raises T' to powers m + 1 - 2 delta, negative at low N or high delta.  Its sums of
    d_r d_s H_rs T'^m cancel (at N = 12, derivative 0 by eight digits), so the gradient and q(T) are bounded
    relative to the sum of the magnitudes of their terms (gradient_reference).  Measured on a B200: 1.2e-11 for
    both at worst (N = 12); a float64 model of the kernel's sums reaches 6e-12, so the bar is 1e-10."""
    torch = torch_cuda
    inc, w_d, w_t = 0.1, 0.1, 1.0
    worst = []
    for D in (1, 3, 5):
        for K in (1, 7, 33):
            coeffs, times = solved_set(oracle, N, delta, D, K, 2, seed=2000 * N + 100 * delta + 10 * D + K)
            times[-1, 0] = 0.1                                     # the clamp: gradient exactly w_t
            if K > 1:
                times[-1, 1] = 0.05
            grad, seg = ms.time_gradient(dev(torch, coeffs), dev(torch, times), inc, w_d, w_t, derivative=delta,
                                         want_segment_cost=True)
            grad, seg = grad.cpu().numpy(), seg.cpu().numpy()
            for b in range(coeffs.shape[0]):
                g_ref, q_ref, g_scale, q_scale = gradient_reference(oracle_ld, coeffs[b], times[b], delta, inc, w_d,
                                                                    w_t)
                g_err = float((np.abs(grad[b] - g_ref) / g_scale).max())
                q_err = float((np.abs(seg[b] - q_ref) / q_scale).max())
                record("time_gradient_rel_to_terms", g_err)
                record("segment_cost_rel_to_terms", q_err)
                worst.append((g_err, q_err, D, K, b))
            assert grad[-1, 0] == w_t and (K == 1 or grad[-1, 1] == w_t)
    assert max(w[0] for w in worst) <= 1e-10, max(worst)
    assert max(w[1] for w in worst) <= 1e-10, max(worst, key=lambda w: w[1])


def test_time_objective_generic_route(ms, oracle, oracle_ld, torch_cuda):
    """minsnap_time_objective on a shape cost_sweep sends to generic_route: add_time_penalty after it."""
    torch = torch_cuda
    N, delta, K, B, S, penalty = 8, 3, 6, 3, 4, 7.5
    assert sweep_variant(K, 3, N, delta) == "generic"
    rng = np.random.default_rng(5)
    pos, times = random_batch(oracle, B, K, seed=61)
    sweep = times[:, None, :] * rng.uniform(0.8, 1.2, (B, S, K))
    obj, cost = ms.time_objective(dev(torch, pos), dev(torch, sweep), penalty, N=N, derivative=delta, want_cost=True)
    obj, cost = obj.cpu().numpy(), cost.cpu().numpy()
    for b in range(B):
        for s in range(S):
            total = seq_total(sweep[b, s])
            want = float(oracle_ld.solve(N, K, 3, delta, standard_mask(K, N), vertex_values(pos[b], N),
                                         sweep[b, s])["cost"])
            assert abs(cost[b, s] / want - 1.0) <= COST_TOL
            assert abs(obj[b, s] / (cost[b, s] + total * total * penalty) - 1.0) <= 1e-15


# ------------------------------------------------------------------------------------------
# cost_sweep
# ------------------------------------------------------------------------------------------
def sweep_inputs(oracle, rng, B, S, K, D, N=10, ends=False, seed=0):
    pos, times = random_batch(oracle, B, K, D, seed=seed)
    sweep = times[:, None, :] * rng.uniform(0.8, 1.25, (B, S, K))
    e = rng.normal(size=(B, 2, N // 2 - 1, D)) if ends else None
    return pos, sweep, e


def sweep_reference(orc, pos, sweep, ends, N, delta, b, s):
    K = sweep.shape[2]
    return float(orc.solve(N, K, pos.shape[2], delta, standard_mask(K, N),
                           end_values(pos[b], N, None if ends is None else ends[b]), sweep[b, s])["cost"])


def check_sweep(oracle, cost, pos, sweep, ends, N=10, delta=4, truth=None, skip=(), key="sweep"):
    B, S, _ = sweep.shape
    for b in range(B):
        for s in range(S):
            if (b, s) in skip:
                continue
            want = sweep_reference(oracle, pos, sweep, ends, N, delta, b, s)
            slack = 0.0
            if truth is not None:
                t = sweep_reference(truth, pos, sweep, ends, N, delta, b, s)
                slack = abs(want / t - 1.0)
                record(key + "_rel_vs_ld", abs(cost[b, s] / t - 1.0))
                assert abs(cost[b, s] / t - 1.0) <= max(COST_TOL, 2.0 * slack), (b, s, slack)
            record(key + "_rel", abs(cost[b, s] / want - 1.0))
            assert abs(cost[b, s] / want - 1.0) <= COST_TOL + 3.0 * slack, (b, s)


@pytest.mark.parametrize("case", SWEEP_CASES, ids=lambda c: "%s-K%d-D%d-S%d-B%d%s" % (c[1], *c[0][:4], "-ends" * c[0][4]))
def test_cost_sweep_two_lane_variants(ms, oracle, torch_cuda, case):
    """Direct reads (K <= 24) and global-memory slots (K > 24) against the oracle, with and without end derivatives
    (the K = 1, 2, 3 boundary couplings read them through rec = prob / S)."""
    torch = torch_cuda
    (K, D, S, B, ends), tag = case
    rng = np.random.default_rng(K * 1000 + D * 100 + S * 10 + B + ends)
    pos, sweep, e = sweep_inputs(oracle, rng, B, S, K, D, ends=ends, seed=K * 7 + D)
    cost = ms.cost_sweep(dev(torch, pos), dev(torch, sweep), None if e is None else dev(torch, e)).cpu().numpy()
    check_sweep(oracle, cost, pos, sweep, e, key="sweep_" + tag)


@pytest.mark.parametrize("N,delta,D", SWEEP_GENERIC_CASES)
def test_cost_sweep_generic_variant(ms, oracle, oracle_ld, torch_cuda, N, delta, D):
    torch = torch_cuda
    K = 5
    assert sweep_variant(K, D, N, delta) == "generic"
    rng = np.random.default_rng(N * 10 + delta + D)
    for S, B in ((1, 3), (6, 2)):
        for ends in (False, True):
            pos, sweep, e = sweep_inputs(oracle, rng, B, S, K, D, N, ends, seed=N + D)
            cost = ms.cost_sweep(dev(torch, pos), dev(torch, sweep), None if e is None else dev(torch, e), N=N,
                                 derivative=delta).cpu().numpy()
            check_sweep(oracle, cost, pos, sweep, e, N, delta, truth=oracle_ld, key="sweep_generic")


@pytest.mark.parametrize("variant,K,N,delta", [("direct", 10, 10, 4), ("global_slots", 64, 10, 4),
                                               ("generic", 6, 8, 3)])
def test_cost_sweep_status_and_unaligned_times(ms, oracle, oracle_ld, torch_cuda, variant, K, N, delta):
    """A zero and a negative segment time flag exactly their own (b, s) with bit 2; times read through an 8-byte-
    offset view give the oracle's costs."""
    torch = torch_cuda
    D, B, S = 3, 3, 7
    assert sweep_variant(K, D, N, delta) == variant
    rng = np.random.default_rng(K)
    pos, sweep, e = sweep_inputs(oracle, rng, B, S, K, D, N, ends=True, seed=K)
    bad = sweep.copy()
    bad[1, 2, K // 2] = 0.0
    bad[2, 5, 0] = -0.5
    cost, st = ms.cost_sweep(dev(torch, pos), dev(torch, bad), dev(torch, e), N=N, derivative=delta, want_status=True)
    st = st.cpu().numpy()
    flagged = {(int(b), int(s)) for b, s in zip(*np.nonzero(st & 2))}
    assert flagged == {(1, 2), (2, 5)}, flagged
    assert (np.delete(st.ravel(), [1 * S + 2, 2 * S + 5]) == 0).all()
    truth = oracle_ld if variant == "generic" else None
    check_sweep(oracle, cost.cpu().numpy(), pos, bad, e, N, delta, truth, skip={(1, 2), (2, 5)}, key="sweep_status")
    cost_u = ms.cost_sweep(offset_view(torch, pos), offset_view(torch, sweep), offset_view(torch, e), N=N,
                           derivative=delta).cpu().numpy()
    check_sweep(oracle, cost_u, pos, sweep, e, N, delta, truth, key="sweep_unaligned")


@pytest.mark.parametrize("D", [1, 2, 3])
def test_cost_sweep_longest_staged_chain(ms, torch_cuda, D):
    """The largest K the input staging admits at each D (the oracle's dense solve takes minutes there): against
    solve_standard with the cost on the flattened problem, another kernel, at 1e-10."""
    torch = torch_cuda
    K = sweep_k_limit(D)
    assert sweep_variant(K, D) == "global_slots" and sweep_variant(K + 1, D) == "generic"
    B, S = 3, 5
    rng = np.random.default_rng(D)
    pos = np.cumsum(rng.uniform(0.3, 2.0, (B, K + 1, D)) * rng.choice([-1.0, 1.0], (B, K + 1, D)), axis=1)
    ends = rng.normal(size=(B, 2, 4, D))
    sweep = rng.uniform(0.5, 1.5, (B, S, K))
    pos_d, sweep_d, ends_d = dev(torch, pos), dev(torch, sweep), dev(torch, ends)
    cost = ms.cost_sweep(pos_d, sweep_d, ends_d)
    flat = ms.solve_standard(pos_d.repeat_interleave(S, 0).contiguous(), sweep_d.reshape(B * S, K).contiguous(),
                             end_derivatives=ends_d.repeat_interleave(S, 0).contiguous(), want_cost=True)
    assert (flat["status"] == 0).all()
    rel = float((cost.reshape(-1) / flat["cost"] - 1.0).abs().max())
    record("sweep_longest_vs_solve", rel)
    assert rel <= 1e-10


def test_cost_sweep_grid_stride(ms, oracle, torch_cuda):
    """More problems than the capped grid's warps take in one pass (direct variant): against solve_standard with the
    cost on the flattened problem at 1e-10, and a few hundred rows against the oracle."""
    torch = torch_cuda
    K, D, S, B = SWEEP_LOOP_K, SWEEP_LOOP_D, SWEEP_LOOP_S, SWEEP_LOOP_B
    assert sweep_variant(K, D) == "direct" and sweep_loops(B * S, K, D)
    pos = ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], 4242)
    pos_d = dev(torch, pos)
    base = ms.estimate_segment_times(pos_d, 3.0, 5.0)
    g = torch.Generator(device="cuda").manual_seed(3)
    sweep_d = base[:, None, :] * (0.8 + 0.45 * torch.rand((B, S, K), generator=g, device="cuda", dtype=torch.float64))
    cost = ms.cost_sweep(pos_d, sweep_d)
    flat = ms.solve_standard(pos_d.repeat_interleave(S, 0), sweep_d.reshape(B * S, K), want_cost=True)
    rel = float((cost.reshape(-1) / flat["cost"] - 1.0).abs().max())
    record("sweep_grid_stride_vs_solve", rel)
    # measured on a B200: 1.08e-10 at worst over these 1.2 M problems (times drawn 0.8x - 1.25x the estimate), and
    # both kernels within 2.1e-10 of the oracle over the direct-variant cases, so the bar is 1e-9
    assert rel <= 1e-9
    del flat
    rng = np.random.default_rng(8)
    rows = np.unique(np.concatenate([[0, B * S - 1], rng.choice(B * S, 300, replace=False)]))
    cost_h = cost.reshape(-1)[torch.from_numpy(rows).cuda()].cpu().numpy()
    times_h = sweep_d.reshape(B * S, K)[torch.from_numpy(rows).cuda()].cpu().numpy()
    mask = standard_mask(K)
    for r, c, t in zip(rows, cost_h, times_h):
        want = float(oracle.solve(10, K, D, 4, mask, vertex_values(pos[r // S]), t)["cost"])
        record("sweep_grid_stride_rel", abs(c / want - 1.0))
        assert abs(c / want - 1.0) <= COST_TOL
