"""minsnap_solve_standard against the oracle on every kernel instantiation and output option behind it
(pytest -m gpu).

The route of each case (tm, pair, pair_long, bcr, chunked, general) comes from the real header through the route
binary of tests/test_standard_routes.py.  Inside a route, the launcher's choice is restated in Python with the lines
it restates: `tm_instantiation`, `tm_ctas` (from the registers cuobjdump reports) and `tm_grid_mode`; `pair_warps`
and `pair_loops`; `bcr_threads` and `bcr_resident`; `chunk_segments` and `chunked_ranges`; `general_solve_warps`.
`variant` gives the variant every case reaches, a GPU test checks it against the device at hand, and
tests/test_kernel_variant_coverage.py (CPU) fails when a variant has no case.

Truth and bars (helpers.py):
  * coefficients COEFF_TOL per polynomial against the long-double truth (helpers.banded_ld_solve, or oracle_ld.solve
    for short chains off N = 10 snap); for N = 10 snap and K <= 64 also against the f64 oracle (oracle.solve), with
    the allowance of compare_with_oracle: twice the f64 oracle's own distance from the truth;
  * cost COST_TOL; free derivatives 1e-8 of each trajectory's largest; device times 1e-14 relative to
    oracle.estimate_segment_times; status exact;
  * the coefficients of one instantiation are the same bits whether or not status and times_out are requested;
    another instantiation of the same shape (cost and extras flipped, tm against pair) agrees within 1e-10.
Rows checked: the first, the last, the last partial batch of 16 and an even spread, at most ~64 per case."""
import ctypes as C
import functools
import os
import re
import subprocess
import sys
import zlib
from collections import namedtuple

import numpy as np
import pytest

import test_gpu_collision_walk as W
from helpers import BASE_SEED, COEFF_TOL, COST_TOL, banded_ld_solve, standard_mask, vertex_values
from test_gpu_kernel_variants import B200_SMS, MAX_DYNAMIC_SMEM, _warp_smem_doubles
from test_standard_routes import run_routes

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
V_MAX, A_MAX = 3.0, 5.0
MEASURED = {}                                  # worst error per bar, for the record
NAN_BITS = np.int64(0x7FF8DEADBEEF0001)


def record(key, value):
    MEASURED[key] = max(MEASURED.get(key, 0.0), float(value))


# ------------------------------------------------------------------------------------------
# Restatements of the launchers' choices
# ------------------------------------------------------------------------------------------
def tm_instantiation(K, D, cost, extras):
    """tm::launch_d, minsnap_standard_tm.cuh:843-850: solve_standard_tm_kernel<D, kCost, kExtras, kOdd>, extras when
    end derivatives are given or free values requested."""
    return (D, bool(cost), bool(extras), K % 2 == 1)


def tmem_columns(K, D):
    """tm::tmem_columns, minsnap_standard_tm.cuh:158-170."""
    mA = (K - 1) // 2
    need = (mA - 1 if mA > 0 else 0) * (32 + 8 * D)
    cols = 32
    while cols < need:
        cols <<= 1
    return cols


def tm_smem_bytes(K, D):
    """WarpSmem<D>(K).total x 8 bytes x 4 warps, minsnap_standard_tm.cuh:175-186 and :838."""
    pos = (16 * (K + 1) * D + 15) & ~15
    tim = (16 * K + 15) & ~15
    return (2 * (pos + tim) + 2 * 2 * 16 * D * 10) * 8 * 4


@functools.lru_cache(maxsize=None)
def tm_resources():
    """{instantiation: (registers, static shared bytes)} of the built library (cuobjdump -res-usage)."""
    from mav_trajectory_generation_cmake_b200 import build
    build.build()
    text = subprocess.run(["cuobjdump", "-res-usage", build.LIB], capture_output=True, text=True, check=True).stdout
    res = {}
    for m in re.finditer(r"solve_standard_tm_kernelILi(\d)ELb(\d)ELb(\d)ELb(\d)E\S*\s+REG:(\d+) STACK:\d+ SHARED:(\d+)",
                         text):
        D, cost, extras, odd, regs, shared = (int(g) for g in m.groups())
        res[(D, bool(cost), bool(extras), bool(odd))] = (regs, shared)
    assert len(res) == 24, sorted(res)
    return res


def tm_ctas(K, D, cost, extras):
    """Resident CTAs per SM, minsnap_standard_tm.cuh:858-871: tensor memory, registers (65,536 per SM, rounded to 8
    per thread, 128 threads) and shared memory (228 KB per SM, 1 KB reserved per CTA)."""
    regs, shared = tm_resources()[tm_instantiation(K, D, cost, extras)]
    ctas = 512 // tmem_columns(K, D)
    ctas = min(ctas, 65536 // ((regs + 7) // 8 * 8 * 4 * 32))
    ctas = min(ctas, (228 * 1024) // (tm_smem_bytes(K, D) + shared + 1024))
    return max(ctas, 1)


def tm_grid_mode(B, ctas, sms):
    """minsnap_standard_tm.cuh:853-884: a warp takes two batches once the CTAs of one batch per warp exceed two waves,
    and the grid is then a whole number of waves, half as many (rounded up) as one batch per warp needs."""
    need, slots = -(-B // 64), sms * ctas
    if need <= 2 * slots:
        return "one batch per warp"
    return "two batches, even waves" if -(-need // slots) % 2 == 0 else "two batches, odd waves"


def pair_warps(K, D):
    """fast::launch_mode in solve mode (staged inputs), minsnap_standard_fast.cuh:861-875."""
    per_warp = _warp_smem_doubles(K, D, False, False) * 8
    warps, best = 1, 0
    for w in range(1, 5):
        if per_warp * w > MAX_DYNAMIC_SMEM:
            break
        resident = min((228 * 1024) // (per_warp * w + 1024) * w, 8)
        if resident > best:
            best, warps = resident, w
    return warps


def pair_loops(B, K, D, sms):
    """Grid capped at SMs x 256 CTAs, minsnap_standard_fast.cuh:885-890."""
    return -(-B // (pair_warps(K, D) * 16)) > sms * 256


def bcr_smem_bytes(K, D):
    """bcr::smem_doubles x 8, minsnap_standard_bcr.cuh:59-73 (record stride (32 + 4 D) | 1)."""
    return ((K - 1) * ((32 + 4 * D) | 1) + 2 * ((K + 1) * D + K + 8 * D)) * 8


def bcr_threads(K):
    """minsnap_standard_bcr.cuh:551-553."""
    return max(64, ((K // 2) + 31) // 32 * 32)


def bcr_resident(K, D):
    """Resident CTAs per SM, minsnap_standard_bcr.cuh:559."""
    return 2 if MAX_DYNAMIC_SMEM + 1024 >= 2 * (bcr_smem_bytes(K, D) + 1024) else 1


def chunk_segments(K):
    """chunked::chunk_segments, minsnap_standard_chunked.cuh:55-59."""
    for m in (12, 10, 8, 6, 4):
        if K % m == 0 and (K // m) % 2 == 0 and K // m >= 4:
            return m
    return 0


def chunked_ranges(B):
    """minsnap_standard_chunked.cuh:733-735: two ranges from 2,048 trajectories, split at a multiple of 16."""
    if B < 2048:
        return [(0, B)]
    mid = (B // 2 + 15) // 16 * 16
    return [(0, mid), (mid, B)]


def general_solve_warps(N, K, D):
    """launch_general_n for the standard mask (minsnap_general.cu:441-444 through W.general_warps)."""
    h = N // 2
    return W.general_warps(K, D, K + N - 1, (K - 1) * (h - 1), N)


def general_solve_steps(N, D, k_max=1000):
    """{warps: (first K, last K)} and the first refused K of the solve instantiation on the standard mask."""
    steps = {}
    for K in range(1, k_max):
        w = general_solve_warps(N, K, D)
        if w is None:
            return steps, K
        steps[w] = (steps.get(w, (K, K))[0], K)
    raise AssertionError(k_max)


# ------------------------------------------------------------------------------------------
# Case tables
# ------------------------------------------------------------------------------------------
# times: "given", "est" (None, not written back), "est_out" (None, written to times_out); extras from end
# derivatives ("ends"), from want_free ("free") or from both
Case = namedtuple("Case", "K D B times ends free cost forced N derivative plant", defaults=(None, 10, 4, False))
TIME_MODES = ("given", "est", "est_out")
EVEN_K, ODD_K = (2, 4, 6, 8, 10, 12), (5, 7, 9, 11)

TM_CASES = []
_i = 0
for _D in (1, 2, 3):
    for _cost in (False, True):
        for _extras in (False, True):
            for _Ks in (EVEN_K, ODD_K):
                for _j in range(2):                                     # two time modes per instantiation
                    _K = _Ks[(_i + 3 * _j) % len(_Ks)]
                    _src = ("ends", "free", "both")[(_i + _j) % 3] if _extras else None
                    TM_CASES.append(Case(_K, _D, 16 * (3 + _j) + 5 + _D, TIME_MODES[(_i + _j) % 3],
                                         _src in ("ends", "both"), _src in ("free", "both"), _cost))
                _i += 1
# two batches per warp on <D, false, false, false>: 4 waves (even) and 3 waves (odd) of CTAs at 148 SMs; D = 1 at
# K = 10 fits 3 CTAs per SM, D = 2 and 3 fit 2 (registers)
for _D, _K, _slots in ((1, 10, 3 * B200_SMS), (2, 8, 2 * B200_SMS), (3, 10, 2 * B200_SMS)):
    for _waves in (4, 3):
        TM_CASES.append(Case(_K, _D, (_waves * _slots - 10) * 64 - 3, "given", False, False, False))

PAIR_CASES = [Case(K, D, 37 + D, TIME_MODES[(K + D) % 3], (K + D) % 2 == 0, K % 2 == 1, cost)
              for K in (1, 3, 13, 24) for D in (1, 2, 3) for cost in (False, True)]
PAIR_CASES += [Case(10, D, 45, "given", False, False, False, "pair") for D in (1, 2, 3)]
PAIR_LOOP = Case(3, 1, B200_SMS * 256 * pair_warps(3, 1) * 16 + 37, "given", False, False, False)
PAIR_CASES.append(PAIR_LOOP)

PAIR_LONG_CASES = [Case(25, D, 7, t, D == 2, free, False, "pair_long") for D in (1, 2, 3) for free in (False, True)
                   for t in TIME_MODES]
PAIR_LONG_CASES += [Case(25, D, 38 * B200_SMS + 77, "given", False, True, True) for D in (1, 2, 3)]
PAIR_LONG_CASES += [Case(K, D, 3, "est_out", True, True, True, "pair_long") for D, K in ((1, 907), (2, 604), (3, 453))]


def _bcr_steps(D):
    steps = {}
    for K in range(25, 514):
        steps.setdefault(bcr_threads(K), []).append(K)
    return steps


def _bcr_resident_switch(D):
    """(last K with 2 resident CTAs, first K with 1)."""
    K = 25
    while bcr_resident(K + 1, D) == 2:
        K += 1
    return K, K + 1


BCR_CASES = []
for _threads, _Ks in sorted(_bcr_steps(3).items()):
    BCR_CASES += [Case(_Ks[0], 3, 3, "given", True, True, False, "bcr"), Case(_Ks[-1], 3, 2, "est_out", False, True,
                                                                              True, "bcr")]
for _D in (1, 2):
    for _threads, _Ks in sorted(_bcr_steps(_D).items()):
        BCR_CASES.append(Case(_Ks[len(_Ks) // 2], _D, 3, TIME_MODES[_threads // 32 % 3], _D == 2, True, _threads > 128,
                              "bcr"))
for _D in (1, 2, 3):
    _last2, _first1 = _bcr_resident_switch(_D)
    BCR_CASES += [Case(_last2, _D, 2, "given", False, True, False, "bcr"),
                  Case(_first1, _D, 2, "given", True, False, True, "bcr")]
    BCR_CASES.append(Case(40, _D, 2 * B200_SMS * bcr_resident(40, _D) + 5, "given", _D == 3, True, True))   # loops
BCR_CASES.append(Case(64, 3, 21, "est", False, False, True, "bcr"))   # cost from scratch times

CHUNKED_CASES = [Case(K, D, B, "est_out", False, True, True, None, 10, 4, True)
                 for K in (56, 36, 32, 40, 48) for D in (1, 2, 3) for B in (1500 + D, 2101 + 16 * D)]

# N, derivative, D through solve_standard's general route
GENERAL_SHAPES = [(4, 1, 3), (6, 2, 3), (8, 3, 3), (12, 5, 3), (12, 4, 2), (10, 2, 3), (10, 3, 3), (10, 4, 4),
                  (10, 4, 5)]
GENERAL_CASES = [Case(6, D, 21, t, ends, False, True, None, N, dv) for N, dv, D in GENERAL_SHAPES
                 for t, ends in (("given", False), ("est_out", True))]

STD_CASES = TM_CASES + PAIR_CASES + PAIR_LONG_CASES + BCR_CASES + CHUNKED_CASES + GENERAL_CASES

# ms.solve (the solve instantiation of solve_general_kernel): (N, K, D, B)
_steps10, REFUSED_GENERAL_SOLVE = general_solve_steps(10, 3)
SOLVE_CASES = [(10, K, 3, 11) for lo_hi in _steps10.values() for K in lo_hi]
SOLVE_CASES += [(12, (lo + hi) // 2, 3, 9) for lo, hi in general_solve_steps(12, 3)[0].values()]
SOLVE_LOOP = (10, 10, 3, B200_SMS * 32 * 8 + 37)
SOLVE_CASES.append(SOLVE_LOOP)

# the first K past the standard-mask kernels at N = 10 snap, per D: the general route takes it and refuses it
REFUSED = {3: 514, 2: 605, 1: 908}


def query(c, sms=B200_SMS):
    return (c.B, c.K, c.D, c.N, c.derivative, sms, True, True, c.forced)


def variant(c, route, sms=B200_SMS):
    """The variant a case reaches inside its route."""
    if route == "tm":
        inst = tm_instantiation(c.K, c.D, c.cost, c.ends or c.free)
        return inst + (tm_grid_mode(c.B, tm_ctas(c.K, c.D, c.cost, c.ends or c.free), sms),)
    if route == "pair":
        return (c.D, c.cost, pair_loops(c.B, c.K, c.D, sms))
    if route == "pair_long":
        return (c.D, "free scratch" if not c.free else "free out", "times scratch" if c.times == "est" else c.times)
    if route == "bcr":
        return (c.D, bcr_threads(c.K), bcr_resident(c.K, c.D), c.B > sms * bcr_resident(c.K, c.D),
                c.cost and c.times == "est")
    if route == "chunked":
        return (c.D, chunk_segments(c.K), len(chunked_ranges(c.B)))
    return (c.N, c.derivative, c.D)


def routes_of(cases, sms=B200_SMS):
    return run_routes([query(c, sms) for c in cases])


def case_id(c):
    return "K%d-D%d-B%d-%s%s%s%s%s%s" % (c.K, c.D, c.B, c.times, "-ends" * c.ends, "-free" * c.free, "-cost" * c.cost,
                                       "-" + c.forced if c.forced else "", "-N%dd%d" % (c.N, c.derivative)
                                       if (c.N, c.derivative) != (10, 4) else "")


# ------------------------------------------------------------------------------------------
# helpers
# ------------------------------------------------------------------------------------------
def dev(torch, a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def make_inputs(c, seed):
    rng = np.random.default_rng(seed)
    pos = np.cumsum(rng.uniform(1.0, 4.0, (c.B, c.K + 1, c.D)) * rng.choice([-1.0, 1.0], (c.B, c.K + 1, c.D)), axis=1)
    ends = rng.uniform(-1.0, 1.0, (c.B, 2, c.N // 2 - 1, c.D)) if c.ends else None
    return rng, pos, ends


def host_times(oracle, pos):
    return np.stack([oracle.estimate_segment_times(p, V_MAX, A_MAX) for p in pos])


def rows_to_check(B, n=48):
    tail = B % 16 or 16
    return sorted({0, B - 1, *range(B - tail, B), *np.linspace(0, B - 1, n).astype(int).tolist()})


def solve(ms, monkeypatch, forced, pos_d, times_d, ends_d, c, **kw):
    with monkeypatch.context() as m:
        if forced:
            m.setenv("MINSNAP_STANDARD_ROUTE", forced)
        else:
            m.delenv("MINSNAP_STANDARD_ROUTE", raising=False)
        args = dict(end_derivatives=ends_d, v_max=V_MAX, a_max=A_MAX, N=c.N, derivative=c.derivative,
                    want_free=c.free, want_cost=c.cost, want_status=True, want_times=c.times == "est_out")
        args.update(kw)
        return ms.solve_standard(pos_d, times_d, **args)


def row_values(c, pos, ends, b):
    v = vertex_values(pos[b], c.N)
    if ends is not None:
        v[0, 1:] = ends[b, 0]
        v[-1, 1:] = ends[b, 1]
    return v


def reference(oracle, oracle_ld, c, values, times):
    """The references of one trajectory: [(coeffs, d_free [n_free][D], cost), allowance], the truth first.  The
    truth is long double (oracle_ld.solve for short chains off N = 10 snap, helpers.banded_ld_solve otherwise); at
    N = 10 snap and K <= 64 the f64 oracle follows with the allowance of compare_with_oracle (test_gpu_parity.py):
    twice its own distance from the truth, for the reference-order f64 arithmetic is itself ~1e-8 off where the
    segment times differ widely."""
    mask = standard_mask(c.K, c.N)
    if c.K > 64 or (c.N, c.derivative) == (10, 4):
        c_t, f_t, cost_t = banded_ld_solve(oracle_ld, c.N, c.derivative, mask, values, times)
    else:
        r = oracle_ld.solve(c.N, c.K, c.D, c.derivative, mask, values, times)
        assert r["status"] == 0
        c_t, f_t, cost_t = r["coeffs"], r["d_free"].T, r["cost"]
    refs = [((c_t, f_t, cost_t), (0.0, 0.0))]
    if c.K <= 64 and (c.N, c.derivative) == (10, 4):
        r = oracle.solve(c.N, c.K, c.D, c.derivative, mask, values, times)
        assert r["status"] == 0
        f = r["d_free"].T
        scale = float(np.abs(f_t).max()) if f_t.size else 1.0
        slack = (2.0 * rel_rows(r["coeffs"], c_t),
                 2.0 * float(np.abs(np.asarray(f - f_t, np.float64)).max(initial=0.0)) / scale)
        refs.append(((r["coeffs"], f, r["cost"]), slack))
    return refs


def rel_rows(a, b):
    """Per-polynomial max-norm relative difference."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    den = np.abs(b).max(axis=-1)
    return float((np.abs(a - b).max(axis=-1) / np.where(den == 0, 1.0, den)).max())


def check_against_truth(oracle, oracle_ld, c, out, pos, ends, times, rows):
    coeffs = out["coeffs"]
    free = out["free_values"]
    cost = out["cost"]
    for b in rows:
        for i, ((want_c, want_f, want_cost), (slack, free_slack)) in enumerate(
                reference(oracle, oracle_ld, c, row_values(c, pos, ends, b), times[b])):
            suffix = "" if i == 0 else " vs f64 oracle"
            err = rel_rows(coeffs[b], want_c)
            record("coeffs" + suffix, err)
            assert err <= COEFF_TOL + slack, (b, err, slack)
            if free is not None and want_f.size:
                scale = float(np.abs(want_f).max())
                ferr = float(np.abs(free[b] - np.asarray(want_f, np.float64)).max()) / scale
                record("free" + suffix, ferr)
                assert ferr <= 1e-8 + free_slack, (b, ferr, free_slack)
            if cost is not None:
                cerr = abs(cost[b] / float(want_cost) - 1.0)
                record("cost" + suffix, cerr)
                assert cerr <= COST_TOL + slack, (b, cerr, slack)


def np_out(out):
    return {k: (v.cpu().numpy() if v is not None else None) for k, v in out.items()}


def run_std_case(ms, oracle, oracle_ld, torch, monkeypatch, c, route, seed):
    rng, pos, ends = make_inputs(c, seed)
    bad = []
    if c.plant:          # coincident consecutive vertices: an estimated time of 0 in a trajectory of each range
        for lo, hi in chunked_ranges(c.B):
            b = (lo + hi) // 2 + 1
            pos[b, 3] = pos[b, 2]
            bad.append(b)
    pos_d = dev(torch, pos)
    ends_d = dev(torch, ends) if ends is not None else None
    times_d = None
    if c.times == "given":
        times_d = ms.estimate_segment_times(pos_d, V_MAX, A_MAX) * dev(torch, rng.uniform(0.8, 1.25, (c.B, c.K)))
    out = solve(ms, monkeypatch, c.forced, pos_d, times_d, ends_d, c)
    torch.cuda.synchronize()
    res = np_out(out)
    rows = [b for b in (rows_to_check(c.B) if c.K <= 64 else (0, c.B // 2, c.B - 1)) if b not in bad]
    if c.times == "given":
        times = res["times"]
    else:
        times = np.zeros((c.B, c.K))
        times[rows] = host_times(oracle, pos[rows])
        if c.times == "est_out":
            terr = float((np.abs(res["times"][rows] - times[rows]) / times[rows]).max())
            record("times", terr)
            assert terr <= 1e-14
    check_against_truth(oracle, oracle_ld, c, res, pos, ends, times, rows)
    status = res["status"]
    want_status = np.zeros(c.B, np.int32)
    assert all(status[b] & 2 for b in bad), status[bad]
    want_status[bad] = status[bad]
    assert np.array_equal(status, want_status), np.nonzero(status != want_status)
    # status and times_out are pure stores: the same coefficients without them
    bare = solve(ms, monkeypatch, c.forced, pos_d, times_d, ends_d, c, want_status=False, want_times=False)
    # (compared as bit patterns: a planted zero time leaves NaN in its trajectory, and NaN != NaN)
    assert torch.equal(bare["coeffs"].view(torch.int64), out["coeffs"].view(torch.int64))
    # another instantiation of the same shape: cost flipped, and extras too where no end derivatives are given
    alt = solve(ms, monkeypatch, route, pos_d, times_d, ends_d, c, want_cost=not c.cost,
                want_free=c.free if c.ends else not c.free)
    others = [alt]
    if route == "tm":
        others.append(solve(ms, monkeypatch, "pair", pos_d, times_d, ends_d, c))
    for o in others:
        torch.cuda.synchronize()
        good = np.setdiff1d(np.arange(c.B), bad)
        cerr = rel_rows(o["coeffs"].cpu().numpy()[good], res["coeffs"][good])
        record("across instantiations", cerr)
        assert cerr <= 1e-10
        if c.times == "est_out" and o["times"] is not None:
            assert np.array_equal(o["times"].cpu().numpy(), res["times"])
    return res


# ------------------------------------------------------------------------------------------
# tests
# ------------------------------------------------------------------------------------------
STD_ROUTE_OF = {}


def expected_route(c):
    if not STD_ROUTE_OF:
        STD_ROUTE_OF.update(zip(STD_CASES, routes_of(STD_CASES)))
    return STD_ROUTE_OF[c]


def test_variant_tags_hold_on_this_device(torch_cuda):
    sms = torch_cuda.cuda.get_device_properties(0).multi_processor_count
    assert sms == B200_SMS, "the batch sizes of the grid cases are set for %d SMs" % B200_SMS
    for c, r148, r in zip(STD_CASES, routes_of(STD_CASES), routes_of(STD_CASES, sms)):
        assert r == r148 and variant(c, r, sms) == variant(c, r148), c


@pytest.mark.parametrize("c", STD_CASES, ids=case_id)
def test_solve_standard_variant(ms, oracle, oracle_ld, torch_cuda, monkeypatch, c):
    route = expected_route(c)
    run_std_case(ms, oracle, oracle_ld, torch_cuda, monkeypatch, c, route, zlib.crc32(case_id(c).encode()))


def test_bench_shape_every_row(ms, oracle, torch_cuda):
    """The benchmark's own call: 65,536 x K = 10, D = 3, given times, no cost, no status (the two-batch grid of
    <3, false, false, false> with a null status pointer), every row against the threaded f64 oracle."""
    torch = torch_cuda
    B, K = 65536, 10
    c = Case(K, 3, B, "given", False, False, False)
    assert routes_of([c]) == ["tm"] and variant(c, "tm")[-1].startswith("two batches")
    pos = ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], BASE_SEED)
    pos_d = dev(torch, pos)
    times_d = ms.estimate_segment_times(pos_d, V_MAX, A_MAX, 6.5)
    got = ms.solve_standard(pos_d, times_d, want_status=False)["coeffs"].cpu().numpy()
    want, _, st = oracle.solve_batch_standard(pos, times_d.cpu().numpy(), n_threads=os.cpu_count() or 1)
    assert st == 0
    err = rel_rows(got, want)
    record("coeffs (bench shape)", err)
    assert err <= COEFF_TOL


@pytest.mark.parametrize("case", SOLVE_CASES, ids=lambda s: "N%d-K%d-D%d-B%d" % s)
def test_general_solve_instantiation(ms, oracle, oracle_ld, torch_cuda, case):
    """ms.solve on the standard mask: the solve instantiation of solve_general_kernel on every warps-per-CTA step.
    Times as in every other case, the estimate of the reference's estimateSegmentTimes perturbed by up to 25%; the
    order minimised is derivative h - 1 (snap at N = 10, derivative 5 at N = 12), as in the reference's tests."""
    torch = torch_cuda
    N, K, D, B = case
    c = Case(K, D, B, "given", False, True, True, None, N, N // 2 - 1)
    rng, pos, _ = make_inputs(c, K * 7 + N)
    times = host_times(oracle, pos) * rng.uniform(0.8, 1.25, (B, K))
    mask = standard_mask(K, N)
    fixed = np.stack([vertex_values(p, N)[mask.astype(bool)] for p in pos])
    out = ms.solve(mask, dev(torch, fixed), dev(torch, times), N=N, derivative=c.derivative)
    res = np_out(out)
    assert (res["status"] == 0).all()
    rows = rows_to_check(B, 16) if K <= 64 else (0, B - 1)
    check_against_truth(oracle, oracle_ld, c, res, pos, None, times, rows)


def raw_solve(ms, torch, B, K, D, pos_d, times_d, ends_d, outs):
    """minsnap_solve_standard through the C ABI on caller-owned outputs (None = not requested)."""
    p = lambda t: None if t is None else C.c_void_p(t.data_ptr())
    return ms.capi.load().minsnap_solve_standard(
        B, K, D, 10, 4, p(pos_d), p(ends_d), p(times_d), V_MAX, A_MAX, 6.5, p(outs.get("times_out")),
        p(outs["coeffs"]), p(outs.get("free")), p(outs.get("cost")), p(outs.get("status")),
        C.c_void_p(torch.cuda.current_stream().cuda_stream))


@pytest.mark.parametrize("D", sorted(REFUSED))
def test_general_route_refusals_write_nothing(ms, torch_cuda, D):
    """The first K the general route refuses at N = 10 snap: MINSNAP_ERR_UNSUPPORTED and every output untouched,
    times_out included (the refusal comes before the time estimate)."""
    torch = torch_cuda
    K = REFUSED[D]
    c = Case(K, D, 2, "given", False, True, True)
    assert routes_of([c]) == ["general"] and general_solve_warps(10, K, D) is None
    _, pos, _ = make_inputs(c, D)
    pos_d = dev(torch, pos)
    for given in (True, False):
        times_d = dev(torch, np.ones((2, K))) if given else None
        outs = {"coeffs": torch.full((2, K, D, 10), 7.0, dtype=torch.float64, device="cuda"),
                "free": torch.full((2, (K - 1) * 4, D), 7.0, dtype=torch.float64, device="cuda"),
                "cost": torch.full((2,), 7.0, dtype=torch.float64, device="cuda"),
                "status": torch.full((2,), 7, dtype=torch.int32, device="cuda"),
                "times_out": None if given else torch.full((2, K), 7.0, dtype=torch.float64, device="cuda")}
        assert raw_solve(ms, torch, 2, K, D, pos_d, times_d, None, outs) == ms.capi.ERR_UNSUPPORTED
        torch.cuda.synchronize()
        for name, t in outs.items():
            if t is not None:
                assert bool((t == 7).all()), (name, given)


# one case per route for the status bits and the guards
ROUTE_SHAPES = {"tm": (10, 3, 53), "pair": (13, 2, 37), "pair_long": (30, 3, 21), "bcr": (40, 1, 19),
                "chunked": (32, 3, 37), "general": (10, 3, 21)}


@pytest.mark.parametrize("route", sorted(ROUTE_SHAPES))
def test_status_bits_on_every_route(ms, torch_cuda, monkeypatch, route):
    """A zero and a negative time in the first, a middle and the last (ragged) trajectory: bit 2 on exactly those,
    every other status 0."""
    torch = torch_cuda
    K, D, B = ROUTE_SHAPES[route]
    c = Case(K, D, B, "given", False, True, True, route)
    assert routes_of([c]) == [route]
    rng, pos, _ = make_inputs(c, 5)
    times = rng.uniform(0.8, 2.0, (B, K))
    bad = [0, B // 2, B - 1]
    for b in bad:
        times[b, (b + 1) % K] = 0.0
        times[b, (b + 4) % K] = -0.5
    out = solve(ms, monkeypatch, route, dev(torch, pos), dev(torch, times), None, c)
    st = out["status"].cpu().numpy()
    assert all(st[b] & 2 for b in bad), st[bad]
    assert not st[np.setdiff1d(np.arange(B), bad)].any()


@pytest.mark.parametrize("route", sorted(ROUTE_SHAPES))
def test_outputs_stay_inside_their_views(ms, oracle, oracle_ld, torch_cuda, monkeypatch, route):
    """Every output a view into a larger buffer whose guard rows hold a NaN bit pattern, the batch ragged: the guards
    are the same bits after the call.  The coefficient view starts 16 doubles (128 bytes, not a row) into its
    buffer, so tm still runs and its tensor map starts mid-allocation."""
    torch = torch_cuda
    K, D, B = ROUTE_SHAPES[route]
    c = Case(K, D, B, "est_out", False, True, True, route)
    _, pos, _ = make_inputs(c, 9)
    pos_d = dev(torch, pos)
    G = 16

    def guarded(n, dtype):
        buf = torch.empty(G + n + 64, dtype=dtype, device="cuda")
        buf.view(torch.int64 if dtype == torch.float64 else torch.int32).fill_(
            int(NAN_BITS) if dtype == torch.float64 else -559038737)
        return buf, buf[G:G + n]

    shapes = {"coeffs": (B * K * D * 10, torch.float64), "free": (B * (K - 1) * 4 * D, torch.float64),
              "cost": (B, torch.float64), "status": (B, torch.int32), "times_out": (B * K, torch.float64)}
    bufs, outs = {}, {}
    for name, (n, dtype) in shapes.items():
        bufs[name], outs[name] = guarded(n, dtype)
    before = {k: v.clone() for k, v in bufs.items()}
    with monkeypatch.context() as m:
        m.setenv("MINSNAP_STANDARD_ROUTE", route)
        assert raw_solve(ms, torch, B, K, D, pos_d, None, None, outs) == 0
    torch.cuda.synchronize()
    for name, buf in bufs.items():
        n = shapes[name][0]
        a = buf.view(torch.int64 if buf.dtype == torch.float64 else torch.int32)
        b = before[name].view(a.dtype)
        assert torch.equal(a[:G], b[:G]) and torch.equal(a[G + n:], b[G + n:]), name
    assert not outs["status"].any()
    res = {"coeffs": outs["coeffs"].view(B, K, D, 10).cpu().numpy(),
           "free_values": outs["free"].view(B, (K - 1) * 4, D).cpu().numpy(), "cost": outs["cost"].cpu().numpy()}
    times = outs["times_out"].view(B, K).cpu().numpy()
    check_against_truth(oracle, oracle_ld, c, res, pos, None, times, (0, B // 2, B - 1))


PDL_SCRIPT = r"""
import sys
import numpy as np
sys.path.insert(0, sys.argv[1])
import torch
import mav_trajectory_generation_cmake_b200 as ms
ms.load()
data = dict(np.load(sys.argv[2]))
out = {}
for key in [k for k in data if k.startswith("pos")]:
    pos = torch.from_numpy(data[key]).cuda()
    times = torch.from_numpy(data[key.replace("pos", "times")]).cuda()
    out[key.replace("pos", "coeffs")] = ms.solve_standard(pos, times)["coeffs"].cpu().numpy()
np.savez(sys.argv[3], **out)
"""


def test_pdl_off_matches_bit_for_bit(ms, torch_cuda, tmp_path):
    """MINSNAP_TM_PDL=0 (read once per process) in one subprocess: one case per tm D at one-batch and two-batch sizes,
    equal bit for bit to the same calls in this process."""
    torch = torch_cuda
    data, want = {}, {}
    for D, K, slots in ((1, 10, 3 * B200_SMS), (2, 8, 2 * B200_SMS), (3, 10, 2 * B200_SMS)):
        for B in (37, (2 * slots + 5) * 64 - 3):
            c = Case(K, D, B, "given", False, False, False)
            assert routes_of([c]) == ["tm"]
            rng, pos, _ = make_inputs(c, D * B)
            times = rng.uniform(0.5, 2.0, (B, K))
            key = "%d_%d" % (D, B)
            data["pos" + key], data["times" + key] = pos, times
            want["coeffs" + key] = ms.solve_standard(dev(torch, pos), dev(torch, times))["coeffs"].cpu().numpy()
    np.savez(tmp_path / "in.npz", **data)
    env = dict(os.environ, MINSNAP_TM_PDL="0")
    env.pop("MINSNAP_STANDARD_ROUTE", None)
    subprocess.run([sys.executable, "-c", PDL_SCRIPT, ROOT, str(tmp_path / "in.npz"), str(tmp_path / "out.npz")],
                   env=env, check=True, timeout=300)
    got = np.load(tmp_path / "out.npz")
    assert set(got.files) == set(want)
    for k in want:
        assert np.array_equal(got[k].view(np.int64), want[k].view(np.int64)), k


def test_zz_report_largest_errors():
    print("\nlargest error per bar:", {k: "%.2e" % v for k, v in sorted(MEASURED.items())})
