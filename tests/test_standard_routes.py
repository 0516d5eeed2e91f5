"""The kernel choice of minsnap_solve_standard (choose_standard_route in minsnap_standard_route.cuh), checked on the
CPU: tests/cpp/standard_routes.cu compiles the route header for sm_100a, instantiates no kernel and prints the route
of each query."""
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "cpp", "standard_routes.cu")
BIN = os.path.join(ROOT, "tests", "cpp", "bin", "standard_routes")
CSRC = os.path.join(ROOT, "mav_trajectory_generation_cmake_b200", "csrc")

SMS = 148   # B200
BATCHES = (1, 1184, 1185, 5624, 5625, 65536)   # either side of 8 x SMs = 1,184 and 38 x SMs = 5,624

# The default decision on 148 SMs, N = 10, snap, every pointer 16-byte aligned: (Ks, Ds, route per batch size).
TABLE = [
    ((1, 3, 13, 24), (1, 2, 3), ("pair",) * 6),
    ((2, 4, 5, 10, 11, 12), (1, 2, 3), ("tm",) * 6),
    ((25, 50, 101, 441), (1, 2, 3), ("bcr",) * 4 + ("pair_long",) * 2),
    ((513,), (1, 2), ("bcr",) * 4 + ("pair_long",) * 2),
    ((513,), (3,), ("bcr",) * 6),
    ((32, 64, 256, 440, 512), (1, 2, 3), ("bcr", "bcr") + ("chunked",) * 4),
    ((514,), (1, 2), ("pair_long",) * 6),
    ((600,), (1, 2), ("pair_long", "pair_long") + ("chunked",) * 4),
    ((514, 600, 1000), (3,), ("general",) * 6),
    ((1000,), (1, 2), ("general",) * 6),
]


def run_routes(queries):
    """The route of each query: (B, K, D, N, derivative, sms, coeffs_aligned16, inputs_aligned16, forced or None).
    Builds the binary when a header is newer (tests/test_gpu_standard_variants.py tags its cases with it too)."""
    deps = [SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(BIN) or any(os.path.getmtime(d) > os.path.getmtime(BIN) for d in deps):
        os.makedirs(os.path.dirname(BIN), exist_ok=True)
        subprocess.check_call(["nvcc", "-gencode", "arch=compute_100a,code=sm_100a", "-std=c++17", SRC, "-o", BIN])
    text = "".join("%d %d %d %d %d %d %d %d %s\n" % (*q[:6], int(q[6]), int(q[7]), q[8] or "-") for q in queries)
    out = subprocess.run([BIN], input=text, capture_output=True, text=True, check=True).stdout.split()
    assert len(out) == len(queries)
    return out


@pytest.fixture(scope="module")
def routes():
    return run_routes


def check(routes, cases):
    """cases: (query, expected route)"""
    got = routes([q for q, _ in cases])
    wrong = [(q, want, g) for (q, want), g in zip(cases, got) if g != want]
    assert not wrong, wrong


def query(B, K, D, coeffs_aligned=True, inputs_aligned=True, forced=None, N=10, derivative=4, sms=SMS):
    return (B, K, D, N, derivative, sms, coeffs_aligned, inputs_aligned, forced)


def test_default_route_table(routes):
    check(routes, [(query(B, K, D), want) for Ks, Ds, row in TABLE for K in Ks for D in Ds
                   for B, want in zip(BATCHES, row)])


def test_default_route_capacity_limits(routes):
    # the two-lane kernel takes K <= 907 / 604 / 453 for D = 1 / 2 / 3, the reduction K <= 513; shapes other than
    # N = 10 snap with D <= 3 go to the general kernels
    cases = []
    for D, k_max, above in ((1, 907, "general"), (2, 604, "general"), (3, 453, "bcr")):
        cases += [(query(65536, k_max, D), "pair_long"), (query(65536, k_max + 1, D), above)]
    cases += [(query(1, 514, 3), "general"), (query(1, 513, 3), "bcr")]
    cases += [(query(1, 10, 4), "general"), (query(1, 10, 3, N=8, derivative=3), "general"),
              (query(1, 10, 3, derivative=3), "general")]
    check(routes, cases)


def test_thresholds_scale_with_the_sm_count(routes):
    check(routes, [(query(8 * 132, 256, 3, sms=132), "bcr"), (query(8 * 132 + 1, 256, 3, sms=132), "chunked"),
                   (query(38 * 132, 25, 3, sms=132), "bcr"), (query(38 * 132 + 1, 25, 3, sms=132), "pair_long")])


def test_default_route_unaligned_pointers(routes):
    cases = [
        (query(65536, 10, 3, False, False), "pair"),
        (query(65536, 11, 1, False, False), "pair"),
        (query(65536, 10, 3, False, True), "pair"),        # the headline kernel needs aligned coefficients only
        (query(65536, 10, 3, True, False), "tm"),
        (query(4096, 256, 3, False, False), "bcr"),        # the partitioned route needs every pointer aligned
        (query(4096, 256, 3, True, False), "bcr"),
        (query(4096, 256, 3, False, True), "bcr"),
        (query(16384, 256, 3, False, False), "pair_long"),
    ]
    cases += [(query(4096, 528, 3, c, i), "general") for c in (False, True) for i in (False, True)]
    check(routes, cases)


def test_forced_routes(routes):
    cases = [
        # a forced route that can take the call runs, whatever the default would be
        (query(65536, 10, 3, forced="tm"), "tm"),
        (query(65536, 10, 3, forced="pair"), "pair"),
        (query(5, 3, 2, forced="pair"), "pair"),
        (query(5, 25, 3, forced="pair_long"), "pair_long"),
        (query(5, 453, 3, forced="pair_long"), "pair_long"),
        (query(65536, 256, 3, forced="bcr"), "bcr"),
        (query(1, 513, 1, forced="bcr"), "bcr"),
        (query(2, 256, 3, forced="chunked"), "chunked"),
        (query(2, 32, 1, forced="chunked"), "chunked"),
        (query(65536, 10, 3, forced="general"), "general"),
        (query(1, 1000, 3, forced="general"), "general"),
        # ... and one that cannot is refused, never replaced by another
        (query(1, 3, 3, forced="tm"), "unsupported"),
        (query(1, 13, 3, forced="tm"), "unsupported"),
        (query(65536, 10, 3, False, True, forced="tm"), "unsupported"),
        (query(1, 25, 3, forced="pair"), "unsupported"),
        (query(1, 24, 3, forced="pair_long"), "unsupported"),
        (query(1, 454, 3, forced="pair_long"), "unsupported"),
        (query(1, 24, 3, forced="bcr"), "unsupported"),
        (query(1, 514, 1, forced="bcr"), "unsupported"),
        (query(1, 50, 3, forced="chunked"), "unsupported"),
        (query(65536, 256, 3, True, False, forced="chunked"), "unsupported"),
        (query(65536, 256, 3, False, True, forced="chunked"), "unsupported"),
        (query(1, 10, 3, N=8, derivative=3, forced="pair"), "unsupported"),
    ]
    check(routes, cases)
