"""CPU tests: pin the oracle (oracle/minsnap_oracle.c) against everything the reference's own
tests hold for the hot path (SURVEY.md section 8c).  Citations: test/test_polynomial_optimization.cpp
of the reference ("T:" below)."""
import math
import os
import shutil
import subprocess

import numpy as np
import pytest

from helpers import (BASE_SEED, check_path, coeff_rel_err, random_batch, standard_mask, vertex_values)

N = 10
SNAP = 4


# ---- known-answer vector, T:700-744 ("2_vertices_setup", Matlab coefficients T:733-737) --------
MATLAB_COEFFS = np.array([-0.000000000000004, 0.000000000000004, -0.000000000000006, 0.000000000000003,
                          -0.000000000000001, 0.201600000000015, -0.134400000000012, 0.034560000000004,
                          -0.004032000000000, 0.000179200000000])


def test_golden_two_vertices_setup(oracle):
    mask = np.ones((2, 5), np.uint8)
    vals = np.zeros((2, 5, 1))
    vals[1, 0, 0] = 5.0
    seg_time = abs(5.0 - 0.0) * 2.0 / 2.0
    out = oracle.solve(N, 1, 1, SNAP, mask, vals, [seg_time])
    assert out["status"] == 0
    c = out["coeffs"][0, 0]
    # CHECK_EIGEN_MATRIX_EQUAL_DOUBLE is an (approximately) exact comparison; the Matlab
    # digits are only given to 1e-15, so compare at that resolution ...
    assert np.abs(c - MATLAB_COEFFS).max() < 2e-14
    # ... and against the closed form 5 (126 s^5 - 420 s^6 + 540 s^7 - 315 s^8 + 70 s^9), s = t/5
    closed = np.zeros(10)
    for p, a in zip(range(5, 10), (126, -420, 540, -315, 70)):
        closed[p] = 5.0 * a / 5.0 ** p
    assert np.abs(c - closed).max() < 1e-13 * np.abs(closed).max()


def test_base_coefficients(oracle):
    b = oracle.base_coefficients(22)
    for d in range(22):
        for j in range(22):
            exact = math.factorial(j) // math.factorial(j - d) if j >= d else 0
            if exact < 2 ** 53:
                assert b[d, j] == float(exact)
            else:
                assert abs(b[d, j] - float(exact)) <= 4e-16 * float(exact)


# ---- A^-1, T:194-204 ("PathPlanning_A_matrix_inversion") ----------------------------------------
def test_mapping_matrix_inversion(oracle, oracle_ld):
    for t in range(1, 61):
        A = oracle.mapping_matrix(N, float(t))
        Ai = oracle.invert_mapping_matrix(A)
        Ai_full = oracle.dense_inverse(A)          # A.inverse()
        assert np.abs(Ai - Ai_full).max() < 1.0e-10, t
        # extended precision agrees as well (relative: entries span 1e-14 .. 1)
        Ai_ld = oracle_ld.invert_mapping_matrix(oracle_ld.mapping_matrix(N, float(t))).astype(np.float64)
        assert np.abs(Ai - Ai_ld).max() < 1.0e-11 * np.abs(Ai_ld).max(), t


# ---- createRandomVertices, T:154-192, and the generator it runs on -------------------------------
def test_vertex_generation_bounds(oracle):
    pos = oracle.create_random_positions(100, [-10, -20, -10], [10, 20, 10], 12345)
    assert pos.shape == (101, 3)
    assert (pos >= [-10, -20, -10]).all() and (pos <= [10, 20, 10]).all()
    assert (np.linalg.norm(np.diff(pos, axis=0), axis=1) > 0.2).all()
    p1 = oracle.create_random_positions(100, [-50], [50], 0)
    assert (p1 >= -50).all() and (p1 <= 50).all()


@pytest.mark.skipif(shutil.which("g++") is None, reason="needs g++")
def test_generator_matches_libstdcxx(oracle, tmp_path):
    """std::mt19937 + std::uniform_real_distribution<double> (src/vertex.cpp:33-44) bit for bit."""
    src = tmp_path / "mt.cpp"
    src.write_text(r"""
#include <cstdio>
#include <cstdlib>
#include <random>
int main(int, char** argv) {
  std::mt19937 g(strtoul(argv[1], 0, 10));
  std::uniform_real_distribution<double> d(atof(argv[2]), atof(argv[3]));
  for (int i = 0; i < atoi(argv[4]); ++i) printf("%a\n", d(g));
}
""")
    exe = tmp_path / "mt"
    subprocess.check_call(["g++", "-O2", "-o", str(exe), str(src)])
    for seed, a, b in [(12345, -10, 10), (1, -1, 1), (978, -50, 50), (0, 0, 1), (12, -20, 20)]:
        ref = np.array([float.fromhex(x.decode()) for x in
                        subprocess.check_output([str(exe), str(seed), str(a), str(b), "3000"]).split()])
        assert np.array_equal(ref, oracle.mt19937_uniform(seed, a, b, 3000))


# ---- reordering, LIN.i:171-250 --------------------------------------------------------------------
def reorder_reference_python(N, K, mask):
    """Literal restatement of the reference's loops with Python sets (slow, tiny cases)."""
    h = N // 2
    all_c, fixed, free = [], set(), set()
    for v in range(K + 1):
        occ = 1 if v in (0, K) else 2
        for _ in range(occ):
            for c in range(h):
                all_c.append((v, c))
                (fixed if mask[v][c] else free).add((v, c))
    cols = sorted(fixed) + sorted(free)
    return np.array([cols.index(x) for x in all_c], np.int32), len(fixed), len(free)


def test_reordering_matches_literal_restatement(oracle):
    rng = np.random.default_rng(7)
    for K in (1, 2, 3, 5, 10):
        for trial in range(6):
            mask = standard_mask(K) if trial == 0 else (rng.random((K + 1, 5)) < 0.5).astype(np.uint8)
            col, nf, npf = oracle.reorder(N, K, mask)
            col_ref, nf_ref, np_ref = reorder_reference_python(N, K, mask)
            assert np.array_equal(col, col_ref) and nf == nf_ref and npf == np_ref


def test_standard_mask_counts(oracle):
    for K in (4, 10, 256):
        _, nf, npf = oracle.reorder(N, K, standard_mask(K))
        assert nf == K + 9 and npf == 4 * (K - 1)


# ---- checkPath + checkCost on the reference's own problem family, T:206-394 ----------------------
def cost_numeric(oracle, coeffs, times, derivative, dt=1e-3):
    """computeCostNumeric, T:61-71 (vectorised Riemann sum)."""
    K, D, _ = coeffs.shape
    total = 0.0
    for i in range(K):
        ts = np.arange(0.0, times[i], dt)
        sq = np.zeros_like(ts)
        for d in range(D):
            c = coeffs[i, d]
            # derivative-scaled coefficients, then Horner (vectorised over ts)
            dc = np.array([np.prod(np.arange(j - derivative + 1, j + 1)) * c[j] for j in range(derivative, N)])
            val = np.zeros_like(ts)
            for a in dc[::-1]:
                val = val * ts + a
            sq += val * val
        total += sq.sum() * dt
    return total


@pytest.mark.parametrize("K,seed,D", [(10, 12, 1), (50, 123, 1), (100, 1234, 1), (100, 12345, 3)])
def test_path_and_cost_properties(oracle, K, seed, D):
    if D == 1:
        pos = oracle.create_random_positions(K, [-10.0], [10.0], seed)
    else:
        pos = oracle.create_random_positions(K, [-10, -20, -10], [10, 20, 10], seed)
    times = oracle.estimate_segment_times(pos, 3.0, 5.0)
    mask = standard_mask(K)
    vals = vertex_values(pos)
    out = oracle.solve(N, K, D, SNAP, mask, vals, times)
    assert out["status"] == 0
    assert check_path(out["coeffs"], times, mask, vals, oracle) < 1e-6
    cn = cost_numeric(oracle, out["coeffs"], times, SNAP)
    assert abs(cn - out["cost"]) <= 0.1 * cn          # checkCost, T:133-152


# ---- "2_vertices_rand", T:747-774: free jerk and snap at both ends --------------------------------
def test_two_vertices_rand(oracle):
    mask = standard_mask(1, max_fixed_derivative=2)
    for i in range(100):
        pos = oracle.create_random_positions(1, [-50.0] * 3, [50.0] * 3, 12345 + i)
        times = oracle.estimate_segment_times(pos, 3.0, 5.0)
        vals = vertex_values(pos)
        out = oracle.solve(N, 1, 3, SNAP, mask, vals, times)
        assert out["status"] == 0
        assert check_path(out["coeffs"], times, mask, vals, oracle) < 1e-6


# ---- "ConstraintPacking", T:777-836 ------------------------------------------------------------------
def test_constraint_packing(oracle):
    K = 5
    mask = standard_mask(K, max_fixed_derivative=3)
    for i in range(100):
        pos = oracle.create_random_positions(K, [-50.0] * 3, [50.0] * 3, 12345 + i)
        times = oracle.estimate_segment_times(pos, 3.0, 5.0)
        out = oracle.solve(N, K, 3, SNAP, mask, vertex_values(pos), times)
        col, nf, npf = oracle.reorder(N, K, mask)
        n_all = nf + npf
        M = np.zeros((N * K, n_all))
        M[np.arange(N * K), col] = 1.0
        Mt = M.T
        M_pinv = Mt / Mt.sum(axis=1, keepdims=True)            # getMpinv, LIN.i:560-571
        A = np.zeros((N * K, N * K))
        A_inv = np.zeros((N * K, N * K))
        for s in range(K):
            As = oracle.mapping_matrix(N, times[s])
            A[s * N:(s + 1) * N, s * N:(s + 1) * N] = As
            A_inv[s * N:(s + 1) * N, s * N:(s + 1) * N] = oracle.invert_mapping_matrix(As)
        for d in range(3):
            d_all = np.concatenate([out["d_fixed"][d], out["d_free"][d]])
            p = A_inv @ M @ d_all
            d_re = M_pinv @ (A @ p)
            assert np.abs(d_all - d_re).max() < 1e-6
            for s in range(K):
                assert np.abs(out["coeffs"][s, d] - p[s * N:(s + 1) * N]).max() < 1e-6


# ---- element-level check of the solve itself: extended precision + optimality condition ---------------
@pytest.mark.parametrize("K", [4, 10, 64])
def test_solve_against_extended_precision_and_kkt(oracle, oracle_ld, K):
    pos, times = random_batch(oracle, 8, K)
    mask = standard_mask(K)
    for b in range(8):
        vals = vertex_values(pos[b])
        o64 = oracle.solve(N, K, 3, SNAP, mask, vals, times[b])
        old = oracle_ld.solve(N, K, 3, SNAP, mask, vals, times[b], want_R=True)
        assert coeff_rel_err(o64["coeffs"], old["coeffs"]) < 2e-9
        # R_pp d_p + R_pf d_f = 0 in long double: the unique minimiser of the QP
        R = old["R"]
        nf = old["d_fixed"].shape[1]
        for d in range(3):
            res = R[nf:, nf:] @ old["d_free"][d] + R[nf:, :nf] @ old["d_fixed"][d]
            scale = np.abs(R[nf:, :nf] @ old["d_fixed"][d]).max()
            assert float(np.abs(res).max()) < 1e-12 * float(scale)
        assert abs(o64["cost"] - float(old["cost"])) < 1e-8 * float(old["cost"])


def test_trajectory_evaluate_semantics(oracle):
    pos, times = random_batch(oracle, 1, 4)
    out = oracle.solve(N, 4, 3, SNAP, standard_mask(4), vertex_values(pos[0]), times[0])
    c, T = out["coeffs"], times[0]
    # a vertex time belongs to the segment on its right (src/trajectory.cpp:45-57)
    t1 = T[0]
    v, seg = oracle.trajectory_evaluate(c, T, t1, 0)
    assert seg == 1
    assert np.abs(v - pos[0, 1]).max() < 1e-6
    # past the end: zeros
    v, seg = oracle.trajectory_evaluate(c, T, T.sum() + 1.0, 0)
    assert seg == -1 and (v == 0).all()
    # evaluateRange emits ceil-ish((t1-t0)/dt) samples with sequentially accumulated times
    vals, ts = oracle.trajectory_evaluate_range(c, T, 0.0, float(T.sum()), 0.01, 1)
    assert abs(len(ts) - T.sum() / 0.01) <= 2
    assert ts[0] == 0.0 and np.all(np.diff(ts) > 0)


@pytest.mark.parametrize("N_,derivative,K,D", [(10, SNAP, 1, 3), (10, SNAP, 2, 1), (10, SNAP, 7, 3), (10, SNAP, 33, 2),
                                               (10, SNAP, 64, 3), (12, 5, 9, 2), (6, 2, 12, 3)])
def test_banded_long_double_reference(oracle_ld, N_, derivative, K, D):
    """helpers.banded_ld_solve (the O(K) reference of the long-chain tests) equals the dense long-double oracle to
    1e-10, with zero and with non-zero end derivatives.  The two eliminate in different orders; measured 6e-12 at
    K = 64 and 1e-11 at N = 12, far below the 1e-8 the kernels are held to."""
    from helpers import banded_ld_solve
    rng = np.random.default_rng(K * 100 + D)
    h = N_ // 2
    pos = np.cumsum(rng.uniform(1.0, 4.0, (K + 1, D)) * rng.choice([-1.0, 1.0], (K + 1, D)), axis=0)
    times = rng.uniform(0.5, 2.0, K)
    mask = standard_mask(K, N_)
    for ends in (False, True):
        vals = vertex_values(pos, N_)
        if ends:
            vals[0, 1:] = rng.uniform(-1.0, 1.0, (h - 1, D))
            vals[K, 1:] = rng.uniform(-1.0, 1.0, (h - 1, D))
        want = oracle_ld.solve(N_, K, D, derivative, mask, vals, times)
        coeffs, free, cost = banded_ld_solve(oracle_ld, N_, derivative, mask, vals, times)
        assert coeff_rel_err(coeffs, want["coeffs"]) <= 1e-10
        if free.size:
            ref = want["d_free"].T
            assert np.abs(free - ref).max() <= 1e-10 * np.abs(ref).max()
        assert abs(cost / want["cost"] - 1) <= 1e-10
