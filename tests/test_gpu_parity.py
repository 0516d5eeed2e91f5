"""GPU parity tests: every CUDA entry point of the C ABI against the CPU oracle on identical
inputs (pytest -m gpu, run on the B200 box).  Tolerances are those of helpers.py / north_star:
index maps bit-exact, coefficients 1e-8 per-polynomial max-norm relative, samples 1e-6
absolute, cost 1e-8 relative."""
import numpy as np
import pytest

from helpers import (BASE_SEED, COEFF_TOL, COST_TOL, SAMPLE_TOL, check_path, coeff_rel_err, compact_fixed,
                     oracle_solve_batch, random_batch, standard_mask, vertex_values)

pytestmark = pytest.mark.gpu

N = 10
SNAP = 4


def dev(torch, a, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    if dtype is not None:
        t = t.to(dtype)
    return t.cuda()


def batch_values(pos, N_=N):
    return np.stack([vertex_values(p, N_) for p in pos])


def solve_on_route(ms, monkeypatch, route, *args, **kwargs):
    """ms.solve_standard through the kernel MINSNAP_STANDARD_ROUTE names: that kernel or an error, never another."""
    with monkeypatch.context() as m:
        m.setenv("MINSNAP_STANDARD_ROUTE", route)
        return ms.solve_standard(*args, **kwargs)


# ------------------------------------------------------------------------------------------
# a10 reordering: bit-exact
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K", [1, 2, 4, 10, 33, 256])
def test_reorder_bit_exact(ms, oracle, torch_cuda, K):
    torch = torch_cuda
    rng = np.random.default_rng(K)
    masks = [standard_mask(K), standard_mask(K, max_fixed_derivative=2), np.ones((K + 1, 5), np.uint8),
             np.zeros((K + 1, 5), np.uint8)]
    masks += [(rng.random((K + 1, 5)) < p).astype(np.uint8) for p in (0.2, 0.5, 0.8) for _ in range(8)]
    m = np.stack(masks).reshape(len(masks), -1)
    col, counts = ms.reorder(dev(torch, m), N, K)
    col, counts = col.cpu().numpy(), counts.cpu().numpy()
    for i, mk in enumerate(masks):
        c_ref, nf, npf = oracle.reorder(N, K, mk)
        assert np.array_equal(col[i], c_ref)
        assert counts[i, 0] == nf and counts[i, 1] == npf


@pytest.mark.parametrize("N_", [4, 6, 8, 12])
def test_reorder_other_orders(ms, oracle, torch_cuda, N_):
    torch = torch_cuda
    rng = np.random.default_rng(N_)
    K = 7
    masks = [(rng.random((K + 1, N_ // 2)) < 0.5).astype(np.uint8) for _ in range(16)]
    col, counts = ms.reorder(dev(torch, np.stack(masks).reshape(16, -1)), N_, K)
    for i, mk in enumerate(masks):
        c_ref, nf, npf = oracle.reorder(N_, K, mk)
        assert np.array_equal(col[i].cpu().numpy(), c_ref)
        assert tuple(counts[i].cpu().numpy()) == (nf, npf)


# ------------------------------------------------------------------------------------------
# a2 estimateSegmentTimes
# ------------------------------------------------------------------------------------------
def test_estimate_segment_times(ms, oracle, torch_cuda):
    torch = torch_cuda
    pos, times = random_batch(oracle, 64, 10)
    got = ms.estimate_segment_times(dev(torch, pos), 3.0, 5.0).cpu().numpy()
    assert np.abs(got / times - 1.0).max() < 1e-14
    got_h = ms.estimate_segment_times_host(pos, 3.0, 5.0)
    assert np.array_equal(got, got_h)


# ------------------------------------------------------------------------------------------
# a5-a9, a11 segment matrices (closed forms) against the reference-order construction
# ------------------------------------------------------------------------------------------
def test_segment_matrices(ms, oracle, oracle_ld, torch_cuda):
    T = np.concatenate([np.arange(1.0, 61.0), [0.1, 0.37, 2.5, 17.3]])
    out = ms.segment_matrices_host(T, N, SNAP)
    for i, t in enumerate(T):
        A = oracle.mapping_matrix(N, t)
        assert np.abs(out["A"][i] - A).max() <= 1e-14 * np.abs(A).max()
        # T:194-204 compares the block inverse with Eigen's A.inverse() at 1e-10 absolute; the
        # oracle's own partial-pivot full inverse is itself only good to ~3e-10 at t = 1, so the
        # bar against it is 1e-9 and the tight check is the extended-precision one below.
        if t >= 1.0:
            assert np.abs(out["Ainv"][i] - oracle.dense_inverse(A)).max() < 1e-9
            Ai_ld_full = oracle_ld.dense_inverse(oracle_ld.mapping_matrix(N, t)).astype(np.float64)
            assert np.abs(out["Ainv"][i] - Ai_ld_full).max() < 1e-10
        Ai_ld = oracle_ld.invert_mapping_matrix(oracle_ld.mapping_matrix(N, t)).astype(np.float64)
        assert np.abs(out["Ainv"][i] - Ai_ld).max() <= 1e-13 * np.abs(Ai_ld).max()
        Q = oracle.cost_matrix(N, SNAP, t)
        assert np.abs(out["Q"][i] - Q).max() <= 1e-13 * np.abs(Q).max()
        H_ld = oracle_ld.segment_hessian(N, SNAP, t).astype(np.float64)
        assert np.abs(out["H"][i] - H_ld).max() <= 1e-12 * np.abs(H_ld).max()
        # the f64 reference-order H carries the cancellation error of Ainv^T Q Ainv
        H64 = oracle.segment_hessian(N, SNAP, t)
        assert np.abs(out["H"][i] - H64).max() <= 1e-7 * np.abs(H_ld).max()


# ------------------------------------------------------------------------------------------
# a10-a13, a16 general solve
# ------------------------------------------------------------------------------------------
def run_general(ms, torch, mask, values, times, N_=N, derivative=SNAP):
    fixed = np.stack([compact_fixed(mask, v) for v in values])
    return ms.solve(mask, dev(torch, fixed), dev(torch, times), N=N_, derivative=derivative)


def compare_with_oracle(oracle, out, mask, values, times, N_=N, derivative=SNAP, coeff_tol=COEFF_TOL, truth=None):
    """GPU vs the f64 oracle at the north-star tolerances.  With `truth` (the long-double build
    of the oracle) the GPU result must be within tolerance of the truth, and the allowance
    against the f64 oracle is widened by that oracle's own distance from the truth -- needed
    only off the north-star shape (exotic masks, N = 12, low derivative orders), where the
    reference-order f64 arithmetic (Ainv^T Q Ainv, cond(A) up to 1e12) is itself ~1e-8 off."""
    ref = oracle_solve_batch(oracle, mask, values, times, N_, derivative)
    assert (ref["status"] == 0).all()
    assert (out["status"].cpu().numpy() == 0).all()
    col_ref, nf, npf = oracle.reorder(N_, mask.shape[0] - 1, mask)
    assert np.array_equal(out["col_of_row"].cpu().numpy(), col_ref)
    coeffs = out["coeffs"].cpu().numpy()
    slack = 0.0
    want_free = np.transpose(ref["d_free"], (0, 2, 1))
    free_slack = 0.0
    if truth is not None:
        ref_t = oracle_solve_batch(truth, mask, values, times, N_, derivative)
        assert coeff_rel_err(coeffs, ref_t["coeffs"]) <= coeff_tol
        slack = 2.0 * coeff_rel_err(ref["coeffs"], ref_t["coeffs"])
        if npf > 0:
            truth_free = np.transpose(ref_t["d_free"], (0, 2, 1))
            scale_t = np.abs(truth_free).max(axis=(1, 2), keepdims=True)
            free = out["free_values"].cpu().numpy()
            assert (np.abs(free - truth_free) / scale_t).max() <= 1e-8
            free_slack = 2.0 * (np.abs(want_free - truth_free) / scale_t).max()
    assert coeff_rel_err(coeffs, ref["coeffs"]) <= coeff_tol + slack
    if npf > 0:
        free = out["free_values"].cpu().numpy()              # [B][n_free][D]
        scale = np.abs(want_free).max(axis=(1, 2), keepdims=True)
        assert (np.abs(free - want_free) / scale).max() <= 1e-8 + free_slack
    if out["cost"] is not None:
        cost = out["cost"].cpu().numpy()
        assert np.abs(cost / ref["cost"] - 1.0).max() <= COST_TOL + slack
    return coeffs, ref


@pytest.mark.parametrize("K,D,B", [(1, 3, 8), (2, 3, 32), (4, 3, 64), (10, 3, 256), (10, 1, 64), (50, 3, 16),
                                   (100, 3, 4), (7, 2, 16), (3, 5, 16)])
def test_general_solve_standard_mask(ms, oracle, torch_cuda, K, D, B):
    pos, times = random_batch(oracle, B, K, D)
    mask = standard_mask(K)
    values = batch_values(pos)
    out = run_general(ms, torch_cuda, mask, values, times)
    coeffs, _ = compare_with_oracle(oracle, out, mask, values, times)
    assert check_path(coeffs[0], times[0], mask, values[0], oracle) < 1e-6


def test_general_solve_golden_vector(ms, torch_cuda):
    """T:700-744: fully constrained single segment, Matlab coefficients."""
    mask = np.ones((2, 5), np.uint8)
    vals = np.zeros((1, 2, 5, 1))
    vals[0, 1, 0, 0] = 5.0
    out = run_general(ms, torch_cuda, mask, vals, np.array([[5.0]]))
    c = out["coeffs"].cpu().numpy()[0, 0, 0]
    gold = np.array([0, 0, 0, 0, 0, 0.2016, -0.1344, 0.03456, -0.004032, 0.0001792])
    assert np.abs(c - gold).max() < 1e-15
    assert out["status"].item() == 0


def test_general_solve_two_vertices_rand(ms, oracle, torch_cuda):
    """T:747-774: one segment, ends fixed up to acceleration, jerk and snap free."""
    mask = standard_mask(1, max_fixed_derivative=2)
    pos, times = random_batch(oracle, 100, 1, 3, box=50.0)
    values = batch_values(pos)
    out = run_general(ms, torch_cuda, mask, values, times)
    coeffs, _ = compare_with_oracle(oracle, out, mask, values, times)
    for b in range(0, 100, 7):
        assert check_path(coeffs[b], times[b], mask, values[b], oracle) < 1e-6


def test_general_solve_constraint_packing(ms, oracle, torch_cuda):
    """T:777-836: 5 segments, ends fixed up to jerk; [d_f; d_p] -> p -> [d_f; d_p] round trip."""
    K = 5
    mask = standard_mask(K, max_fixed_derivative=3)
    pos, times = random_batch(oracle, 100, K, 3, box=50.0)
    values = batch_values(pos)
    out = run_general(ms, torch_cuda, mask, values, times)
    coeffs, ref = compare_with_oracle(oracle, out, mask, values, times)
    col = out["col_of_row"].cpu().numpy()
    free = out["free_values"].cpu().numpy()
    fixed = np.stack([compact_fixed(mask, v) for v in values])
    mats = ms.segment_matrices_host(times.reshape(-1), N, SNAP)
    A = mats["A"].reshape(100, K, N, N)
    Ainv = mats["Ainv"].reshape(100, K, N, N)
    for b in range(100):
        d_all = np.concatenate([fixed[b], free[b]], axis=0)          # [n_all][D]
        for d in range(3):
            for s in range(K):
                d_seg = d_all[col[s * N:(s + 1) * N], d]              # M * d_all
                p = Ainv[b, s] @ d_seg
                assert np.abs(p - coeffs[b, s, d]).max() < 1e-6
                assert np.abs(A[b, s] @ p - d_seg).max() < 1e-6


def test_general_solve_random_masks_and_values(ms, oracle, oracle_ld, torch_cuda):
    """Arbitrary fixed/free patterns (position always fixed so the QP is strictly convex) with
    non-zero derivative constraints."""
    rng = np.random.default_rng(3)
    for K in (2, 5, 9):
        for trial in range(4):
            mask = (rng.random((K + 1, 5)) < 0.4).astype(np.uint8)
            mask[:, 0] = 1
            B = 24
            pos, times = random_batch(oracle, B, K, 3, seed=100 * K + trial)
            values = batch_values(pos)
            values[:, :, 1:, :] = rng.normal(size=values[:, :, 1:, :].shape)
            out = run_general(ms, torch_cuda, mask, values, times)
            coeffs, _ = compare_with_oracle(oracle, out, mask, values, times, truth=oracle_ld)
            assert check_path(coeffs[0], times[0], mask, values[0], oracle) < 1e-6


@pytest.mark.parametrize("N_,derivative", [(10, 3), (10, 2), (8, 3), (6, 2), (12, 5), (4, 1)])
def test_general_solve_other_orders(ms, oracle, oracle_ld, torch_cuda, N_, derivative):
    K, B = 6, 16
    h = N_ // 2
    pos, times = random_batch(oracle, B, K, 3, seed=77)
    mask = standard_mask(K, N_)
    values = batch_values(pos, N_)
    out = run_general(ms, torch_cuda, mask, values, times, N_, derivative)
    compare_with_oracle(oracle, out, mask, values, times, N_, derivative, truth=oracle_ld)
    assert out["coeffs"].shape == (B, K, 3, N_) and h * (K + 1) == mask.size


def test_general_solve_flags_bad_inputs(ms, oracle, torch_cuda):
    pos, times = random_batch(oracle, 4, 4)
    times[1, 2] = 0.0
    times[2, 0] = -1.0
    out = run_general(ms, torch_cuda, standard_mask(4), batch_values(pos), times)
    st = out["status"].cpu().numpy()
    assert st[0] == 0 and st[3] == 0
    assert st[1] & 2 and st[2] & 2                                  # MINSNAP_STATUS_BAD_TIME


def test_long_horizon_parity(ms, oracle, torch_cuda):
    """Config 4 shape (K = 256, n_free = 1020) on a batch the dense-QR oracle finishes in seconds."""
    K, B = 256, 2
    pos, times = random_batch(oracle, B, K)
    mask = standard_mask(K)
    values = batch_values(pos)
    out = run_general(ms, torch_cuda, mask, values, times)
    compare_with_oracle(oracle, out, mask, values, times)


# ------------------------------------------------------------------------------------------
# standard-mask entry point (the bench path)
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("K,B", [(10, 512), (4, 64), (2, 16), (1, 8), (3, 33), (16, 40), (24, 17), (25, 17), (50, 8),
                                 (101, 5), (256, 3)])
def test_solve_standard_against_oracle(ms, oracle, torch_cuda, K, B):
    torch = torch_cuda
    pos, times = random_batch(oracle, B, K)
    out = ms.solve_standard(dev(torch, pos), dev(torch, times), want_free=True, want_cost=True)
    mask = standard_mask(K)
    values = batch_values(pos)
    ref = oracle_solve_batch(oracle, mask, values, times)
    assert (out["status"].cpu().numpy() == 0).all()
    coeffs = out["coeffs"].cpu().numpy()
    assert coeff_rel_err(coeffs, ref["coeffs"]) <= COEFF_TOL
    assert np.abs(out["cost"].cpu().numpy() / ref["cost"] - 1.0).max() <= COST_TOL
    if K > 1:
        want = np.transpose(ref["d_free"], (0, 2, 1))
        scale = np.abs(want).max(axis=(1, 2), keepdims=True)
        assert (np.abs(out["free_values"].cpu().numpy() - want) / scale).max() <= 1e-8
    assert check_path(coeffs[B // 2], times[B // 2], mask, values[B // 2], oracle) < 1e-6


@pytest.mark.parametrize("D", [1, 2, 3])
def test_long_chain_kernels_agree(ms, oracle, torch_cuda, monkeypatch, D):
    """K > 24 has two kernels: block cyclic reduction (one CTA per trajectory, small batches) and the
    two-lane kernel with its blocks in global memory (large batches, K > 513).  Both are checked against
    the oracle elsewhere (K = 25, 50, 101, 256 above; whichever kernel the batch size selects); here
    they are checked against each other over chain lengths around every power of two, with non-zero
    boundary derivatives, device-side segment times and all optional outputs."""
    torch = torch_cuda
    rng = np.random.default_rng(21 + D)
    # the two-lane kernel stages the inputs of 16 trajectories in shared memory: K <= ~440 at D = 3
    long_ks = [511, 512, 513] if D < 3 else [400, 440]
    for K in list(range(25, 40)) + [63, 64, 65, 100, 127, 128, 129, 255, 256, 257, 300] + long_ks:
        B = 5
        pos = np.cumsum(rng.uniform(0.3, 2.0, (B, K + 1, D)) * rng.choice([-1.0, 1.0], (B, K + 1, D)), axis=1)
        ends = rng.normal(size=(B, 2, 4, D))
        outs = {}
        for which in ("bcr", "pair_long"):
            outs[which] = solve_on_route(ms, monkeypatch, which, dev(torch, pos), None, end_derivatives=dev(torch, ends),
                                         v_max=3.0, a_max=5.0, want_free=True, want_cost=True, want_times=True)
        a, b = outs["bcr"], outs["pair_long"]
        assert (a["status"] == 0).all() and (b["status"] == 0).all()
        assert torch.equal(a["times"], b["times"])
        assert coeff_rel_err(a["coeffs"].cpu().numpy(), b["coeffs"].cpu().numpy()) <= 1e-9, K
        scale = b["free_values"].abs().amax(dim=(1, 2), keepdim=True)
        assert float(((a["free_values"] - b["free_values"]).abs() / scale).max()) <= 1e-9, K
        assert float((a["cost"] / b["cost"] - 1.0).abs().max()) <= 1e-9, K
    if D == 3:
        # the reduction reaches K = 513 at D = 3 (the two-lane kernel does not): checked against the oracle
        K = 513
        pos, times = random_batch(oracle, 1, K)
        out = ms.solve_standard(dev(torch, pos), dev(torch, times), want_cost=True)
        ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos), times)
        assert coeff_rel_err(out["coeffs"].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
        assert abs(float(out["cost"][0]) / ref["cost"][0] - 1.0) <= COST_TOL
    if D == 1:
        # chains beyond the reduction's thread budget (K > 513) fall back to the two-lane kernel
        K = 600
        pos, times = random_batch(oracle, 2, K, D=1)
        out = ms.solve_standard(dev(torch, pos), dev(torch, times))
        assert (out["status"] == 0).all()
        mask, values = standard_mask(K), batch_values(pos)
        assert check_path(out["coeffs"].cpu().numpy()[0], times[0], mask, values[0], oracle) < 1e-6


@pytest.mark.parametrize("D", [1, 2, 3])
def test_long_chain_partitioned_route(ms, oracle, torch_cuda, monkeypatch, D):
    """The partitioned route (chunk Schur complements, separator solve, every chunk through the headline kernel;
    minsnap_standard_chunked.cuh) against the cyclic-reduction kernel on every chain length it takes -- K a multiple
    of an even chunk length <= 12 with an even number of chunks -- with non-zero boundary derivatives, device-side
    segment times and all optional outputs, ragged batches included; and against the oracle at K = 256."""
    torch = torch_cuda
    rng = np.random.default_rng(77 + D)
    for K, B in ((32, 5), (40, 3), (48, 17), (64, 33), (96, 2), (120, 1), (128, 40), (192, 7), (256, 19), (384, 4), (512 if D < 3 else 480, 3)):
        pos = np.cumsum(rng.uniform(0.3, 2.0, (B, K + 1, D)) * rng.choice([-1.0, 1.0], (B, K + 1, D)), axis=1)
        ends = rng.normal(size=(B, 2, 4, D))
        outs = {}
        for which in ("bcr", "chunked"):
            outs[which] = solve_on_route(ms, monkeypatch, which, dev(torch, pos), None, end_derivatives=dev(torch, ends),
                                         v_max=3.0, a_max=5.0, want_free=True, want_cost=True, want_times=True)
        a, b = outs["bcr"], outs["chunked"]
        assert (a["status"] == 0).all() and (b["status"] == 0).all(), K
        # the partitioned route runs the stand-alone estimateSegmentTimes kernel, the reduction kernel its own copy
        assert float((a["times"] / b["times"] - 1.0).abs().max()) <= 1e-14
        assert coeff_rel_err(a["coeffs"].cpu().numpy(), b["coeffs"].cpu().numpy()) <= 1e-9, K
        scale = a["free_values"].abs().amax(dim=(1, 2), keepdim=True)
        assert float(((a["free_values"] - b["free_values"]).abs() / scale).max()) <= 1e-9, K
        assert float((a["cost"] / b["cost"] - 1.0).abs().max()) <= 1e-9, K
    # against the oracle, rest-to-rest, given times, K = 256 (BASELINE config 4's shape)
    K = 256
    pos, times = random_batch(oracle, 2, K, D=D)
    out = solve_on_route(ms, monkeypatch, "chunked", dev(torch, pos), dev(torch, times), want_cost=True)
    ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos), times)
    assert (out["status"] == 0).all()
    assert coeff_rel_err(out["coeffs"].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    assert np.abs(out["cost"].cpu().numpy() / ref["cost"] - 1.0).max() <= COST_TOL
    # a non-positive segment time inside a chunk is reported for its trajectory only
    bad = times.copy()
    bad[1, 100] = -1.0
    out = solve_on_route(ms, monkeypatch, "chunked", dev(torch, pos), dev(torch, bad))
    st = out["status"].cpu().numpy()
    assert st[0] == 0 and (st[1] & 2)


def test_long_chain_status_bits(ms, oracle, torch_cuda):
    torch = torch_cuda
    K, B = 64, 4
    pos, times = random_batch(oracle, B, K)
    times[1, 10] = -1.0
    out = ms.solve_standard(dev(torch, pos), dev(torch, times))
    st = out["status"].cpu().numpy()
    assert st[0] == 0 and st[2] == 0 and st[3] == 0
    assert st[1] & 2                                              # MINSNAP_STATUS_BAD_TIME


def test_solve_standard_nonzero_end_derivatives(ms, oracle, torch_cuda):
    torch = torch_cuda
    K, B = 10, 64
    rng = np.random.default_rng(11)
    pos, times = random_batch(oracle, B, K)
    ends = rng.normal(size=(B, 2, 4, 3))
    out = ms.solve_standard(dev(torch, pos), dev(torch, times), end_derivatives=dev(torch, ends), want_cost=True)
    values = batch_values(pos)
    values[:, 0, 1:, :] = ends[:, 0]
    values[:, K, 1:, :] = ends[:, 1]
    ref = oracle_solve_batch(oracle, standard_mask(K), values, times)
    assert coeff_rel_err(out["coeffs"].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    assert np.abs(out["cost"].cpu().numpy() / ref["cost"] - 1.0).max() <= COST_TOL


def test_solve_standard_device_times_and_host_entry(ms, oracle, torch_cuda):
    torch = torch_cuda
    K, B = 10, 300
    pos, times = random_batch(oracle, B, K)
    out = ms.solve_standard(dev(torch, pos), None, v_max=3.0, a_max=5.0, want_times=True)
    t_dev = out["times"].cpu().numpy()
    assert np.abs(t_dev / times - 1.0).max() < 1e-14
    ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos), t_dev)
    assert coeff_rel_err(out["coeffs"].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    # host-buffer entry point == device entry point, bit for bit
    host = ms.solve_standard_host(pos, times, want_cost=True, want_status=True)
    devo = ms.solve_standard(dev(torch, pos), dev(torch, times), want_cost=True)
    assert np.array_equal(host["coeffs"], devo["coeffs"].cpu().numpy())
    assert np.array_equal(host["cost"], devo["cost"].cpu().numpy())
    assert (host["status"] == 0).all()


def test_solve_standard_matches_general_route(ms, oracle, torch_cuda):
    """The fast route and the general kernels are two implementations of the same algebra."""
    torch = torch_cuda
    K, B = 10, 2048
    pos = ms.random_positions_host(B, K, [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0], BASE_SEED)
    pos_d = dev(torch, pos)
    times = ms.estimate_segment_times(pos_d, 3.0, 5.0)
    fast = ms.solve_standard(pos_d, times, want_cost=True)
    mask = standard_mask(K)
    fixed = np.stack([compact_fixed(mask, vertex_values(p)) for p in pos])
    gen = ms.solve(mask, dev(torch, fixed), times)
    assert coeff_rel_err(fast["coeffs"].cpu().numpy(), gen["coeffs"].cpu().numpy()) <= 1e-9
    assert (fast["cost"] / gen["cost"] - 1.0).abs().max().item() <= 1e-9


def test_full_size_properties(ms, oracle, torch_cuda):
    """Config 2 at full size (65,536 x K=10): size-independent properties on the whole batch
    (constraints met, C^4 continuity, linearity in the positions) and oracle parity on a
    random subset of 4096 problems."""
    torch = torch_cuda
    K, B = 10, 65536
    lo, hi = [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0]
    pos = ms.random_positions_host(B, K, lo, hi, BASE_SEED)
    pos_d = dev(torch, pos)
    times = ms.estimate_segment_times(pos_d, 3.0, 5.0)
    out = ms.solve_standard(pos_d, times, want_cost=True)
    assert int((out["status"] != 0).sum().item()) == 0
    c = out["coeffs"]                                                   # [B][K][D][N]
    # derivatives 0..4 at both ends of every segment, evaluated with torch (test code)
    j = torch.arange(N, device="cuda", dtype=torch.float64)
    T = times[:, :, None, None]
    worst_cont, worst_fix = 0.0, 0.0
    for k in range(5):
        fall = torch.ones(N, device="cuda", dtype=torch.float64)
        for q in range(k):
            fall = fall * (j - q)
        at0 = c[..., k] * fall[k]                                         # [B][K][D]
        powers = torch.where(j >= k, T ** (j - k).clamp(min=0), torch.zeros_like(T * j))
        atT = (c * fall * powers).sum(-1)
        worst_cont = max(worst_cont, (atT[:, :-1] - at0[:, 1:]).abs().max().item())
        if k == 0:
            worst_fix = max(worst_fix, (at0 - pos_d[:, :-1]).abs().max().item(), (atT - pos_d[:, 1:]).abs().max().item())
        else:
            worst_fix = max(worst_fix, at0[:, 0].abs().max().item(), atT[:, -1].abs().max().item())
    assert worst_fix < 1e-6 and worst_cont < 1e-6
    # linearity: solve(p + q) == solve(p) + solve(q) for equal segment times
    perm = torch.randperm(B, device="cuda")
    both = ms.solve_standard(pos_d + pos_d[perm], times)["coeffs"]
    second = ms.solve_standard(pos_d[perm].contiguous(), times)["coeffs"]
    scale = c.abs().amax(dim=-1, keepdim=True).clamp(min=1e-300)
    assert ((both - c - second).abs() / scale).max().item() < 1e-7
    # oracle parity on a random subset
    rng = np.random.default_rng(5)
    idx = np.sort(rng.choice(B, 4096, replace=False))
    t_h = times.cpu().numpy()
    ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos[idx]), t_h[idx])
    assert coeff_rel_err(c[torch.from_numpy(idx).cuda()].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    assert np.abs(out["cost"].cpu().numpy()[idx] / ref["cost"] - 1.0).max() <= COST_TOL


# ------------------------------------------------------------------------------------------
# a13 alone, a16 alone
# ------------------------------------------------------------------------------------------
def test_coeffs_from_constraints_and_cost(ms, oracle, torch_cuda):
    torch = torch_cuda
    K, B = 5, 32
    rng = np.random.default_rng(2)
    mask = standard_mask(K, max_fixed_derivative=3)
    pos, times = random_batch(oracle, B, K)
    values = batch_values(pos)
    fixed = np.stack([compact_fixed(mask, v) for v in values])
    col, nf, npf = oracle.reorder(N, K, mask)
    free = rng.normal(size=(B, npf, 3))
    got = ms.coeffs_from_constraints(mask, dev(torch, fixed), dev(torch, free), dev(torch, times)).cpu().numpy()
    got_host = ms.coeffs_from_constraints_host(mask, fixed, free, times)
    assert np.array_equal(got, got_host)
    for b in range(B):
        d_all = np.concatenate([fixed[b], free[b]], axis=0).T.copy()     # [D][n_all]
        want = oracle.coeffs_from_constraints(N, K, 3, col, d_all, times[b])
        assert coeff_rel_err(got[b], want) <= COEFF_TOL
    cost = ms.cost(dev(torch, got), dev(torch, times)).cpu().numpy()
    want_cost = np.array([float(oracle.compute_cost(N, K, 3, SNAP, got[b], times[b])) for b in range(B)])
    # random (non-optimal) free derivatives make c^T Q c a sum of large cancelling terms: the two
    # summation orders agree to ~1e-10; the north-star bar for cost is 1e-8 relative
    assert np.abs(cost / want_cost - 1.0).max() <= 1e-9
    assert np.array_equal(cost, ms.cost_host(got, times))


# ------------------------------------------------------------------------------------------
# a17-a20 sampling
# ------------------------------------------------------------------------------------------
def solved_batch(ms, oracle, torch, B, K):
    pos, times = random_batch(oracle, B, K)
    out = ms.solve_standard(dev(torch, pos), dev(torch, times))
    return out["coeffs"], dev(torch, times), pos, times


@pytest.mark.parametrize("K,B,M", [(10, 16, 1000), (4, 8, 257), (1, 4, 64), (100, 3, 2000)])
def test_sample_uniform_against_oracle(ms, oracle, torch_cuda, K, B, M):
    torch = torch_cuda
    coeffs, times_d, _, times = solved_batch(ms, oracle, torch, B, K)
    out, t = ms.sample_uniform(coeffs, times_d, M, 5, want_times=True)
    out, t = out.cpu().numpy(), t.cpu().numpy()
    c = coeffs.cpu().numpy()
    for b in range(B):
        total = 0.0
        for x in times[b]:
            total += x
        assert np.array_equal(t[b], np.arange(M) * (total / M))
        want = oracle.trajectory_sample(c[b], times[b], t[b], 5)
        assert np.abs(out[b] - want).max() <= SAMPLE_TOL
        scale = np.abs(want).max(axis=(0, 2), keepdims=True)
        assert (np.abs(out[b] - want) / scale).max() <= 1e-11


def test_sample_at_segment_choice_and_range(ms, oracle, torch_cuda):
    torch = torch_cuda
    K, B = 10, 8
    coeffs, times_d, pos, times = solved_batch(ms, oracle, torch, B, K)
    c = coeffs.cpu().numpy()
    ends = np.cumsum(times, axis=1)
    # instants exactly on vertices, just around them, at 0, at/after the end, NaN
    t = np.concatenate([np.zeros((B, 1)), ends, np.nextafter(ends, 0), np.nextafter(ends, 1e9),
                        ends[:, -1:] + 3.0, np.full((B, 1), np.nan)], axis=1)
    out, seg = ms.sample_at(coeffs, times_d, dev(torch, t), 5, want_segment=True)
    out, seg = out.cpu().numpy(), seg.cpu().numpy()
    for b in range(B):
        for m in range(t.shape[1]):
            if np.isnan(t[b, m]):
                assert seg[b, m] == -1 and (out[b, m] == 0).all()
                continue
            for k in range(5):
                want, s_ref = oracle.trajectory_evaluate(c[b], times[b], t[b, m], k)
                assert seg[b, m] == s_ref
                assert np.abs(out[b, m, k] - want).max() <= SAMPLE_TOL
    # shared instants row + host entry point
    shared = np.linspace(0.0, ends.min() * 0.999, 100)
    o1 = ms.sample_at(coeffs, times_d, dev(torch, shared), 3).cpu().numpy()
    o2, _ = ms.sample_at_host(c, times, shared, 3)
    assert np.array_equal(o1, o2)
    want = oracle.trajectory_sample(c[3], times[3], shared, 3)
    assert np.abs(o1[3] - want).max() <= SAMPLE_TOL


@pytest.mark.parametrize("derivative,dt", [(0, 0.01), (1, 0.1), (4, 0.037)])
def test_evaluate_range_against_oracle(ms, oracle, torch_cuda, derivative, dt):
    torch = torch_cuda
    K, B = 10, 6
    coeffs, times_d, _, times = solved_batch(ms, oracle, torch, B, K)
    c = coeffs.cpu().numpy()
    t_end = float(times.sum(axis=1).min())
    max_samples = int(t_end / dt) + 8
    out, t_out, count = ms.evaluate_range(coeffs, times_d, 0.5, t_end, dt, derivative, max_samples)
    out, t_out, count = out.cpu().numpy(), t_out.cpu().numpy(), count.cpu().numpy()
    for b in range(B):
        want, want_t = oracle.trajectory_evaluate_range(c[b], times[b], 0.5, t_end, dt, derivative)
        assert count[b] == len(want_t)
        assert np.array_equal(t_out[b, :count[b]], want_t)              # sequential accumulation, bit-exact
        assert np.abs(out[b, :count[b]] - want).max() <= SAMPLE_TOL
    o_h, t_h, n_h = ms.evaluate_range_host(c[0], times[0], 0.5, t_end, dt, derivative, max_samples)
    assert n_h == count[0] and np.array_equal(o_h, out[0, :n_h]) and np.array_equal(t_h, t_out[0, :n_h])


# ------------------------------------------------------------------------------------------
# config 5: segment-time sweep
# ------------------------------------------------------------------------------------------
def test_cost_sweep_against_oracle(ms, oracle, torch_cuda):
    torch = torch_cuda
    K, B, S = 10, 24, 16
    rng = np.random.default_rng(9)
    pos, times = random_batch(oracle, B, K)
    sweep = times[:, None, :] * (1.0 + 0.2 * (rng.random((B, S, K)) - 0.5))
    sweep[:, 0, :] = times
    cost = ms.cost_sweep(dev(torch, pos), dev(torch, sweep)).cpu().numpy()
    mask = standard_mask(K)
    for b in range(B):
        vals = vertex_values(pos[b])
        want = np.array([float(oracle.solve(N, K, 3, SNAP, mask, vals, sweep[b, s])["cost"]) for s in range(S)])
        assert np.abs(cost[b] / want - 1.0).max() <= COST_TOL


def test_fp64_peak_is_plausible(ms, torch_cuda):
    tf = ms.fp64_peak(3)
    assert 5.0 < tf < 100.0


# ------------------------------------------------------------------------------------------
# edge cases of the batched entry points: ragged batch sizes, empty batch, unaligned buffers, D
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("B", [1, 2, 15, 16, 17, 31, 33, 100])
def test_solve_standard_ragged_batches(ms, oracle, torch_cuda, B):
    torch = torch_cuda
    K = 10
    pos, times = random_batch(oracle, B, K, seed=500 + B)
    out = ms.solve_standard(dev(torch, pos), dev(torch, times), want_cost=True)
    ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos), times)
    assert out["coeffs"].shape == (B, K, 3, N)
    assert coeff_rel_err(out["coeffs"].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    assert np.abs(out["cost"].cpu().numpy() / ref["cost"] - 1.0).max() <= COST_TOL
    assert (out["status"].cpu().numpy() == 0).all()


def test_empty_batches_are_no_ops(ms, torch_cuda):
    torch = torch_cuda
    pos = torch.empty((0, 11, 3), dtype=torch.float64, device="cuda")
    times = torch.empty((0, 10), dtype=torch.float64, device="cuda")
    out = ms.solve_standard(pos, times)
    assert out["coeffs"].shape == (0, 10, 3, 10)
    smp = ms.sample_uniform(out["coeffs"], times, 16, 5)
    assert smp.shape == (0, 16, 5, 3)
    host = ms.solve_standard_host(np.zeros((0, 11, 3)), np.zeros((0, 10)))
    assert host["coeffs"].shape == (0, 10, 3, 10)


def test_unaligned_device_buffers(ms, oracle, torch_cuda):
    """Pointers that are only 8-byte aligned take the 8-byte copy / store paths."""
    torch = torch_cuda
    K, B = 10, 40
    pos, times = random_batch(oracle, B, K, seed=900)
    pos_buf = torch.empty(pos.size + 1, dtype=torch.float64, device="cuda")
    tim_buf = torch.empty(times.size + 1, dtype=torch.float64, device="cuda")
    out_buf = torch.empty(B * K * 3 * N + 1, dtype=torch.float64, device="cuda")
    pos_d = pos_buf[1:].view(B, K + 1, 3)
    tim_d = tim_buf[1:].view(B, K)
    coeffs_d = out_buf[1:].view(B, K, 3, N)
    pos_d.copy_(torch.from_numpy(pos))
    tim_d.copy_(torch.from_numpy(times))
    assert pos_d.data_ptr() % 16 == 8 and coeffs_d.data_ptr() % 16 == 8
    ms.solve_standard(pos_d, tim_d, coeffs=coeffs_d)
    ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos), times)
    assert coeff_rel_err(coeffs_d.cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    smp_buf = torch.empty(B * 64 * 15 + 1, dtype=torch.float64, device="cuda")
    smp = smp_buf[1:].view(B, 64, 5, 3)
    ms.sample_uniform(coeffs_d.contiguous(), tim_d.contiguous(), 64, 5, out=smp)
    aligned = ms.sample_uniform(coeffs_d.contiguous(), tim_d.contiguous(), 64, 5)
    assert torch.equal(smp, aligned)


@pytest.mark.parametrize("D", [1, 2])
def test_solve_standard_other_dimensions(ms, oracle, torch_cuda, D):
    torch = torch_cuda
    K, B = 10, 50
    pos, times = random_batch(oracle, B, K, D, seed=40 + D)
    out = ms.solve_standard(dev(torch, pos), dev(torch, times), want_free=True, want_cost=True)
    ref = oracle_solve_batch(oracle, standard_mask(K), batch_values(pos), times)
    assert coeff_rel_err(out["coeffs"].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL
    assert np.abs(out["cost"].cpu().numpy() / ref["cost"] - 1.0).max() <= COST_TOL
    want = np.transpose(ref["d_free"], (0, 2, 1))
    scale = np.abs(want).max(axis=(1, 2), keepdims=True)
    assert (np.abs(out["free_values"].cpu().numpy() - want) / scale).max() <= 1e-8


@pytest.mark.parametrize("K", [2, 4, 5, 6, 7, 8, 9, 10, 11, 12])
@pytest.mark.parametrize("D", [1, 2, 3])
def test_two_kernel_generations_agree(ms, oracle, torch_cuda, monkeypatch, K, D):
    """The second-generation kernel (tensor-memory block storage, TMA copy-out: K = 2 and 4 <= K <= 12, odd K with
    the bottom-up lane one block short) against the
    first-generation thread-pair kernel on the same inputs, with non-zero end derivatives, cost, status,
    free derivatives, a ragged batch, and times computed on the device."""
    torch = torch_cuda
    B = 16 * 9 + 5
    rng = np.random.default_rng(4242 + 10 * K + D)
    # random walks whose steps are at least 1 in every dimension: consecutive vertices stay apart also for D = 1
    steps = rng.uniform(1.0, 4.0, size=(B, K + 1, D)) * rng.choice([-1.0, 1.0], size=(B, K + 1, D))
    pos = np.cumsum(steps, axis=1)
    end = rng.uniform(-1.0, 1.0, size=(B, 2, 4, D))
    pos_d, end_d = dev(torch, pos), dev(torch, end)
    results = {}
    for name in ("tm", "pair"):
        results[name] = solve_on_route(ms, monkeypatch, name, pos_d, None, end_derivatives=end_d, v_max=3.0, a_max=5.0,
                                       want_cost=True, want_free=True, want_times=True)
        torch.cuda.synchronize()
    a, b = results["tm"], results["pair"]
    assert int((a["status"] != 0).sum()) == 0 and int((b["status"] != 0).sum()) == 0
    assert np.array_equal(a["times"].cpu().numpy(), b["times"].cpu().numpy())
    assert coeff_rel_err(a["coeffs"].cpu().numpy(), b["coeffs"].cpu().numpy()) <= 1e-10
    fa, fb = a["free_values"].cpu().numpy(), b["free_values"].cpu().numpy()
    if fb.size:
        assert np.abs(fa - fb).max() <= 1e-12 * max(1.0, np.abs(fb).max())
    assert np.abs(a["cost"].cpu().numpy() / b["cost"].cpu().numpy() - 1.0).max() <= 1e-10
    # and against the oracle (reference-order arithmetic) on a few problems
    t = a["times"].cpu().numpy()
    mask = standard_mask(K)
    for i in (0, B // 2, B - 1):
        vals = np.zeros((K + 1, 5, D))
        vals[:, 0, :] = pos[i]
        vals[0, 1:, :] = end[i, 0]
        vals[K, 1:, :] = end[i, 1]
        ref = oracle.solve(10, K, D, 4, mask, vals, t[i])
        assert coeff_rel_err(a["coeffs"][i].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL


@pytest.mark.parametrize("K,D", [(4, 2), (12, 1), (10, 3), (9, 3), (5, 2)])
def test_two_batches_per_warp(ms, oracle, torch_cuda, monkeypatch, K, D):
    """Above two waves of CTAs a warp of the second-generation kernel takes two batches (second input buffer,
    one allocation / table / drain per CTA): a ragged batch just above that threshold against the first-generation
    kernel, with non-zero end derivatives, cost, free derivatives and device-side times."""
    torch = torch_cuda
    B = 2 * 296 * 64 + 5 * 64 + 7
    rng = np.random.default_rng(999 + 10 * K + D)
    steps = rng.uniform(1.0, 4.0, size=(B, K + 1, D)) * rng.choice([-1.0, 1.0], size=(B, K + 1, D))
    pos = np.cumsum(steps, axis=1)
    end = rng.uniform(-1.0, 1.0, size=(B, 2, 4, D))
    pos_d, end_d = dev(torch, pos), dev(torch, end)
    results = {}
    for name in ("tm", "pair"):
        results[name] = solve_on_route(ms, monkeypatch, name, pos_d, None, end_derivatives=end_d, v_max=3.0, a_max=5.0,
                                       want_cost=True, want_free=True, want_times=True)
        torch.cuda.synchronize()
    a, b = results["tm"], results["pair"]
    assert int((a["status"] != 0).sum()) == 0 and int((b["status"] != 0).sum()) == 0
    assert torch.equal(a["times"], b["times"])
    ca, cb = a["coeffs"], b["coeffs"]
    scale = cb.abs().amax(dim=3, keepdim=True).clamp_min(1e-300)
    assert float(((ca - cb).abs() / scale).max()) <= 1e-10
    assert float((a["cost"] / b["cost"] - 1.0).abs().max()) <= 1e-10
    assert float((a["free_values"] - b["free_values"]).abs().max()) <= 1e-12 * max(1.0, float(b["free_values"].abs().max()))
    # the last, ragged batch against the oracle
    t = a["times"].cpu().numpy()
    mask = standard_mask(K)
    for i in (0, B - 1):
        vals = np.zeros((K + 1, 5, D))
        vals[:, 0, :] = pos[i]
        vals[0, 1:, :] = end[i, 0]
        vals[K, 1:, :] = end[i, 1]
        ref = oracle.solve(10, K, D, 4, mask, vals, t[i])
        assert coeff_rel_err(a["coeffs"][i].cpu().numpy(), ref["coeffs"]) <= COEFF_TOL


def test_partitioned_route_two_batches_per_warp(ms, torch_cuda, monkeypatch):
    """The partitioned long-chain route with more chunks than two waves of the headline kernel (4,800 x K = 64 is
    38,400 chunks of 8 segments, 8 per trajectory: a warp's batch of 16 chunks spans two trajectories) against the
    cyclic-reduction kernel."""
    torch = torch_cuda
    B, K, D = 4800, 64, 3
    rng = np.random.default_rng(31337)
    pos = np.cumsum(rng.uniform(0.3, 2.0, (B, K + 1, D)) * rng.choice([-1.0, 1.0], (B, K + 1, D)), axis=1)
    ends = rng.normal(size=(B, 2, 4, D))
    outs = {}
    for which in ("bcr", "chunked"):
        outs[which] = solve_on_route(ms, monkeypatch, which, dev(torch, pos), None, end_derivatives=dev(torch, ends),
                                     v_max=3.0, a_max=5.0, want_cost=True)
        torch.cuda.synchronize()
    a, b = outs["bcr"], outs["chunked"]
    assert (a["status"] == 0).all() and (b["status"] == 0).all()
    scale = a["coeffs"].abs().amax(dim=3, keepdim=True).clamp_min(1e-300)
    assert float(((a["coeffs"] - b["coeffs"]).abs() / scale).max()) <= 1e-9
    assert float((a["cost"] / b["cost"] - 1.0).abs().max()) <= 1e-9


def test_forced_route_never_falls_back(ms, oracle, torch_cuda, monkeypatch):
    """A route forced through MINSNAP_STANDARD_ROUTE that cannot take the call is an error, not another kernel; so
    is a name that is no route."""
    torch = torch_cuda
    for route, K in (("tm", 3), ("chunked", 50)):
        pos, times = random_batch(oracle, 4, K)
        with pytest.raises(ms.MinsnapError) as err:
            solve_on_route(ms, monkeypatch, route, dev(torch, pos), dev(torch, times))
        assert err.value.code == ms.capi.ERR_UNSUPPORTED, route
    pos, times = random_batch(oracle, 4, 10)
    with pytest.raises(ms.MinsnapError) as err:
        solve_on_route(ms, monkeypatch, "no_such_route", dev(torch, pos), dev(torch, times))
    assert err.value.code == ms.capi.ERR_ARG


def test_second_generation_status_bits(ms, torch_cuda):
    """A non-positive segment time is flagged by the recovery phase of the second-generation kernel."""
    torch = torch_cuda
    K, B = 10, 40
    rng = np.random.default_rng(77)
    pos = np.cumsum(rng.uniform(1.0, 4.0, size=(B, K + 1, 3)), axis=1)
    times = rng.uniform(1.0, 3.0, size=(B, K))
    times[7, 3] = -1.0
    times[33, 9] = 0.0
    out = ms.solve_standard(dev(torch, pos), dev(torch, times))
    st = out["status"].cpu().numpy()
    assert st[7] & 2 and st[33] & 2
    assert int((st[np.setdiff1d(np.arange(B), [7, 33])] != 0).sum()) == 0


def test_randomised_shapes_fast_route_vs_general_route(ms, torch_cuda):
    """120 random (K, D, B) shapes, boundary derivatives and time sources: the standard-mask kernels (two-lane,
    cyclic reduction) against the general banded kernel, two independent implementations of the same algebra
    that are each checked against the oracle elsewhere."""
    torch = torch_cuda
    rng = np.random.default_rng(20261018)
    worst = 0.0
    for trial in range(120):
        K = int(rng.integers(1, 41))
        D = int(rng.integers(1, 4))
        B = int(rng.integers(1, 70))
        pos = np.cumsum(rng.uniform(0.4, 3.0, (B, K + 1, D)) * rng.choice([-1.0, 1.0], (B, K + 1, D)), axis=1)
        ends = rng.normal(size=(B, 2, 4, D)) if trial % 3 else None
        pos_d = dev(torch, pos)
        if trial % 2:
            times = ms.estimate_segment_times(pos_d, 2.0 + 3.0 * rng.random(), 2.0 + 4.0 * rng.random())
            fast = ms.solve_standard(pos_d, times, end_derivatives=None if ends is None else dev(torch, ends),
                                     want_free=True, want_cost=True)
        else:
            v, a = 2.0 + 3.0 * rng.random(), 2.0 + 4.0 * rng.random()
            fast = ms.solve_standard(pos_d, None, end_derivatives=None if ends is None else dev(torch, ends), v_max=v,
                                     a_max=a, want_free=True, want_cost=True, want_times=True)
            times = fast["times"]
        mask = standard_mask(K)
        values = np.zeros((B, K + 1, 5, D))
        values[:, :, 0, :] = pos
        if ends is not None:
            values[:, 0, 1:, :] = ends[:, 0]
            values[:, K, 1:, :] = ends[:, 1]
        fixed = np.stack([compact_fixed(mask, v_) for v_ in values])
        gen = ms.solve(mask, dev(torch, fixed), times)
        assert (fast["status"] == 0).all() and (gen["status"] == 0).all(), (trial, K, D, B)
        err = coeff_rel_err(fast["coeffs"].cpu().numpy(), gen["coeffs"].cpu().numpy())
        worst = max(worst, err)
        assert err <= 1e-8, (trial, K, D, B, err)
        assert float((fast["cost"] / gen["cost"] - 1.0).abs().max()) <= 1e-8, (trial, K, D, B)
        if K > 1:
            scale = gen["free_values"].abs().amax(dim=(1, 2), keepdim=True).clamp_min(1e-300)
            assert float(((fast["free_values"] - gen["free_values"]).abs() / scale).max()) <= 1e-8, (trial, K, D, B)
    assert worst > 0.0
