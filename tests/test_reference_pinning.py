"""The oracle against the REFERENCE ITSELF (CPU).  oracle/_ref/libmav_ref_core.so is the reference's own
src/vertex.cpp, polynomial.cpp, segment.cpp, trajectory.cpp, motion_defines.cpp and rpoly.cpp compiled from the
reference's sources against the Eigen / glog stand-ins of oracle/ref_shim/ (oracle/Makefile target `ref`).  Everything
whose arithmetic order is the same is required to agree BIT FOR BIT: the input generator, the segment-time heuristic,
the base-coefficient table, Horner evaluation, the segment search of Trajectory::evaluate, the time accumulation of
evaluateRange, the candidate polynomial of the extrema search.  Extrema values depend on the root finder
(Jenkins-Traub in the reference, interval isolation in the oracle) and agree to 1e-8.

Without the library the bit-exact tests compare with what it returned for the same calls, stored in
tests/golden/reference_pinning.npz (tests/golden/README.md: provenance, and how to regenerate it from the library).
The tests marked live_only need the library itself."""
import hashlib
import os

import numpy as np
import pytest

from oracle.oracle_py import Oracle, ReferenceCore, standard_mask, vertex_values_from_positions

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pinning.npz")
LIVE = ReferenceCore.available()
live_only = pytest.mark.skipif(not LIVE, reason="needs the reference library oracle/_ref/libmav_ref_core.so")
INLINE_BYTES = 8192     # larger return values are stored as their SHA-256 and shape


def _call_key(name, args, index):
    h = hashlib.sha256(name.encode())
    for a in args:
        h.update(np.ascontiguousarray(np.asarray(a, np.float64)).tobytes() + b"|")
    return "%s#%s" % (h.hexdigest()[:40], index)


class Digest:
    """A stored return value too large to keep: its shape and the SHA-256 of its float64 bytes."""

    def __init__(self, sha, shape):
        self.sha, self.shape = sha, shape

    def __len__(self):
        return self.shape[0]


def same(got, want):
    """np.array_equal, also against a Digest."""
    if isinstance(want, Digest):
        got = np.ascontiguousarray(np.asarray(got, np.float64))
        return got.shape == want.shape and hashlib.sha256(got.tobytes()).hexdigest() == want.sha
    return np.array_equal(got, want)


class GoldenReference:
    """Answers the bit-exact tests' calls of ReferenceCore's methods from the stored return values."""

    def __init__(self, path):
        z = np.load(path)
        self.entries = {}
        for k, kind, shape, lo, hi, sha in zip(z["key"], z["kind"], z["shape"], z["start"], z["stop"], z["sha"]):
            shape = tuple(int(n) for n in shape if n >= 0)
            if kind == 1:
                self.entries[k.decode()] = Digest(sha.decode(), shape)
            else:
                v = z["values"][lo:hi].reshape(shape)
                self.entries[k.decode()] = float(v) if shape == () else v

    def __getattr__(self, name):
        def call(*args):
            single = self.entries.get(_call_key(name, args, -1))
            if single is not None:
                return single
            out, i = [], 0
            while _call_key(name, args, i) in self.entries:
                out.append(self.entries[_call_key(name, args, i)])
                i += 1
            assert out, "no stored reference result for %s; regenerate %s from the library" % (name, GOLDEN)
            return tuple(out)
        return call


class RecordingReference:
    """Wraps the live library and writes every call's return value in GoldenReference's format (regeneration:
    tests/golden/README.md)."""

    def __init__(self, lib):
        self.lib, self.calls = lib, {}

    def __getattr__(self, name):
        def call(*args):
            r = getattr(self.lib, name)(*args)
            for i, v in ([(-1, r)] if not isinstance(r, tuple) else enumerate(r)):
                self.calls[_call_key(name, args, i)] = np.asarray(v, np.float64)
            return r
        return call

    def save(self, path):
        keys, kind, shape, start, stop, sha, values, n = [], [], [], [], [], [], [], 0
        for k, v in sorted(self.calls.items()):
            v = np.ascontiguousarray(v)
            keys.append(k)
            shape.append(list(v.shape) + [-1] * (2 - v.ndim))
            big = v.nbytes > INLINE_BYTES
            kind.append(1 if big else 0)
            sha.append(hashlib.sha256(v.tobytes()).hexdigest() if big else "")
            start.append(n)
            if not big:
                values.append(v.reshape(-1))
                n += v.size
            stop.append(n)
        np.savez_compressed(path, key=np.array(keys, "S"), kind=np.array(kind, np.int8), shape=np.array(shape, np.int64),
                            start=np.array(start, np.int64), stop=np.array(stop, np.int64), sha=np.array(sha, "S"),
                            values=np.concatenate(values))


BOX_LO, BOX_HI = [-10.0, -20.0, -10.0], [10.0, 20.0, 10.0]


@pytest.fixture(scope="module")
def ref():
    """The library when it is present (REFERENCE_PINNING_RECORD=1 also rewrites the golden file from it), else the
    stored return values."""
    if not LIVE:
        yield GoldenReference(GOLDEN)
    elif os.environ.get("REFERENCE_PINNING_RECORD") == "1":
        rec = RecordingReference(ReferenceCore())
        yield rec
        rec.save(GOLDEN)
    else:
        yield ReferenceCore()


@pytest.fixture(scope="module")
def orc():
    return Oracle("f64")


@pytest.fixture(scope="module")
def solved(orc):
    """A few solved trajectories (oracle coefficients) to evaluate with both sides."""
    out = []
    for K, seed in ((4, 12345), (10, 978), (10, 12346), (25, 4711)):
        pos = orc.create_random_positions(K, BOX_LO, BOX_HI, seed)
        times = orc.estimate_segment_times(pos, 3.0, 5.0, 6.5)
        sol = orc.solve(10, K, 3, 4, standard_mask(K), vertex_values_from_positions(pos), times)
        out.append((np.asarray(sol["coeffs"], np.float64), np.asarray(times, np.float64)))
    return out


@pytest.mark.parametrize("seed", [12, 123, 1234, 12345, 978, 12345 + 65535])
@pytest.mark.parametrize("K", [1, 4, 10, 100])
def test_create_random_vertices_bit_exact(ref, orc, seed, K):
    """ref createRandomVertices (src/vertex.cpp:27-79): draw order, rejection rule, constraint counts."""
    pos, n_constraints = ref.create_random_positions(4, K, BOX_LO, BOX_HI, seed)
    assert np.array_equal(pos, orc.create_random_positions(K, BOX_LO, BOX_HI, seed))
    want = np.ones(K + 1, np.int32)
    want[0] = want[K] = 5          # makeStartOrEnd(position, 4): derivatives 0..4
    assert np.array_equal(n_constraints, want)
    # 1-D variant of the reference's tests (createRandomVertices1D)
    pos1, _ = ref.create_random_positions(4, K, [-50.0], [50.0], seed)
    assert np.array_equal(pos1, orc.create_random_positions(K, [-50.0], [50.0], seed))


@pytest.mark.parametrize("v_a", [(3.0, 5.0), (2.0, 2.0), (1.0, 10.0)])
def test_estimate_segment_times_bit_exact(ref, orc, v_a):
    """ref estimateSegmentTimes (src/vertex.cpp:162-178)."""
    for seed in (12345, 978, 5):
        pos = orc.create_random_positions(50, BOX_LO, BOX_HI, seed)
        assert np.array_equal(ref.estimate_segment_times(pos, v_a[0], v_a[1], 6.5),
                              orc.estimate_segment_times(pos, v_a[0], v_a[1], 6.5))


def test_base_coefficients_bit_exact(ref, orc):
    """ref computeBaseCoefficients (src/polynomial.cpp:140-155), the 22 x 22 table and smaller ones."""
    for n in (4, 10, 12, 22):
        assert np.array_equal(ref.base_coefficients(n), orc.base_coefficients(n))


def test_base_coeffs_with_time_match_mapping_matrix(ref, orc):
    """ref baseCoeffsWithTime (polynomial.h:215-233) builds the rows of A (LIN.i:101-111)."""
    for N in (6, 10, 12):
        for T in (0.0, 0.7, 3.0, 25.0):
            A = orc.mapping_matrix(N, T)
            for d in range(N // 2):
                assert np.array_equal(A[d], ref.base_coeffs_with_time(N, d, 0.0))
                assert np.array_equal(A[N // 2 + d], ref.base_coeffs_with_time(N, d, T))


def test_polynomial_evaluate_bit_exact(ref, orc):
    """ref Polynomial::evaluate(t, derivative) and evaluate(t, VectorXd*) (polynomial.h:120-151)."""
    rng = np.random.default_rng(3)
    for N in (4, 10, 12):
        for _ in range(40):
            c = rng.normal(size=N) * 10.0 ** rng.integers(-6, 3, size=N)
            t = float(rng.uniform(-2.0, 30.0))
            every = ref.polynomial_evaluate_all(c, t, min(N, 6))
            for d in range(N + 2):
                got = orc.polynomial_evaluate(c, t, d)
                assert got == ref.polynomial_evaluate(c, t, d)
                if d < len(every):
                    assert got == every[d]


@live_only
def test_candidate_polynomial_bit_exact(ref, orc, solved):
    """ref Segment::computeMinMaxMagnitudeCandidateTimes (src/segment.cpp:93-116): getCoefficients, head, convolve
    and the order in which the dimensions are added."""
    for coeffs, _ in solved:
        for seg in coeffs[:: max(1, len(coeffs) // 4)]:
            for k in (0, 1, 2, 3):
                N = seg.shape[1]
                want = np.zeros((N - k) + (N - k - 1) - 1)
                for d in range(seg.shape[0]):
                    a = ref.polynomial_get_coefficients(seg[d], k)[: N - k]
                    b = ref.polynomial_get_coefficients(seg[d], k + 1)[: N - k - 1]
                    want = want + ref.convolve(a, b)
                got = orc.candidate_polynomial(seg, k)
                assert np.array_equal(got[: len(want)], want)


def test_trajectory_evaluate_bit_exact(ref, orc, solved):
    """ref Segment::evaluate (src/segment.cpp:51-58) and Trajectory::evaluate (src/trajectory.cpp:41-66):
    the strict '>' segment choice (a vertex instant belongs to the segment on its right), local time."""
    rng = np.random.default_rng(11)
    for coeffs, times in solved:
        total = ref.trajectory_max_time(coeffs, times)
        acc = np.cumsum(times)
        instants = list(rng.uniform(0.0, total, size=60)) + list(acc[:-1]) + list(np.nextafter(acc[:-1], 0.0)) + \
            list(np.nextafter(acc[:-1], np.inf)) + [0.0]
        for t in instants:
            if not t < total:
                continue
            for d in range(5):
                want = ref.trajectory_evaluate(coeffs, times, float(t), d)
                got, _ = orc.trajectory_evaluate(coeffs, times, float(t), d)
                assert np.array_equal(got, want), (t, d)
        for k, T in enumerate(times[:3]):
            for t in (0.0, 0.3 * T, T):
                for d in range(5):
                    want = ref.segment_evaluate(coeffs[k], T, t, d)
                    got = np.array([orc.polynomial_evaluate(coeffs[k][dim], t, d) for dim in range(3)])
                    assert np.array_equal(got, want)


@pytest.mark.parametrize("dt", [0.01, 0.1, 0.37])
def test_evaluate_range_bit_exact(ref, orc, solved, dt):
    """ref Trajectory::evaluateRange (src/trajectory.cpp:68-128): sample count, sampling times (accumulated, not
    multiplied) and values."""
    for coeffs, times in solved:
        total = float(np.sum(times))
        for t0, t1 in ((0.0, total), (0.0, 0.5 * total), (0.31 * total, 0.9 * total), (times[0], total)):
            for d in (0, 2):
                want, want_t = ref.trajectory_evaluate_range(coeffs, times, t0, t1, dt, d)
                got, got_t = orc.trajectory_evaluate_range(coeffs, times, t0, t1, dt, d)
                assert len(got) == len(want)
                assert same(got_t, want_t)
                assert same(got, want)


@live_only
def test_minmax_magnitude_against_reference(ref, orc, solved):
    """ref Trajectory::computeMinMaxMagnitude (src/trajectory.cpp:181-217) over the reference's own Jenkins-Traub
    roots, against the oracle's interval isolation: extremal values to 1e-8 relative, same segment."""
    for coeffs, times in solved:
        for k in (1, 2):
            ok, mn, mx = ref.trajectory_minmax_magnitude(coeffs, times, k)
            assert ok
            r = orc.minmax_magnitude(coeffs, times, k, 1)
            assert abs(r["max"][1] - mx[1]) <= 1e-8 * max(1.0, abs(mx[1]))
            assert abs(r["min"][1] - mn[1]) <= 1e-8 * max(1.0, abs(mn[1]))
            assert r["max"][2] == mx[2]
            # one dimension: Polynomial::computeMinMax route (src/polynomial.cpp:95-108)
            ok, mn1, mx1 = ref.trajectory_minmax_magnitude(coeffs, times, k, dims=[1])
            r1 = orc.minmax_magnitude(coeffs, times, k, 1, dims=[1])
            assert ok and abs(r1["max"][1] - mx1[1]) <= 1e-8 * max(1.0, abs(mx1[1]))


@live_only
def test_segment_candidates_against_reference(ref, orc, solved):
    """ref Segment::computeMinMaxMagnitudeCandidates (src/segment.cpp:132-156): the largest candidate value of an
    inner segment agrees with the oracle's segment maximum."""
    coeffs, times = solved[1]
    for s in (2, 5, 7):
        got = ref.segment_minmax_candidates(coeffs[s], times[s], 1, 0.0, times[s])
        assert got is not None
        _, values = got
        cand = orc.segment_candidate_roots(coeffs[s], 1, 0.0, times[s])
        best = max([orc.segment_magnitude(coeffs[s], 1, t) for t in list(cand) + [0.0, times[s]]])
        ref_best = max(list(values) + [orc.segment_magnitude(coeffs[s], 1, 0.0), orc.segment_magnitude(coeffs[s], 1, times[s])])
        assert abs(best - ref_best) <= 1e-8 * max(1.0, ref_best)


def test_product_input_generator_against_reference(ref):
    """The product's host-side createRandomVertices (csrc/minsnap_host_inputs.cpp, no GPU involved) against the
    reference's own function, bit for bit."""
    import mav_trajectory_generation_cmake_b200 as ms
    got = ms.random_positions_host(64, 10, BOX_LO, BOX_HI, 12345)
    for b in (0, 1, 17, 63):
        want, _ = ref.create_random_positions(4, 10, BOX_LO, BOX_HI, 12345 + b)
        assert np.array_equal(got[b], want)


@live_only
@pytest.mark.gpu
def test_gpu_path_against_reference_itself(ref):
    """Solve on the GPU, then sample and evaluate ranges on the GPU, and compare with the REFERENCE's own
    Trajectory::evaluate / evaluateRange / estimateSegmentTimes on the GPU's coefficients (no oracle in between)."""
    import torch
    import mav_trajectory_generation_cmake_b200 as ms
    B, K = 32, 10
    pos = ms.random_positions_host(B, K, BOX_LO, BOX_HI, 978)
    pos_d = torch.from_numpy(pos).cuda()
    times_d = ms.estimate_segment_times(pos_d, 3.0, 5.0)
    times = times_d.cpu().numpy()
    for b in range(B):
        want = ref.estimate_segment_times(pos[b], 3.0, 5.0, 6.5)
        assert np.abs(times[b] - want).max() <= 4e-16 * np.abs(want).max()
    out = ms.solve_standard(pos_d, times_d)
    coeffs = out["coeffs"].cpu().numpy()
    samples, ts = ms.sample_uniform(out["coeffs"], times_d, 97, 5, want_times=True)
    samples, ts = samples.cpu().numpy(), ts.cpu().numpy()
    for b in range(0, B, 5):
        for m in range(0, 97, 3):
            for d in range(5):
                want = ref.trajectory_evaluate(coeffs[b], times[b], float(ts[b, m]), d)
                assert np.abs(samples[b, m, d] - want).max() <= 1e-6
    vals, t_out, count = ms.evaluate_range(out["coeffs"][:4], times_d[:4], 0.0, float(times[:4].sum(1).min()), 0.05, 1, 4096)
    vals, t_out, count = vals.cpu().numpy(), t_out.cpu().numpy(), count.cpu().numpy()
    for b in range(4):
        want, want_t = ref.trajectory_evaluate_range(coeffs[b], times[b], 0.0, float(times[:4].sum(1).min()), 0.05, 1)
        assert count[b] == len(want)
        assert np.array_equal(t_out[b, : count[b]], want_t)
        assert np.abs(vals[b, : count[b]] - want).max() <= 1e-6
