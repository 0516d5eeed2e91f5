"""Shared test helpers: problem generators built on the oracle, and the parity metrics.

Tolerances (BASELINE.json north_star, SURVEY.md section 8d):
  * index maps, n_fixed, n_free                      bit-exact
  * coefficients: per-polynomial max-norm relative   <= 1e-8   (COEFF_TOL)
  * sampled derivatives 0..4                          <= 1e-6 absolute (SAMPLE_TOL)
  * cost                                              <= 1e-8 relative (COST_TOL)
"""
import numpy as np

COEFF_TOL = 1e-8
SAMPLE_TOL = 1e-6
COST_TOL = 1e-8

BOX_MIN = np.array([-10.0, -20.0, -10.0])
BOX_MAX = np.array([10.0, 20.0, 10.0])
BASE_SEED = 12345


def standard_mask(K, N=10, max_fixed_derivative=None):
    h = N // 2
    if max_fixed_derivative is None:
        max_fixed_derivative = h - 1
    m = np.zeros((K + 1, h), np.uint8)
    m[:, 0] = 1
    m[0, : max_fixed_derivative + 1] = 1
    m[K, : max_fixed_derivative + 1] = 1
    return m


def random_batch(oracle, B, K, D=3, seed=BASE_SEED, v_max=3.0, a_max=5.0, box=None):
    """positions[B][K+1][D], times[B][K] exactly as the reference's tests make them
    (createRandomVertices seed + b, estimateSegmentTimes).  box=None: the 3-D box of
    test_polynomial_optimization.cpp:357-361, else the cube [-box, box]^D."""
    if box is None:
        lo, hi = (BOX_MIN, BOX_MAX) if D == 3 else (-10.0 * np.ones(D), 10.0 * np.ones(D))
    else:
        lo, hi = -box * np.ones(D), box * np.ones(D)
    pos = np.stack([oracle.create_random_positions(K, lo, hi, seed + b) for b in range(B)])
    times = np.stack([oracle.estimate_segment_times(pos[b], v_max, a_max) for b in range(B)])
    return pos, times.astype(np.float64)


def vertex_values(positions, N=10):
    """[K+1][D] -> [K+1][h][D] constraint table with zero derivatives."""
    K1, D = positions.shape
    v = np.zeros((K1, N // 2, D), positions.dtype)
    v[:, 0, :] = positions
    return v


def compact_fixed(mask, values):
    """values[(K+1)][h][D] -> fixed_values[n_fixed][D] in (vertex, derivative) order."""
    mask = np.asarray(mask, bool)
    return values[mask]


def oracle_solve_batch(oracle, mask, values, times, N=10, derivative=4):
    """values[B][(K+1)][h][D] -> dict of stacked oracle outputs (coeffs [B][K][D][N] ...)."""
    B = values.shape[0]
    K = mask.shape[0] - 1
    D = values.shape[-1]
    outs = [oracle.solve(N, K, D, derivative, mask, values[b], times[b]) for b in range(B)]
    return dict(
        coeffs=np.stack([o["coeffs"] for o in outs]).astype(np.float64),
        d_free=np.stack([o["d_free"] for o in outs]).astype(np.float64),   # [B][D][n_free]
        d_fixed=np.stack([o["d_fixed"] for o in outs]).astype(np.float64),
        cost=np.array([float(o["cost"]) for o in outs]),
        status=np.array([o["status"] for o in outs]),
    )


def coeff_rel_err(c, c_ref):
    """Per-polynomial max-norm relative error, maximised over the batch."""
    c = np.asarray(c, np.float64)
    c_ref = np.asarray(c_ref, np.float64)
    num = np.abs(c - c_ref).max(axis=-1)
    den = np.abs(c_ref).max(axis=-1)
    den = np.where(den == 0, 1.0, den)
    return float((num / den).max())


def check_path(coeffs, times, mask, values, oracle, tol=1e-6, N=10):
    """The reference's checkPath (test/test_polynomial_optimization.cpp:73-131) for one
    trajectory: fixed constraints met at both segment ends, derivatives 0..h-1 continuous."""
    K, D, _ = coeffs.shape
    h = N // 2
    worst = 0.0
    for i in range(K):
        for end, v in ((0, i), (1, i + 1)):
            t = 0.0 if end == 0 else times[i]
            for c in range(h):
                if mask[v, c]:
                    for d in range(D):
                        val = float(oracle.polynomial_evaluate(coeffs[i, d], t, c))
                        worst = max(worst, abs(val - values[v, c, d]))
        if i > 0:
            for c in range(h):
                for d in range(D):
                    a = float(oracle.polynomial_evaluate(coeffs[i - 1, d], times[i - 1], c))
                    b = float(oracle.polynomial_evaluate(coeffs[i, d], 0.0, c))
                    worst = max(worst, abs(a - b))
    return worst


# ---- time-only objective and numeric time gradient, literally as the reference computes them ----
def oracle_objective(oracle, pos, times, penalty):
    K = times.shape[0]
    r = oracle.solve(10, K, pos.shape[1], 4, standard_mask(K), vertex_values(pos), times)
    total = 0.0
    for t in times:
        total += t
    return float(r["cost"]) + total * total * penalty, float(r["cost"])


def oracle_gradient(oracle, pos, times, increment, w_d, w_t):
    K, D = times.shape[0], pos.shape[1]
    mask, vals = standard_mask(K), vertex_values(pos)
    base = oracle.solve(10, K, D, 4, mask, vals, times)
    d_all = np.concatenate([base["d_fixed"], base["d_free"]], axis=1)   # [D][n_fixed + n_free]

    def J_d(t):
        R = oracle.solve(10, K, D, 4, mask, vals, t, want_R=True)["R"]
        return float(sum(d_all[k] @ R @ d_all[k] for k in range(D)))

    grad = np.zeros(K)
    for n in range(K):
        smaller, bigger = times.copy(), times.copy()
        smaller[n] = 0.1 if smaller[n] <= 0.1 else smaller[n] - increment
        bigger[n] = 0.1 if bigger[n] <= 0.1 else bigger[n] + increment
        grad[n] = w_d * (J_d(bigger) - J_d(smaller)) / (2.0 * increment) + w_t
    return grad, J_d(times)


def banded_ld_solve(oracle_ld, N, derivative, mask, values, times):
    """The linear solve of one trajectory in long double, in O(K): R_pp d_p = -R_pf d_f by banded elimination.

    R is assembled from oracle_ld.segment_hessian and the column map of oracle.reorder exactly as the dense oracle
    assembles it (R[col[i N + r]][col[i N + s]] += H_i[r][s]).  Free columns are ordered by (vertex, derivative), so
    two free columns that share a segment are at most N - 1 apart: R_pp has half bandwidth N - 1.  The reference's
    A^-T Q A^-1 is symmetric only to ~1e-14 relative, so both halves of the band are kept (an LDL^T of the lower half
    would differ from the dense oracle by that asymmetry times the condition number, 1e-10 at K = 64).
    mask[(K+1)][h], values[(K+1)][h][D], times[K] -> coeffs [K][D][N], d_free [n_free][D], cost (long double)."""
    mask = np.asarray(mask, bool)
    K, D = mask.shape[0] - 1, values.shape[-1]
    col, nf, npf = oracle_ld.reorder(N, K, mask)
    col = col.reshape(K, N)
    ld, w = np.longdouble, N - 1
    d = np.zeros((nf + npf, D), ld)
    d[:nf] = np.asarray(values, ld)[mask]              # fixed columns in (vertex, derivative) order
    band = np.zeros((npf + w, 2 * w + 1), ld)          # band[c][w + j] = R_pp[c][c + j]
    rhs = np.zeros((npf + w, D), ld)                   # -R_pf d_f
    for i in range(K):
        H = oracle_ld.segment_hessian(N, derivative, times[i])
        for r in range(N):
            cr = col[i, r]
            if cr < nf:
                continue
            for s in range(N):
                cs = col[i, s]
                if cs < nf:
                    rhs[cr - nf] -= H[r, s] * d[cs]
                else:
                    band[cr - nf, w + cs - cr] += H[r, s]
    for c in range(npf):                               # elimination without pivoting, forward substitution
        for j in range(1, w + 1):
            f = band[c + j, w - j] / band[c, w]
            band[c + j, w - j : 2 * w + 1 - j] -= f * band[c, w:]
            rhs[c + j] -= f * rhs[c]
    x = np.zeros((npf + w, D), ld)
    for c in range(npf - 1, -1, -1):
        x[c] = (rhs[c] - band[c, w + 1 :] @ x[c + 1 : c + w + 1]) / band[c, w]
    d[nf:] = x[:npf]
    coeffs = oracle_ld.coeffs_from_constraints(N, K, D, col.ravel(), np.ascontiguousarray(d.T), times)
    return coeffs, d[nf:].copy(), oracle_ld.compute_cost(N, K, D, derivative, coeffs, times)
