// Extrema of the magnitude of a derivative over solved trajectories (SURVEY.md section 8 (f) 1).
//
// Reference (relative to /root/reference/mav_trajectory_generation/, LIN.i =
// include/mav_trajectory_generation/impl/polynomial_optimization_linear_impl.h):
//   PolynomialOptimization::computeMaximumOfMagnitude            LIN.i:470-503   (mode 0)
//   PolynomialOptimization::computeSegmentMaximumMagnitudeCandidates  LIN.i:378-437
//   Trajectory::computeMinMaxMagnitude                            src/trajectory.cpp:181-217 (mode 1)
//   Segment::computeMinMaxMagnitudeCandidate[Time]s, selectMinMaxMagnitudeFromCandidates
//                                                                 src/segment.cpp:82-199
//   Polynomial::convolve src/polynomial.cpp:157-175, getCoefficients polynomial.h:100-117,
//   trailing-coefficient removal src/rpoly.cpp:44-75.
//
// Candidate times of a segment are the real roots inside [0, T] of
//   g(t) = sum_dim p_dim^(k)(t) p_dim^(k+1)(t)        (several dimensions; d/dt of |p^(k)|^2 / 2)
//   g(t) = p^(k+1)(t)                                   (one dimension)
// The reference hands g to a Jenkins-Traub root finder (TOMS 493, serial, global state) and keeps
// the real roots in range.  Here every thread owns one segment and isolates the real roots
// directly: the real roots of g^(m+1) split [0, T] into intervals on which g^(m) is monotone, so
// each sign change brackets exactly one root, refined by a safeguarded Newton iteration; the
// recursion starts at the linear derivative.  No complex arithmetic, no deflation.  The kernel is
// a template over the length of g and the recursion level, so g and the coefficients of the
// current level live in registers and every Horner step is two DFMA with no memory access; all
// threads of a warp are at the same level at the same time (FP64-pipe bound, divergence only in
// the number of brackets and Newton steps).  A second kernel folds the per-segment results in
// the reference's candidate order.
#include <cfloat>

#include "minsnap_device.cuh"
#include "minsnap_launch.h"

namespace minsnap {

namespace {

constexpr int kMaxG = 22;  // coefficients of g: 2N - 2k - 2 <= 22 for N <= 12

struct SegmentExtremum {
  double max_t, max_v, min_t, min_v;
};

// C(i, m): derivative level m of g divided by m! has coefficients C(j+m, m) g[j+m].  Every
// intermediate value is an integer below 2^53, so the result is exact.
__host__ __device__ constexpr double binomial(int i, int m) {
  double c = 1.0;
  for (int q = 1; q <= m; ++q) c = c * (double)(i - m + q) / (double)q;
  return c;
}

// Horner evaluations with compile-time degree: the coefficients stay in registers.
template <int DEG>
__device__ __forceinline__ double poly_value(const double (&d)[DEG + 1], double t) {
  double a = d[DEG];
#pragma unroll
  for (int j = DEG - 1; j >= 0; --j) a = fma(a, t, d[j]);
  return a;
}

// Value, slope and a running bound of the rounding error of the value (Horner with
// e <- e |t| + |a|; the computed value differs from the exact one by at most ~eps * e).
template <int DEG>
__device__ __forceinline__ void poly_value_slope_bound(const double (&d)[DEG + 1], double t, double& f, double& fp,
                                                       double& e) {
  const double at = fabs(t);
  double a = d[DEG], b = 0.0, err = fabs(a);
#pragma unroll
  for (int j = DEG - 1; j >= 0; --j) {
    b = fma(b, t, a);
    a = fma(a, t, d[j]);
    err = fma(err, at, fabs(a));
  }
  f = a;
  fp = b;
  e = err;
}

template <int DEG>
__device__ __forceinline__ void poly_value_slope(const double (&d)[DEG + 1], double t, double& f, double& fp) {
  double a = d[DEG], b = 0.0;
#pragma unroll
  for (int j = DEG - 1; j >= 0; --j) {
    b = fma(b, t, a);
    a = fma(a, t, d[j]);
  }
  f = a;
  fp = b;
}

// 1/x to ~40 bits (hardware seed + one Newton step): a Newton or secant step does not need a correctly
// rounded quotient -- an inexact step is corrected by the next one, and the bracket logic below catches
// anything wild (a flushed subnormal slope gives inf, which falls back to bisection).  The IEEE division
// it replaces is a ~20-instruction sequence per Newton iteration.
__device__ __forceinline__ double quick_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  return fma(r, fma(-x, r, 1.0), r);
}

// One root of a monotone piece: f(lo) and f(hi) have opposite signs.  Starts from the secant
// point of the bracket, then Newton, with bisection whenever the step leaves the bracket.  Stops
// when |f| is inside the rounding error of its own evaluation (bound taken at the starting point;
// nothing more can be learnt from the sign of f), when the step is below rel_tol, or when the
// bracket has collapsed.  Roots of the derivative levels only separate monotone pieces of the next
// level, so they are refined to 1e-10 only; the roots of g itself to full precision.
// (Measured alternative: collecting the brackets of a level first and refining the r-th bracket of
// every lane together was slower, 3.9 ms against 2.5 ms, although more lanes are active per step.)
template <int DEG>
__device__ __forceinline__ double refine_bracket(const double (&d)[DEG + 1], double lo, double hi, double f_lo,
                                                 double f_hi, double rel_tol) {
  const bool lo_negative = f_lo < 0.0;
  double x = lo - f_lo * ((hi - lo) * quick_rcp(f_hi - f_lo));
  if (!(x > lo && x < hi)) x = 0.5 * (lo + hi);
  double f_noise = 0.0;
  for (int it = 0; it < 64; ++it) {
    double f, fp;
    if (it == 0) {
      double e;
      poly_value_slope_bound<DEG>(d, x, f, fp, e);
      f_noise = DBL_EPSILON * e;
    } else {
      poly_value_slope<DEG>(d, x, f, fp);
    }
    if (fabs(f) <= f_noise) return x;
    if ((f < 0.0) == lo_negative) lo = x; else hi = x;
    double next = fp != 0.0 ? fma(-f, quick_rcp(fp), x) : lo - 1.0;
    if (!(next > lo && next < hi)) next = 0.5 * (lo + hi);
    if (next == lo || next == hi) return next;
    if (fabs(next - x) <= rel_tol * fabs(next)) return next;
    x = next;
  }
  return x;
}

// Level M of the recursion: the real roots of g^(M) inside [t0, t1] (written to `cur`, ascending;
// returns how many), given those of g^(M+1) in `prev`.  The level index is a template parameter
// so that every coefficient index is a compile-time constant and g stays in registers; all
// threads of a warp are at the same level at the same time.
template <int LEN, int M>
__device__ __noinline__ int root_level(const double (&g)[LEN], double t0, double t1, const double* prev, int n_prev,
                                       double* cur) {
  constexpr int DEG = LEN - 1 - M;
  double d[DEG + 1];
#pragma unroll
  for (int j = 0; j <= DEG; ++j) d[j] = binomial(j + M, M) * g[j + M];
  int n_cur = 0;
  double left = t0;
  double f_left = poly_value<DEG>(d, left);
  if (f_left == 0.0) cur[n_cur++] = left;
  for (int i = 0; i <= n_prev; ++i) {
    const double right = i < n_prev ? prev[i] : t1;
    if (!(right > left)) continue;
    const double f_right = poly_value<DEG>(d, right);
    if (f_right == 0.0) {
      cur[n_cur++] = right;
    } else if (f_left != 0.0 && (f_left < 0.0) != (f_right < 0.0)) {
      cur[n_cur++] = refine_bracket<DEG>(d, left, right, f_left, f_right, M == 0 ? 2.0 * DBL_EPSILON : 1e-10);
    }
    left = right;
    f_left = f_right;
  }
  return n_cur;
}

template <int LEN, int M>
__device__ __forceinline__ int dispatch_level(int m, const double (&g)[LEN], double t0, double t1, const double* prev,
                                              int n_prev, double* cur) {
  if (m == M) return root_level<LEN, M>(g, t0, t1, prev, n_prev, cur);
  if constexpr (M > 0) return dispatch_level<LEN, M - 1>(m, g, t0, t1, prev, n_prev, cur);
  return 0;
}

// Real roots of g inside [t0, t1]; coefficients above index `last` are zero (removed trailing
// coefficients): the levels whose polynomial would be constant are skipped.  Returns the buffer
// that holds the roots.
template <int LEN>
__device__ __forceinline__ const double* real_roots(const double (&g)[LEN], int last, double t0, double t1,
                                                    double* buf_a, double* buf_b, int& n_roots) {
  double* prev = buf_a;
  double* cur = buf_b;
  int n_prev = 0;
  // every thread walks all levels so that a warp stays at one level; a level above the thread's
  // own degree is skipped by predicate
  for (int m = LEN - 2; m >= 0; --m) {
    if (m > last - 1) continue;
    n_prev = dispatch_level<LEN, LEN - 2>(m, g, t0, t1, prev, n_prev, cur);
    double* swap = prev;
    prev = cur;
    cur = swap;
  }
  n_roots = n_prev;
  return prev;
}

struct ExtremaParams {
  long B;
  int K, D, N, derivative, mode;
  bool keep_small;
  uint32_t dim_mask;
  const double* coeffs;
  const double* times;
  SegmentExtremum* per_segment;  // [B][K]
  double* cand_times;            // optional [B][K][max_roots + 2]: start, end, roots
  double* cand_values;           // optional, same shape: the magnitude at each candidate
  int32_t* root_count;           // optional [B][K]
  int max_roots;
};

// ref polynomial.h:138-151 (Horner with the base coefficient folded in at every step)
__device__ inline double evaluate_derivative(const double* c, int N, int k, double t) {
  if (k >= N) return 0.0;
  double r = falling_factorial(k, N - 1) * c[N - 1];
  for (int j = N - 2; j >= k; --j) {
    r *= t;
    r += falling_factorial(k, j) * c[j];
  }
  return r;
}

__device__ inline double magnitude_at(const double* seg, int D, int N, uint32_t mask, int k, double t) {
  double s = 0.0;
  for (int dim = 0; dim < D; ++dim) {
    if (!((mask >> dim) & 1u)) continue;
    const double v = evaluate_derivative(seg + dim * N, N, k, t);
    s += v * v;
  }
  return sqrt(s);
}

// One thread per segment.  LEN (even) is the smallest instantiated size that holds the candidate
// polynomial; shorter polynomials are padded with zero coefficients, which the removal of
// trailing coefficients then treats like the reference's own zeros.
template <int LEN>
__global__ void __launch_bounds__(128) segment_extrema_kernel(ExtremaParams p) {
  const long tid_global = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (tid_global >= p.B * p.K) return;
  // segment-major thread order: a warp holds the same segment of 32 trajectories (the first and last
  // segments of a rest-to-rest trajectory have a different root structure from the inner ones, and
  // lanes with similar work diverge less)
  const long idx = (tid_global % p.B) * p.K + tid_global / p.B;
  const int N = p.N, D = p.D, k = p.derivative;
  const double* seg = p.coeffs + idx * D * N;
  const double T = p.times[idx];
  const int n_dims = __popc(p.dim_mask);

  double g[LEN];
#pragma unroll
  for (int i = 0; i < LEN; ++i) g[i] = 0.0;
  if (n_dims > 1) {
    // g = sum over dimensions of convolve(d, dd) (ref LIN.i:396-404 / src/segment.cpp:103-112);
    // convolve sums kernel[j] data[i-j] from the highest j down (src/polynomial.cpp:164-172).
    constexpr int ND = LEN / 2 + 1, NDD = LEN / 2;   // LEN = ND + NDD - 1
    for (int dim = 0; dim < D; ++dim) {
      if (!((p.dim_mask >> dim) & 1u)) continue;
      const double* c = seg + dim * N;
      double pd[ND], pdd[NDD];
#pragma unroll
      for (int j = 0; j < ND; ++j) pd[j] = j + k < N ? c[j + k] * falling_factorial(k, j + k) : 0.0;
#pragma unroll
      for (int j = 0; j < NDD; ++j) pdd[j] = j + k + 1 < N ? c[j + k + 1] * falling_factorial(k + 1, j + k + 1) : 0.0;
#pragma unroll
      for (int i = 0; i < LEN; ++i) {
        double acc = 0.0;
#pragma unroll
        for (int j = NDD - 1; j >= 0; --j)
          if (j <= i && i - j < ND) acc += pdd[j] * pd[i - j];
        g[i] += acc;
      }
    }
  } else {
    // one dimension: the roots of the next derivative (ref LIN.i:412-416, src/polynomial.cpp:57-78)
    int dim = 0;
    while (dim < D - 1 && !((p.dim_mask >> dim) & 1u)) ++dim;
    const double* c = seg + dim * N;
#pragma unroll
    for (int j = 0; j < LEN; ++j) g[j] = j + k + 1 < N ? c[j + k + 1] * falling_factorial(k + 1, j + k + 1) : 0.0;
  }
  // ref src/rpoly.cpp:44-55: drop trailing coefficients below machine epsilon.  The threshold is
  // absolute, so on long segments (T above ~12 s) the reference truncates coefficients that
  // matter near t = T; reproduced by default, keep_small removes exact zeros only.
  int last = -1;
#pragma unroll
  for (int i = 0; i < LEN; ++i) {
    const bool keep = p.keep_small ? g[i] != 0.0 : fabs(g[i]) >= DBL_EPSILON;
    if (keep) last = i;
  }
#pragma unroll
  for (int i = 0; i < LEN; ++i)
    if (i > last) g[i] = 0.0;

  double buf_a[LEN], buf_b[LEN];
  int n_roots = 0;
  const double* roots = buf_a;
  if (last >= 1 && T >= 0.0) roots = real_roots<LEN>(g, last, 0.0, T, buf_a, buf_b, n_roots);

  // Candidate list in the order of Segment::computeMinMaxMagnitudeCandidates (src/polynomial.cpp:39-40,
  // src/segment.cpp:133-156): start, end, then the roots.
  const bool list = p.cand_times != nullptr || p.cand_values != nullptr;
  const long stride = p.max_roots + 2;
  double* ct = p.cand_times ? p.cand_times + idx * stride : nullptr;
  double* cv = p.cand_values ? p.cand_values + idx * stride : nullptr;
  if (p.root_count) p.root_count[idx] = n_roots;

  SegmentExtremum e;
  const bool last_segment = (idx % p.K) == p.K - 1;
  const double v_start = magnitude_at(seg, D, N, p.dim_mask, k, 0.0);
  const bool need_end = p.mode != 0 || last_segment || list;
  const double v_end = need_end ? magnitude_at(seg, D, N, p.dim_mask, k, T) : 0.0;
  if (ct) { ct[0] = 0.0; ct[1] = T; }
  if (cv) { cv[0] = v_start; cv[1] = v_end; }
  e.max_t = e.min_t = 0.0;
  e.max_v = e.min_v = v_start;
  if (p.mode != 0) {
    // mode 1: start, end, roots (strict comparisons: the first extremal candidate wins)
    if (e.max_v < v_end) { e.max_v = v_end; e.max_t = T; }
    if (v_end < e.min_v) { e.min_v = v_end; e.min_t = T; }
  }
  for (int i = 0; i < n_roots; ++i) {
    const double t = roots[i];
    const double v = magnitude_at(seg, D, N, p.dim_mask, k, t);
    if (ct) ct[2 + i] = t;
    if (cv) cv[2 + i] = v;
    if (e.max_v < v) { e.max_v = v; e.max_t = t; }
    if (v < e.min_v) { e.min_v = v; e.min_t = t; }
  }
  if (p.mode == 0) {
    // mode 0: 0, roots, and the end of the last segment only (LIN.i:486-499); no minimum
    if (last_segment && e.max_v < v_end) { e.max_v = v_end; e.max_t = T; }
    e.min_t = 0.0;
    e.min_v = 0.0;
  }
  p.per_segment[idx] = e;
}

struct FoldParams {
  long B;
  int K, mode;
  const SegmentExtremum* per_segment;
  double *max_time, *max_value, *min_time, *min_value;
  int32_t *max_segment, *min_segment;
};

__global__ void __launch_bounds__(128) fold_extrema_kernel(FoldParams p) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  const SegmentExtremum* e = p.per_segment + b * p.K;
  // mode 0 starts from Extremum() = (0, 0, 0) (LIN.i:477); mode 1 from lowest()/max() (src/trajectory.cpp:186-187)
  double max_t = 0.0, max_v = p.mode == 0 ? 0.0 : -DBL_MAX, min_t = 0.0, min_v = DBL_MAX;
  int max_s = 0, min_s = 0;
  for (int s = 0; s < p.K; ++s) {
    const SegmentExtremum c = e[s];
    if (c.max_v > max_v) { max_v = c.max_v; max_t = c.max_t; max_s = s; }
    if (p.mode != 0 && c.min_v < min_v) { min_v = c.min_v; min_t = c.min_t; min_s = s; }
  }
  if (p.max_time) p.max_time[b] = max_t;
  if (p.max_value) p.max_value[b] = max_v;
  if (p.max_segment) p.max_segment[b] = max_s;
  if (p.mode != 0) {
    if (p.min_time) p.min_time[b] = min_t;
    if (p.min_value) p.min_value[b] = min_v;
    if (p.min_segment) p.min_segment[b] = min_s;
  }
}

struct SoftFoldParams {
  long B;
  int K, n_constraints;
  double limit[kMaxSoftConstraints];
  double weight, maximum_cost;
  const SegmentExtremum* per_segment;  // [n_constraints][B][K]
  double *soft, *terms, *max_value;
  double* objective;
  const double* cost;
  const int32_t* status;
  const double* times;
  double time_penalty;
};

// One thread per trajectory.  Each constraint's maximum is folded from its per-segment maxima with the comparisons
// and order of fold_extrema_kernel in mode 0, so it is the same bits as minsnap_extrema's max_value.  The term is
// std::min(maximum_cost, exp(...)) as the reference writes it (a NaN exponent gives maximum_cost), the soft cost
// their sum from 0 in constraint order (NL.i:2396-2426).  Optional epilogue: the objective of objectiveFunctionTime
// (NL.i:778-800), cost_trajectory + cost_time + cost_constraints in that order, each operation rounded on its own;
// a non-zero solve status makes it NaN.
__global__ void __launch_bounds__(128) soft_constraint_fold_kernel(SoftFoldParams p) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= p.B) return;
  double soft = 0.0;
  for (int c = 0; c < p.n_constraints; ++c) {
    const SegmentExtremum* e = p.per_segment + ((long)c * p.B + b) * p.K;
    double max_v = 0.0;
    for (int s = 0; s < p.K; ++s) {
      const double v = e[s].max_v;
      if (v > max_v) max_v = v;
    }
    const double x = exp(__dmul_rn(__ddiv_rn(__dsub_rn(max_v, p.limit[c]), p.limit[c]), p.weight));
    const double term = x < p.maximum_cost ? x : p.maximum_cost;
    soft = __dadd_rn(soft, term);
    if (p.terms) p.terms[b * p.n_constraints + c] = term;
    if (p.max_value) p.max_value[b * p.n_constraints + c] = max_v;
  }
  if (p.soft) p.soft[b] = soft;
  if (p.objective) {
    double total = 0.0;
    for (int k = 0; k < p.K; ++k) total += p.times[b * p.K + k];   // ref computeTotalTrajectoryTime: left to right
    double obj = __dadd_rn(__dadd_rn(p.cost[b], __dmul_rn(__dmul_rn(total, total), p.time_penalty)), soft);
    if (p.status && p.status[b] != 0) obj = __longlong_as_double(0x7ff8000000000000ll);
    p.objective[b] = obj;
  }
}

struct SoftGradientParams {
  long B;
  int K, D, n_constraints, n_fixed, n_free;
  int derivative[kMaxSoftConstraints];
  double limit[kMaxSoftConstraints];
  double weight, maximum_cost;
  const SegmentExtremum* per_segment;  // [n_constraints][B][K], as launch_soft_constraint_cost left it
  const double* coeffs;                // [B][K][D][N]
  const double* times;                 // [B][K]
  const int32_t* col_of_row;           // [N K]
  double* grad_free;                   // [B][n_free][D], or null when n_free == 0
  double* grad_times;                  // optional [B][K]
  bool add_times;                      // grad_times += times_weight g_T instead of grad_times = g_T
  double times_weight;
  double* max_time;                    // optional [B][n_constraints]
  int32_t* max_segment;                // optional [B][n_constraints]
};

// Gradient of the soft cost in the free derivatives and in the segment times with the end-point derivatives d held
// fixed.  One warp per trajectory.  Each constraint's argmax (segment s*, time t*) is folded from its per-segment
// maxima with the comparisons of fold_extrema_kernel, so ties go to the first strict maximum (a subgradient).  With
// x = exp((m - L) / L weight), dtau/dm = x weight / L below maximum_cost and 0 when saturated or at m = 0.  Every
// mode-0 candidate is a stationary point of m^2 in t or a segment start, so (envelope theorem) dm/dtheta is taken at
// fixed t*: sum_dim p_dim^(k)(t*) dp_dim^(k)(t*)/dtheta / m, plus the drift sum_dim p^(k) p^(k+1)(T) / m when t* is
// the end of the last segment and theta is its time.  With c = A^-1(T) d_seg, u = t*/T and k_r the derivative order
// of end-point row r:
//   dp^(k)(t*)/dd_r = T^(k_r - k)     sum_n b(k, n) u^(n-k) A1inv[n][r]
//   dp^(k)(t*)/dT   = sum_r d_r T^(k_r - k - 1) sum_n b(k, n) u^(n-k) (k_r - n) A1inv[n][r]
// Lanes run over (row, dimension) of s*; row r lands on its free column through col_of_row (fixed rows drop out).
// The constraints add in constraint order, each free entry on one lane and each time on one lane: no atomics.
template <int N>
__global__ void __launch_bounds__(128) soft_constraint_gradient_kernel(SoftGradientParams p) {
  constexpr int h = N / 2;
  const int lane = threadIdx.x & 31;
  const long warps = (long)gridDim.x * (blockDim.x / 32);
  const double* A1inv = UnitTables<N>::a1inv();
  const long nfd = (long)p.n_free * p.D;
  for (long b = (long)blockIdx.x * (blockDim.x / 32) + uniform_warp_index(); b < p.B; b += warps) {
    double* gf = p.grad_free ? p.grad_free + b * nfd : nullptr;
    if (gf)
      for (long j = lane; j < nfd; j += 32) gf[j] = 0.0;
    // lane c keeps constraint c's segment s* and its time derivative
    int my_seg = -1;
    double my_gt = 0.0;
    for (int c = 0; c < p.n_constraints; ++c) {
      __syncwarp();   // this constraint's additions to the free columns see the zeroing and the previous constraints'
      const SegmentExtremum* e = p.per_segment + ((long)c * p.B + b) * p.K;
      double max_v = 0.0, max_t = 0.0;
      int max_s = 0;
      for (int s = 0; s < p.K; ++s) {
        const SegmentExtremum x = e[s];
        if (x.max_v > max_v) { max_v = x.max_v; max_t = x.max_t; max_s = s; }
      }
      if (lane == 0) {
        if (p.max_time) p.max_time[b * p.n_constraints + c] = max_t;
        if (p.max_segment) p.max_segment[b * p.n_constraints + c] = max_s;
      }
      const int k = p.derivative[c];
      const double L = p.limit[c];
      const double x = exp(__dmul_rn(__ddiv_rn(__dsub_rn(max_v, L), L), p.weight));
      const double dtau_over_m = (x < p.maximum_cost && max_v > 0.0) ? x * p.weight / L / max_v : 0.0;
      if (lane == c) my_seg = max_s;
      if (dtau_over_m == 0.0) continue;
      const long si = b * p.K + max_s;
      const double T = p.times[si];
      const double* seg = p.coeffs + si * p.D * N;
      const double u = max_t / T;
      const bool drift = max_s == p.K - 1 && max_t == T;
      double acc_t = 0.0;
      for (int q = lane; q < N * p.D; q += 32) {
        const int r = q / p.D, dim = q - r * p.D;
        const int kr = r % h;
        const double* cd = seg + dim * N;
        const double w = dtau_over_m * evaluate_derivative(cd, N, k, max_t);   // dtau/dm p_dim^(k)(t*) / m
        double bd = 0.0, bt = 0.0, up = 1.0;
        for (int n = k; n < N; ++n) {
          const double f = falling_factorial(k, n) * up * A1inv[n * N + r];
          bd += f;
          bt += (double)(kr - n) * f;
          up *= u;
        }
        const double Tp = int_power(T, kr - k);
        if (gf) {
          const int col = p.col_of_row[max_s * N + r] - p.n_fixed;
          if (col >= 0) gf[col * p.D + dim] += w * (bd * Tp);
        }
        if (p.grad_times) {
          acc_t += w * evaluate_derivative(cd, N, kr, r < h ? 0.0 : T) * (bt * Tp / T);
          if (drift && r == 0) acc_t += w * evaluate_derivative(cd, N, k + 1, T);
        }
      }
      if (p.grad_times) {
        acc_t = warp_sum(acc_t);
        if (lane == c) my_gt = acc_t;
      }
    }
    if (p.grad_times) {
      for (int s0 = 0; s0 < p.K; s0 += 32) {
        const int s = s0 + lane;
        double g = 0.0;
        for (int c = 0; c < p.n_constraints; ++c) {
          const int sc = __shfl_sync(0xffffffffu, my_seg, c);
          const double gc = __shfl_sync(0xffffffffu, my_gt, c);
          if (sc == s) g += gc;
        }
        if (s >= p.K) continue;
        double* dst = p.grad_times + b * p.K + s;
        *dst = p.add_times ? __dadd_rn(*dst, __dmul_rn(p.times_weight, g)) : g;
      }
    }
  }
}

template <int LEN>
cudaError_t launch_segments(const ExtremaParams& p, cudaStream_t stream) {
  const long n = p.B * p.K;
  segment_extrema_kernel<LEN><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(p);
  return cudaGetLastError();
}

}  // namespace

int extrema_max_roots(int N, int derivative, int n_dims) {
  const int n_d = N - derivative, n_dd = n_d - 1;
  const int len = n_dims > 1 ? n_d + n_dd - 1 : n_dd;
  return len > 1 ? len - 1 : 0;
}

cudaError_t launch_extrema(const ExtremaArgs& a, cudaStream_t stream) {
  if (a.B == 0) return cudaSuccess;
  const int len = extrema_max_roots(a.N, a.derivative, __builtin_popcount(a.dim_mask)) + 1;
  if (len > kMaxG) return cudaErrorInvalidValue;
  cudaError_t e;
  void* scratch = nullptr;
  if ((e = cudaMallocAsync(&scratch, sizeof(SegmentExtremum) * (size_t)a.B * a.K, stream)) != cudaSuccess) return e;
  ExtremaParams p;
  p.B = a.B; p.K = a.K; p.D = a.D; p.N = a.N; p.derivative = a.derivative; p.mode = a.mode;
  p.keep_small = a.keep_small;
  p.dim_mask = a.dim_mask;
  p.coeffs = a.d_coeffs; p.times = a.d_times;
  p.per_segment = static_cast<SegmentExtremum*>(scratch);
  p.cand_times = a.d_cand_times; p.cand_values = a.d_cand_values; p.root_count = a.d_root_count;
  p.max_roots = a.max_roots;
  e = len <= 4    ? launch_segments<4>(p, stream)
      : len <= 6  ? launch_segments<6>(p, stream)
      : len <= 8  ? launch_segments<8>(p, stream)
      : len <= 10 ? launch_segments<10>(p, stream)
      : len <= 12 ? launch_segments<12>(p, stream)
      : len <= 14 ? launch_segments<14>(p, stream)
      : len <= 16 ? launch_segments<16>(p, stream)
      : len <= 18 ? launch_segments<18>(p, stream)
      : len <= 20 ? launch_segments<20>(p, stream)
                  : launch_segments<22>(p, stream);
  if (e == cudaSuccess) {
    FoldParams f;
    f.B = a.B; f.K = a.K; f.mode = a.mode; f.per_segment = p.per_segment;
    f.max_time = a.d_max_time; f.max_value = a.d_max_value; f.max_segment = a.d_max_segment;
    f.min_time = a.d_min_time; f.min_value = a.d_min_value; f.min_segment = a.d_min_segment;
    fold_extrema_kernel<<<(unsigned)((a.B + 127) / 128), 128, 0, stream>>>(f);
    e = cudaGetLastError();
  }
  cudaFreeAsync(scratch, stream);
  return e;
}

size_t soft_constraint_scratch_bytes(long B, int K, int n_constraints) {
  return sizeof(SegmentExtremum) * (size_t)n_constraints * B * K;
}

// One segment_extrema_kernel launch per constraint (mode 0, all dimensions) into its slab of the caller's scratch,
// then one fold over all constraints.
cudaError_t launch_soft_constraint_cost(const SoftConstraintArgs& a, cudaStream_t stream) {
  if (a.B == 0) return cudaSuccess;
  SegmentExtremum* per_segment = static_cast<SegmentExtremum*>(a.d_scratch);
  const uint32_t all = a.D == 32 ? 0xffffffffu : ((1u << a.D) - 1u);
  for (int c = 0; c < a.n_constraints; ++c) {
    const int len = extrema_max_roots(a.N, a.derivative[c], a.D) + 1;
    if (len > kMaxG) return cudaErrorInvalidValue;
    ExtremaParams p;
    p.B = a.B; p.K = a.K; p.D = a.D; p.N = a.N; p.derivative = a.derivative[c]; p.mode = 0;
    p.keep_small = a.keep_small;
    p.dim_mask = all;
    p.coeffs = a.d_coeffs; p.times = a.d_times;
    p.per_segment = per_segment + (size_t)c * a.B * a.K;
    p.cand_times = nullptr; p.cand_values = nullptr; p.root_count = nullptr;
    p.max_roots = len - 1;
    const cudaError_t e = len <= 4    ? launch_segments<4>(p, stream)
                          : len <= 6  ? launch_segments<6>(p, stream)
                          : len <= 8  ? launch_segments<8>(p, stream)
                          : len <= 10 ? launch_segments<10>(p, stream)
                          : len <= 12 ? launch_segments<12>(p, stream)
                          : len <= 14 ? launch_segments<14>(p, stream)
                          : len <= 16 ? launch_segments<16>(p, stream)
                          : len <= 18 ? launch_segments<18>(p, stream)
                          : len <= 20 ? launch_segments<20>(p, stream)
                                      : launch_segments<22>(p, stream);
    if (e != cudaSuccess) return e;
  }
  SoftFoldParams f;
  f.B = a.B; f.K = a.K; f.n_constraints = a.n_constraints;
  for (int c = 0; c < kMaxSoftConstraints; ++c) f.limit[c] = c < a.n_constraints ? a.limit[c] : 0.0;
  f.weight = a.weight; f.maximum_cost = a.maximum_cost;
  f.per_segment = per_segment;
  f.soft = a.d_soft; f.terms = a.d_terms; f.max_value = a.d_max_value;
  f.objective = a.d_objective; f.cost = a.d_cost; f.status = a.d_status; f.times = a.d_times;
  f.time_penalty = a.time_penalty;
  soft_constraint_fold_kernel<<<(unsigned)((a.B + 127) / 128), 128, 0, stream>>>(f);
  return cudaGetLastError();
}

cudaError_t launch_soft_constraint_gradient(const SoftGradientArgs& a, cudaStream_t stream) {
  const SoftConstraintArgs& s = a.soft;
  if (s.B == 0) return cudaSuccess;
  SoftGradientParams p;
  p.B = s.B; p.K = s.K; p.D = s.D; p.n_constraints = s.n_constraints; p.n_fixed = a.n_fixed; p.n_free = a.n_free;
  for (int c = 0; c < kMaxSoftConstraints; ++c) {
    p.derivative[c] = c < s.n_constraints ? s.derivative[c] : 0;
    p.limit[c] = c < s.n_constraints ? s.limit[c] : 0.0;
  }
  p.weight = s.weight; p.maximum_cost = s.maximum_cost;
  p.per_segment = static_cast<const SegmentExtremum*>(s.d_scratch);
  p.coeffs = s.d_coeffs; p.times = s.d_times; p.col_of_row = a.d_col_of_row;
  p.grad_free = a.n_free > 0 ? a.d_grad_free : nullptr;
  p.grad_times = a.d_grad_times; p.add_times = a.add_times; p.times_weight = a.times_weight;
  p.max_time = a.d_max_time; p.max_segment = a.d_max_segment;
  long grid = (s.B + 3) / 4;
  if (grid > sm_count() * 32) grid = sm_count() * 32;
  switch (s.N) {
    case 4: soft_constraint_gradient_kernel<4><<<(unsigned)grid, 128, 0, stream>>>(p); break;
    case 6: soft_constraint_gradient_kernel<6><<<(unsigned)grid, 128, 0, stream>>>(p); break;
    case 8: soft_constraint_gradient_kernel<8><<<(unsigned)grid, 128, 0, stream>>>(p); break;
    case 10: soft_constraint_gradient_kernel<10><<<(unsigned)grid, 128, 0, stream>>>(p); break;
    case 12: soft_constraint_gradient_kernel<12><<<(unsigned)grid, 128, 0, stream>>>(p); break;
    default: return cudaErrorInvalidValue;
  }
  return cudaGetLastError();
}

}  // namespace minsnap
