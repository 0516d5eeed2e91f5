/*
 * minsnap_b200.h -- C ABI of the B200-native batched minimum-snap solver.
 *
 * This is the drop-in boundary for the reference's hot path
 *   Vertex -> estimateSegmentTimes -> PolynomialOptimization<N>::setupFromVertices ->
 *   solveLinear -> getSegments/getTrajectory -> Segment/Polynomial/Trajectory::evaluate
 * (magrimm/mav_trajectory_generation_cmake).  The reference has no FFI layer of its own: its
 * boundary is a header-only C++ class API.  The C++ mirror of that API lives in
 * include/mav_trajectory_generation/ and calls ONLY the functions below; any other host
 * language binds the same functions (see INTEGRATION.md).
 *
 * Citations "ref:" are relative to /root/reference/mav_trajectory_generation/ with
 *   LIN.h = include/mav_trajectory_generation/polynomial_optimization_linear.h
 *   LIN.i = include/mav_trajectory_generation/impl/polynomial_optimization_linear_impl.h
 *
 * Conventions
 *   - plain pointers and sizes only; every function returns an int status (MINSNAP_OK == 0),
 *     never throws, keeps no mutable global state and is re-entrant;
 *   - "d_" pointers are DEVICE pointers on the current CUDA device, "h_" pointers are host
 *     pointers; `stream` is a cudaStream_t passed as void* (NULL = default stream);
 *   - device entry points are asynchronous on `stream`; *_host entry points are synchronous
 *     and include the host<->device copies;
 *   - all arithmetic is IEEE double; there is NO CPU fallback: without a usable sm_100 GPU
 *     every compute entry point returns MINSNAP_ERR_NO_DEVICE / MINSNAP_ERR_CUDA.
 *
 * Array layouts (row-major, last index fastest), with h = N/2:
 *   fixed_mask    [(K+1)][h]          uint8, non-zero = the vertex constrains that derivative
 *                                     (ref: a Vertex's constraint map, include/.../vertex.h:42-107)
 *   fixed_values  [B][n_fixed][D]     constraint values in the reference's column order: sorted
 *                                     by (vertex, derivative) (ref: fixed_constraints_compact_,
 *                                     LIN.i:228-246; transposed so that D is fastest)
 *   free_values   [B][n_free][D]      optimised free derivatives d_p, same ordering rule
 *                                     (ref: free_constraints_compact_, LIN.i:360-365)
 *   positions     [B][K+1][D]         vertex positions (standard-mask fast path)
 *   times         [B][K]              segment durations
 *   coeffs        [B][K][D][N]        polynomial coefficients, increasing powers
 *                                     (ref: Segment/Polynomial, include/.../polynomial.h:34-38)
 *   col_of_row    [N*K]  int32        column of the single 1 in each row of the reordering
 *                                     matrix C (ref: constraint_reordering_, LIN.i:171-250)
 *   samples       [B][M][n_deriv][D]  derivatives 0..n_deriv-1 at M instants
 */
#ifndef MINSNAP_B200_H_
#define MINSNAP_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define MINSNAP_API __attribute__((visibility("default")))
#else
#define MINSNAP_API
#endif

/* ---- return codes ------------------------------------------------------------------ */
enum {
  MINSNAP_OK = 0,
  MINSNAP_ERR_ARG = 1,         /* NULL / out-of-range argument (the reference CHECK-aborts) */
  MINSNAP_ERR_CUDA = 2,        /* a CUDA runtime call failed; see minsnap_last_cuda_error() */
  MINSNAP_ERR_UNSUPPORTED = 3, /* shape not built (N not in {4,6,8,10,12}, K too large ...)  */
  MINSNAP_ERR_NO_DEVICE = 4,   /* no CUDA device / not sm_100                                */
  MINSNAP_ERR_WORKSPACE = 5    /* workspace pointer NULL or too small                        */
};

/* ---- per-problem status bits written to d_status[b] ---------------------------------- */
enum {
  MINSNAP_STATUS_OK = 0,
  MINSNAP_STATUS_NONPOSITIVE_PIVOT = 1, /* R_pp not positive definite (ref never checks, LIN.i:355-357) */
  MINSNAP_STATUS_BAD_TIME = 2,          /* a segment time <= 0 or NaN (ref: CHECK_GT, LIN.i:287) */
  MINSNAP_STATUS_NONFINITE = 4          /* a non-finite coefficient was produced */
};

typedef void* minsnap_stream_t; /* cudaStream_t */

/* ---- runtime ---------------------------------------------------------------------- */
MINSNAP_API int minsnap_abi_version(void);
MINSNAP_API const char* minsnap_error_string(int code);
/* Text of the last CUDA error seen by the calling thread ("" when none). */
MINSNAP_API const char* minsnap_last_cuda_error(void);
/* Fills the properties of the current device; MINSNAP_ERR_NO_DEVICE when there is none. */
MINSNAP_API int minsnap_device_info(int* device, int* sm_count, int* cc_major, int* cc_minor,
                                    size_t* global_mem_bytes);

/* ---- a10: constraint reordering (ref: setupConstraintReorderingMatrix, LIN.i:171-250) ---
 * One index map per mask.  d_mask[n_masks][(K+1)*h] -> d_col_of_row[n_masks][N*K],
 * d_counts[n_masks][2] = {n_fixed, n_free}.  Integer work: bit-exact with the reference. */
MINSNAP_API int minsnap_reorder(int N, int K, long n_masks, const uint8_t* d_mask,
                                int32_t* d_col_of_row, int32_t* d_counts, minsnap_stream_t stream);

/* ---- a2: segment-time heuristic (ref: estimateSegmentTimes, src/vertex.cpp:162-178) ----- */
MINSNAP_API int minsnap_estimate_segment_times(long B, int K, int D, const double* d_positions,
                                               double v_max, double a_max, double magic,
                                               double* d_times, minsnap_stream_t stream);

/* ---- a5-a9, a11: per-segment matrices for the accessor / test path ---------------------
 * For each of n segment times: A (ref: setupMappingMatrix, LIN.i:101-111), A^-1 (ref:
 * invertMappingMatrix, LIN.i:132-169), Q (ref: computeQuadraticCostJacobian, LIN.i:573-589)
 * and H = A^-T Q A^-1 (ref: constructR, LIN.i:305-308); each [n][N][N], any may be NULL. */
MINSNAP_API int minsnap_segment_matrices(long n, int N, int derivative, const double* d_T,
                                         double* d_A, double* d_Ainv, double* d_Q, double* d_H,
                                         minsnap_stream_t stream);

/* ---- a10-a13 (+a16): general batched setup + solveLinear -------------------------------
 * (ref: setupFromVertices LIN.i:46-99, updateSegmentTimes :275-295, constructR :297-326,
 *  solveLinear :328-369, updateSegmentsFromCompactConstraints :252-273, computeCost :113-130)
 * One constraint structure (h_fixed_mask, HOST pointer) shared by the whole batch -- the
 * reference requires the same of all dimensions (LIN.h:104-107).  Any mask, any K that fits
 * shared memory, any D.  Optional outputs may be NULL.
 * d_workspace: minsnap_solve_workspace_bytes(N, K) bytes of device memory. */
MINSNAP_API size_t minsnap_solve_workspace_bytes(int N, int K);
MINSNAP_API int minsnap_solve(long B, int K, int D, int N, int derivative,
                              const uint8_t* h_fixed_mask, const double* d_fixed_values,
                              const double* d_times, double* d_coeffs, double* d_free_values,
                              double* d_cost, int32_t* d_status, int32_t* d_col_of_row,
                              void* d_workspace, size_t workspace_bytes, minsnap_stream_t stream);

/* ---- a13 alone (ref: setFreeConstraints -> updateSegmentsFromCompactConstraints,
 *      LIN.i:505-514, 252-273): coefficients from given [d_f; d_p] ----------------------- */
MINSNAP_API int minsnap_coeffs_from_constraints(long B, int K, int D, int N,
                                                const uint8_t* h_fixed_mask,
                                                const double* d_fixed_values,
                                                const double* d_free_values, const double* d_times,
                                                double* d_coeffs, void* d_workspace,
                                                size_t workspace_bytes, minsnap_stream_t stream);

/* ---- a16 alone (ref: computeCost, LIN.i:113-130): 0.5 * sum c^T Q c -------------------- */
MINSNAP_API int minsnap_cost(long B, int K, int D, int N, int derivative, const double* d_coeffs,
                             const double* d_times, double* d_cost, minsnap_stream_t stream);

/* ---- fast path: the createRandomVertices mask (ref: src/vertex.cpp:59,71-76) -------------
 * End vertices fix derivatives 0..h-1, interior vertices fix position only; N = 10, snap.
 * d_end_derivatives [B][2][h-1][D] (start then end vertex, derivatives 1..h-1) or NULL = zeros.
 * d_times NULL => times are computed on the device from (v_max, a_max, magic) exactly as
 * minsnap_estimate_segment_times does and, when d_times_out != NULL, written there.
 * A shape no kernel takes (MINSNAP_ERR_UNSUPPORTED) writes no output, d_times_out included.
 * The environment variable MINSNAP_STANDARD_ROUTE=tm|pair|pair_long|bcr|chunked|general (read on every call) runs
 * the named kernel instead of the one the shape and batch size select, for tests that compare two kernels:
 * MINSNAP_ERR_UNSUPPORTED when that kernel cannot take the call, MINSNAP_ERR_ARG for any other name. */
MINSNAP_API int minsnap_solve_standard(long B, int K, int D, int N, int derivative,
                                       const double* d_positions, const double* d_end_derivatives,
                                       const double* d_times, double v_max, double a_max,
                                       double magic, double* d_times_out, double* d_coeffs,
                                       double* d_free_values, double* d_cost, int32_t* d_status,
                                       minsnap_stream_t stream);

/* ---- a17-a19: sampling (ref: Polynomial::evaluate polynomial.h:138-151, Segment::evaluate
 *      src/segment.cpp:51-58, Trajectory::evaluate src/trajectory.cpp:41-66) ---------------
 * Segment choice: first i with (T_0 + ... + T_i) > t, the sum accumulated left to right; an
 * instant at or past the end of the trajectory yields zeros (the reference is undefined at
 * exactly t == max time) and segment index -1.
 * minsnap_sample_uniform: t_m = m * (T_total / M), m = 0..M-1, on [0, T_total).
 * minsnap_sample_at:      explicit instants d_t[B][M] (t_stride = M) or one shared row
 *                         d_t[M] (t_stride = 0).
 * d_out [B][M][n_deriv][D]; optional d_t_out [B][M], d_segment [B][M]. */
MINSNAP_API int minsnap_sample_uniform(long B, int K, int D, int N, const double* d_coeffs,
                                       const double* d_times, int M, int n_deriv, double* d_out,
                                       double* d_t_out, minsnap_stream_t stream);
MINSNAP_API int minsnap_sample_at(long B, int K, int D, int N, const double* d_coeffs,
                                  const double* d_times, int M, const double* d_t, long t_stride,
                                  int n_deriv, double* d_out, int32_t* d_segment,
                                  minsnap_stream_t stream);

/* ---- a20: Trajectory::evaluateRange (ref: src/trajectory.cpp:68-128) ----------------------
 * Sequential-accumulation sampler: time_in_segment += dt, one derivative per call.
 * d_out [B][max_samples][D], d_t_out [B][max_samples] (optional), d_count [B] = number of
 * samples the reference would emit (clamped writes beyond max_samples are dropped). */
MINSNAP_API int minsnap_evaluate_range(long B, int K, int D, int N, const double* d_coeffs,
                                       const double* d_times, double t_start, double t_end,
                                       double dt, int derivative, int max_samples, double* d_out,
                                       double* d_t_out, int32_t* d_count, minsnap_stream_t stream);

/* ---- config 5: segment-time sweep, cost only (ref: objectiveFunctionTime's
 *      updateSegmentTimes + solveLinear + computeCost, NL.i:778-781) -----------------------
 * Standard mask; d_times [B][S][K] -> d_cost [B][S]; optional d_status [B][S]. */
MINSNAP_API int minsnap_cost_sweep(long B, int S, int K, int D, int N, int derivative,
                                   const double* d_positions, const double* d_end_derivatives,
                                   const double* d_times, double* d_cost, int32_t* d_status,
                                   minsnap_stream_t stream);

/* ---- SURVEY 8(f)1: extrema of the magnitude of a derivative --------------------------------
 * ref: PolynomialOptimization::computeMaximumOfMagnitude<Derivative> (LIN.i:470-503) with
 *      computeSegmentMaximumMagnitudeCandidates (LIN.i:378-437)              -> mode 0
 *      Trajectory::computeMinMaxMagnitude (src/trajectory.cpp:181-217) with
 *      Segment::computeMinMaxMagnitudeCandidates / selectMinMaxMagnitudeFromCandidates
 *      (src/segment.cpp:82-199)                                              -> mode 1
 *      root finder findRootsJenkinsTraub (src/rpoly.cpp), replaced by real-root isolation.
 * Candidate times of a segment: the real roots inside [0, T] of sum_dim p^(k) p^(k+1) (several
 * dimensions) or of p^(k+1) (one dimension), trailing coefficients below machine epsilon removed
 * as the reference does (src/rpoly.cpp:44-75).
 *   mode 0 (MINSNAP_EXTREMA_OPTIMIZATION): per segment t = 0 and the roots, plus the end of the
 *          last segment; maximum only, starting from (time 0, value 0, segment 0); d_min_* unused.
 *   mode 1 (MINSNAP_EXTREMA_TRAJECTORY): per segment start, end and the roots; minimum and maximum.
 * A later candidate replaces the incumbent only when strictly larger (smaller).
 * MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS may be OR-ed into mode: the reference's coefficient
 * threshold is absolute (2.2e-16), which on segments longer than about 12 s removes terms of the
 * candidate polynomial that matter near the end of the segment, so the reference (and this
 * function by default, for parity) can miss extrema there; with the flag only exact zeros are
 * removed and the result agrees with dense sampling.
 * dim_mask: bit d set => dimension d takes part; 0 => all D dimensions (D <= 32).
 * Times are relative to the start of the reported segment, as in the reference's Extremum.
 * Outputs [B] each, any may be NULL.  Optional per-segment candidate lists in the order of
 * Segment::computeMinMaxMagnitudeCandidates (start, end, then the roots, ascending):
 * d_cand_times / d_cand_values [B][K][max_roots + 2] (max_roots from minsnap_extrema_max_roots;
 * entries past 2 + count are not written) and d_root_count [B][K] = number of roots. */
#define MINSNAP_EXTREMA_OPTIMIZATION 0
#define MINSNAP_EXTREMA_TRAJECTORY 1
#define MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS 16
MINSNAP_API int minsnap_extrema_max_roots(int N, int derivative, int n_dims);
MINSNAP_API int minsnap_extrema(long B, int K, int D, int N, const double* d_coeffs,
                                const double* d_times, int derivative, int mode, uint32_t dim_mask,
                                double* d_max_time, double* d_max_value, int32_t* d_max_segment,
                                double* d_min_time, double* d_min_value, int32_t* d_min_segment,
                                double* d_cand_times, double* d_cand_values, int32_t* d_root_count,
                                minsnap_stream_t stream);

/* ---- SURVEY 8(f)2: the time-only objective and its numeric gradient ------------------------
 * minsnap_time_objective (ref objectiveFunctionTime, NL.i:765-832, without the collision and
 * soft-constraint terms; minsnap_time_objective_soft below adds the soft terms): for every trajectory b and
 * candidate time allocation s
 *   objective[b][s] = computeCost(solveLinear(times[b][s])) + time_penalty * (sum_k times[b][s][k])^2.
 * Standard mask (as minsnap_cost_sweep, which it runs); d_cost [B][S] optional.
 * minsnap_time_gradient (ref getCostAndGradientTime, NL.i:2155-2243): central differences of
 * J_d = d^T R d (= 2 computeCost; ref getCostAndGradientDerivative, NL.i:1452-1521) in each
 * segment time, the end-point derivatives d of the solved trajectory held fixed as in the
 * reference; a time <= 0.1 is moved to 0.1 instead of -/+ increment:
 *   gradient[b][n] = w_d (J_d(T_n+) - J_d(T_n-)) / (2 increment) + w_t.
 * Input: the solved coefficients.  d_segment_cost [B][K] optional: the per-segment terms of J_d
 * at the given times (their sum over n is J_d). */
MINSNAP_API int minsnap_time_objective(long B, int S, int K, int D, int N, int derivative,
                                       const double* d_positions, const double* d_end_derivatives,
                                       const double* d_times, double time_penalty,
                                       double* d_objective, double* d_cost, int32_t* d_status,
                                       minsnap_stream_t stream);
MINSNAP_API int minsnap_time_gradient(long B, int K, int D, int N, int derivative,
                                      const double* d_coeffs, const double* d_times,
                                      double increment, double w_d, double w_t, double* d_gradient,
                                      double* d_segment_cost, minsnap_stream_t stream);

/* minsnap_optimize_segment_times: an additive batched driver for the time-only problem (the reference runs one
 * NLopt instance per trajectory on the host, NL.i:230-330; NLopt is an absent third-party dependency, so no
 * parity is claimed for the optimiser -- only for the objective and gradient it is built from).  Every
 * trajectory descends  computeCost + time_penalty * total_time^2  along its own numeric gradient; per iteration
 * n_steps step lengths (max_relative_step / 2^s of the step that would zero a segment time, times clamped at
 * min_time) are evaluated by one cost sweep and the first minimum is accepted when it improves the incumbent.
 * Five launches per iteration, all on `stream`, no host round trip.  d_times [B][K] is updated in place;
 * d_history (optional) [iterations + 1][B] receives the incumbent objective after every iteration. */
MINSNAP_API int minsnap_optimize_segment_times(long B, int K, int D, int N, int derivative,
                                               const double* d_positions,
                                               const double* d_end_derivatives, double* d_times,
                                               int iterations, double time_penalty, int n_steps,
                                               double max_relative_step, double min_time,
                                               double gradient_increment, double* d_history,
                                               minsnap_stream_t stream);

/* ---- the time-only objective with the reference's soft limits on max |p^(k)| ------------------
 * ref: objectiveFunctionTime with use_soft_constraints (NL.i:765-832), evaluateMaximumMagnitudeAsSoftConstraint
 *      (NL.i:2396-2426) over evaluateMaximumMagnitudeConstraint (NL.i:2346-2392), i.e. computeMaximumOfMagnitude.
 * Constraint c (1 <= n_constraints <= 4) limits derivative h_derivatives[c] (0 .. N-2) over all dimensions to
 * h_limits[c] > 0; its term is
 *   term_c = min(maximum_cost, exp((max_c - limit_c) / limit_c * weight))     (std::min: a NaN exponent gives
 *            maximum_cost, as in the reference),
 * max_c bit-identical to minsnap_extrema(..., MINSNAP_EXTREMA_OPTIMIZATION | extrema_flags)'s max_value.  The soft
 * cost is the sum of the terms from 0 in constraint order.  weight and maximum_cost are positive and finite;
 * extrema_flags is 0 (the reference's coefficient truncation) or MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS.  The host
 * arrays reach the device in kernel parameters, not by a copy, so every call can be captured into a CUDA graph once
 * it has run eagerly on the thread.  Temporary device memory is allocated stream-ordered (cudaMallocAsync).
 *
 * minsnap_soft_constraint_cost: solved trajectories d_coeffs [B][K][D][N], d_times [B][K] (D <= 32) -> d_cost [B];
 * optional d_terms [B][n_constraints] (term_c) and d_max_value [B][n_constraints] (max_c). */
MINSNAP_API int minsnap_soft_constraint_cost(long B, int K, int D, int N, const double* d_coeffs,
                                             const double* d_times, int n_constraints,
                                             const int32_t* h_derivatives, const double* h_limits,
                                             double weight, double maximum_cost, int extrema_flags,
                                             double* d_cost, double* d_terms, double* d_max_value,
                                             minsnap_stream_t stream);

/* minsnap_time_objective_soft: for every trajectory b and candidate allocation s (standard mask, the shapes
 * minsnap_solve_standard takes; MINSNAP_ERR_UNSUPPORTED otherwise, before any device work)
 *   objective[b][s] = computeCost + time_penalty * (sum_k times[b][s][k])^2 + soft cost,
 * the time sum left to right and the three parts added in that order (cost_trajectory + cost_time +
 * cost_constraints).  A solve with a non-zero status (e.g. a time <= 0) gives a NaN objective.  d_positions
 * [B][K+1][D], d_end_derivatives as in minsnap_solve_standard or NULL, d_times [B][S][K] -> d_objective [B][S];
 * optional d_cost [B][S] (computeCost), d_soft [B][S] (soft cost), d_terms [B][S][n_constraints]. */
MINSNAP_API int minsnap_time_objective_soft(long B, int S, int K, int D, int N, int derivative,
                                            const double* d_positions, const double* d_end_derivatives,
                                            const double* d_times, double time_penalty, int n_constraints,
                                            const int32_t* h_derivatives, const double* h_limits,
                                            double weight, double maximum_cost, int extrema_flags,
                                            double* d_objective, double* d_cost, double* d_soft,
                                            double* d_terms, minsnap_stream_t stream);

/* minsnap_optimize_segment_times_soft: minsnap_optimize_segment_times on the objective above (no parity is claimed
 * for the optimiser, NLopt being absent; only for the objective and its pieces).  Per iteration, at the incumbent:
 * solve, minsnap_time_gradient (w_d = 0.5, w_t = 0); the 2K allocations T -/+ gradient_increment e_n of every
 * trajectory (a time <= 0.1 moved to 0.1 on both sides) are re-solved and their soft cost's central difference is
 * added to the gradient; the step ladder of minsnap_optimize_segment_times (which adds the penalty's gradient);
 * minsnap_time_objective_soft over the n_steps candidates; the first minimum among the finite objectives is accepted
 * when strictly below the incumbent.  All launches are on `stream` and nothing returns to the host.  The workspace is
 * one cudaMallocAsync of, with R = max(2K, n_steps), h = N/2 and n_c = n_constraints,
 *   8 B (R ((K+1) D + 2 (h-1) D [only with end derivatives] + K D N + K + 3) + K + 1) + 4 B R + 32 B R K n_c bytes
 * (plus alignment): 4.47 GB at B = 65,536, K = 10, n_steps = 16, D = 3, N = 10, n_c = 2 (computed from the shapes).
 * d_times [B][K] in/out; d_history (optional) [iterations + 1][B]: the incumbent objective, first at the initial
 * times; d_max_value (optional) [B][n_constraints]: the maxima at the returned times. */
MINSNAP_API int minsnap_optimize_segment_times_soft(long B, int K, int D, int N, int derivative,
                                                    const double* d_positions,
                                                    const double* d_end_derivatives, double* d_times,
                                                    int iterations, double time_penalty, int n_steps,
                                                    double max_relative_step, double min_time,
                                                    double gradient_increment, int n_constraints,
                                                    const int32_t* h_derivatives, const double* h_limits,
                                                    double weight, double maximum_cost, int extrema_flags,
                                                    double* d_history, double* d_max_value,
                                                    minsnap_stream_t stream);

/* ---- SURVEY 8(f)3: collision cost of solved trajectories against a signed-distance grid ------
 * ref: PolynomialOptimizationNonLinear::getCostAndGradientCollision (NL.i:1523-1709, cost and collision flag),
 *      getCostAndGradientPotentialESDF (NL.i:1713-1806), getDistanceSDF (NL.i:1843-1905), getCostPotential
 *      (NL.i:2319-2345), triLerp (NL.i:2451-2464).
 * The trajectory is walked at the fixed time increment `dt` (coll_check_time_increment; t advances by repeated
 * addition, segment by segment); a sample is charged once the path length since the last charged sample reaches
 * `map_resolution`, with  potential(position) * |velocity| * (time since the last charged sample).
 * potential(d): d -= robot_radius;  d <= 0: coll_pot_multiplier * (-d) + epsilon / 2 (collision);
 *               d <= epsilon: (d - epsilon)^2 / (2 epsilon);  else 0.
 * The map classes of the reference (voxblox ESDF, sdf_tools) are un-vendored; the map here is a dense grid:
 *   d_sdf[(i ny + j) nz + k] = distance at the CENTRE of cell (i, j, k), h_dims = {nx, ny, nz};
 *   cell of a point: i = floor((x - origin_x) / resolution); centre of a cell: origin + (i + 0.5) resolution;
 *   a point outside the grid reads oob_value.
 * use_continuous_distance != 0 (ref use_continous_distance): inside [min_bound + map_resolution,
 * max_bound - map_resolution] the distance is the reference's trilinear blend of the 8 cells idx +- 1 (falls back
 * to the cell value when one of them is outside the grid); otherwise the value of the cell that holds the point.
 * D must be 3, N 10.  d_cost [B]; optional d_is_collision [B] (1 when a charged sample was in collision),
 * d_charged [B] (number of charged samples). */
MINSNAP_API int minsnap_collision_cost(long B, int K, int D, int N, const double* d_coeffs,
                                       const double* d_times, const double* d_sdf, const int32_t* h_dims,
                                       const double* h_origin, double resolution, double oob_value,
                                       const double* h_min_bound, const double* h_max_bound,
                                       int use_continuous_distance, double dt, double map_resolution,
                                       double epsilon, double robot_radius, double coll_pot_multiplier,
                                       double* d_cost, int32_t* d_is_collision, int32_t* d_charged,
                                       minsnap_stream_t stream);

/* The same walk with the gradient of the collision cost w.r.t. the free derivatives d_p (ref
 * getCostAndGradientCollision with gradients != NULL, NL.i:1666-1686, "paper equation (14)"): per charged sample
 * whose speed exceeds 1e-6, axis k receives
 *   |v| time_sum dc/dx_k (T^T L_pp)  +  time_sum c v_k / |v| (T^T V L_pp),
 * dc/dx the central difference of the potential over +-map_resolution (getCostAndGradientPotentialESDF,
 * NL.i:1756-1785), L = A^-1 M (NL.i:200-222).  As in the reference, the dependence of the running sums on d_p is
 * not differentiated.  d_col_of_row [N K] = the constraint index map of minsnap_reorder (free columns are
 * n_fixed ..), or NULL for the standard mask (n_free must then be (K-1)(N/2-1)); d_grad_free [B][n_free][3] in
 * the layout of free_values.  d_cost, d_is_collision, d_charged as above. */
MINSNAP_API int minsnap_collision_gradient(long B, int K, int D, int N, const double* d_coeffs,
                                           const double* d_times, const double* d_sdf, const int32_t* h_dims,
                                           const double* h_origin, double resolution, double oob_value,
                                           const double* h_min_bound, const double* h_max_bound,
                                           int use_continuous_distance, double dt, double map_resolution,
                                           double epsilon, double robot_radius, double coll_pot_multiplier,
                                           const int32_t* d_col_of_row, int n_fixed, int n_free,
                                           double* d_cost, double* d_grad_free, int32_t* d_is_collision,
                                           int32_t* d_charged, minsnap_stream_t stream);

/* ---- the free derivatives (and segment times) against the collision cost ---------------------
 * J = w_d J_d + w_c J_c + w_t sum(T), the objective of the reference's nonlinear optimiser over d_p (and T):
 *   J_d = sum_dim d^T R d with d = [d_f; d_p]  (ref getCostAndGradientDerivative, NL.i:1452-1521) -- this is
 *         2 computeCost, NOT computeCost;
 *   J_c = the collision cost of minsnap_collision_cost  (ref getCostAndGradientCollision, NL.i:1523-1709);
 *   w_t sum(T), whose time gradient is the w_t of minsnap_time_gradient  (ref getCostAndGradientTime,
 *         NL.i:2155-2243).
 * h_fixed_mask is a HOST pointer as in minsnap_solve; it reaches the device in a kernel's parameters, not by a copy.
 *
 * minsnap_derivative_gradient: at the given (d_f, d_p, T), any mask, any supported N and D:
 *   d_cost_Jd [B]            J_d = d^T R d (2 computeCost);
 *   d_grad_free [B][n_free][D] dJ_d/dd_p = 2 (R_pf d_f + R_pp d_p), in the layout of free_values;
 *   d_diag_free [B][n_free]  (optional) diag(R_pp);
 *   d_coeffs [B][K][D][N]    (optional) the coefficients, bit-identical to minsnap_coeffs_from_constraints.
 * Deterministic: no atomics, the same bits on every run.  d_workspace: minsnap_solve_workspace_bytes(N, K) bytes. */
MINSNAP_API int minsnap_derivative_gradient(long B, int K, int D, int N, int derivative,
                                            const uint8_t* h_fixed_mask, const double* d_fixed_values,
                                            const double* d_free_values, const double* d_times,
                                            double* d_coeffs, double* d_cost_Jd, double* d_grad_free,
                                            double* d_diag_free, void* d_workspace, size_t workspace_bytes,
                                            minsnap_stream_t stream);

/* minsnap_free_objective: J for S candidates per trajectory.  d_fixed_values [B][n_fixed][D] is shared by the S
 * candidates of trajectory b; d_free_values [B][S][n_free][D], d_times [B][S][K] -> d_objective [B][S]; optional
 * d_Jd, d_Jc [B][S] (the two terms before weighting) and d_is_collision [B][S].  The map and walk parameters are
 * those of minsnap_collision_cost; D must be 3 and N 10 (MINSNAP_ERR_UNSUPPORTED otherwise).  Temporary device
 * memory is allocated stream-ordered (cudaMallocAsync). */
MINSNAP_API int minsnap_free_objective(long B, int S, int K, int D, int N, int derivative,
                                       const uint8_t* h_fixed_mask, const double* d_fixed_values,
                                       const double* d_free_values, const double* d_times, double w_d,
                                       double w_c, double w_t, const double* d_sdf, const int32_t* h_dims,
                                       const double* h_origin, double resolution, double oob_value,
                                       const double* h_min_bound, const double* h_max_bound,
                                       int use_continuous_distance, double dt, double map_resolution,
                                       double epsilon, double robot_radius, double coll_pot_multiplier,
                                       double* d_objective, double* d_Jd, double* d_Jc,
                                       int32_t* d_is_collision, minsnap_stream_t stream);

/* minsnap_optimize_free_constraints: an additive batched driver (NLopt, which the reference uses, is absent, so no
 * parity is claimed for the optimiser -- only for the objective and the gradients it is built from).  Every
 * trajectory descends J over its free derivatives d_p (d_free_values [B][n_free][D], in/out) and, with
 * optimize_times != 0, its segment times (d_times [B][K], in/out).  Per iteration, at the incumbent: J_d, its
 * gradient g_d and diag(R_pp) (minsnap_derivative_gradient), J_c and g_c (minsnap_collision_gradient), with
 * optimize_times the time gradient w_d dJ_d/dT + w_t (minsnap_time_gradient, increment gradient_increment).  Then
 * n_steps candidates, s = 0 .. n_steps-1, move both blocks with the same ladder index:
 *   d_p - 2^-s (w_d g_d + w_c g_c) / (2 w_d diag(R_pp))   (at s = 0 and w_c = 0: the Jacobi step on J_d);
 *   T   as minsnap_optimize_segment_times moves it without a penalty: T - (max_relative_step / 2^s) scale g_T,
 *       scale = min_k T_k / |g_T,k|, clamped at min_time; the times stay when optimize_times == 0.
 * minsnap_free_objective evaluates the candidates; the first minimum among the finite ones is accepted when it is
 * strictly below the incumbent.  w_d > 0.  All launches are on `stream`, the workspace is one cudaMallocAsync and
 * nothing returns to the host: the call can be captured into a CUDA graph once it has run eagerly on the thread.
 * d_history (optional) [iterations + 1][B]: the incumbent J, first at the initial state; d_is_collision (optional)
 * [B]: the collision flag at the returned state.  D must be 3 and N 10. */
MINSNAP_API int minsnap_optimize_free_constraints(long B, int K, int D, int N, int derivative,
                                                  const uint8_t* h_fixed_mask, const double* d_fixed_values,
                                                  double* d_free_values, double* d_times, int optimize_times,
                                                  double w_d, double w_c, double w_t, const double* d_sdf,
                                                  const int32_t* h_dims, const double* h_origin,
                                                  double resolution, double oob_value,
                                                  const double* h_min_bound, const double* h_max_bound,
                                                  int use_continuous_distance, double dt,
                                                  double map_resolution, double epsilon,
                                                  double robot_radius, double coll_pot_multiplier,
                                                  int iterations, int n_steps, double max_relative_step,
                                                  double min_time, double gradient_increment,
                                                  double* d_history, int32_t* d_is_collision,
                                                  minsnap_stream_t stream);

/* ---- the soft limits of minsnap_soft_constraint_cost in the free-derivative problem ---------------------------
 * minsnap_soft_constraint_gradient: the soft cost of solved trajectories d_coeffs [B][K][D][N], d_times [B][K]
 * (D <= 32, any mask h_fixed_mask [(K+1)][N/2]) and its gradient in closed form, in the free derivatives d_p
 * (d_grad_free [B][n_free][D], the layout of d_free_values; required when n_free > 0) and, with the end-point
 * derivatives d held fixed as minsnap_time_gradient holds them, in the segment times (d_grad_times [B][K],
 * optional).  It runs the extrema passes of minsnap_soft_constraint_cost once, then one gradient kernel on their
 * per-segment maxima: for constraint c the maximum m is attained at segment s*, time t* (the first strict maximum in
 * the fold's order: at ties the result is a subgradient), the term is tau = min(maximum_cost, exp((m - L) / L *
 * weight)) and dtau/dm = exp(...) weight / L below maximum_cost, 0 when saturated or when m = 0.  Every mode-0
 * candidate is a stationary point of |p^(k)|^2 in t or a segment start, so dm/dtheta is taken at fixed t*:
 * sum_dim p_dim^(k)(t*) dp_dim^(k)(t*)/dtheta / m, plus the drift sum_dim p^(k) p^(k+1)(T) / m in T when t* is the
 * end of the last segment.  Only segment s* contributes; rows of d_seg that map to fixed constraints drop out.  The
 * terms add in constraint order without atomics, so every run gives the same bits.  d_cost [B] and d_max_value
 * [B][n_constraints] (optional) are those of minsnap_soft_constraint_cost bit for bit; d_max_time and
 * d_max_segment [B][n_constraints] (optional) are t* and s*.  The mask reaches the device in kernel parameters and
 * the scratch is one cudaMallocAsync, so the call can be captured into a CUDA graph. */
MINSNAP_API int minsnap_soft_constraint_gradient(long B, int K, int D, int N, const uint8_t* h_fixed_mask,
                                                 const double* d_coeffs, const double* d_times, int n_constraints,
                                                 const int32_t* h_derivatives, const double* h_limits,
                                                 double weight, double maximum_cost, int extrema_flags,
                                                 double* d_cost, double* d_grad_free, double* d_grad_times,
                                                 double* d_max_value, double* d_max_time, int32_t* d_max_segment,
                                                 minsnap_stream_t stream);

/* minsnap_free_objective_soft: minsnap_free_objective plus w_sc times the soft cost of the recovered candidate
 * coefficients, added last: J = ((w_d J_d + w_c J_c) + w_t sum(T)) + w_sc soft.  w_sc >= 0 and finite; with
 * w_sc = 0 the objective is minsnap_free_objective's bit for bit.  d_soft (optional) [B][S]: the soft cost. */
MINSNAP_API int minsnap_free_objective_soft(long B, int S, int K, int D, int N, int derivative,
                                            const uint8_t* h_fixed_mask, const double* d_fixed_values,
                                            const double* d_free_values, const double* d_times, double w_d,
                                            double w_c, double w_t, const double* d_sdf, const int32_t* h_dims,
                                            const double* h_origin, double resolution, double oob_value,
                                            const double* h_min_bound, const double* h_max_bound,
                                            int use_continuous_distance, double dt, double map_resolution,
                                            double epsilon, double robot_radius, double coll_pot_multiplier,
                                            int n_constraints, const int32_t* h_derivatives,
                                            const double* h_limits, double weight, double maximum_cost,
                                            int extrema_flags, double w_sc, double* d_objective, double* d_Jd,
                                            double* d_Jc, int32_t* d_is_collision, double* d_soft,
                                            minsnap_stream_t stream);

/* minsnap_optimize_free_constraints_soft: minsnap_optimize_free_constraints on the objective of
 * minsnap_free_objective_soft.  Per iteration, at the incumbent, the soft cost's maxima and the gradient of
 * minsnap_soft_constraint_gradient join the other gradients:
 *   d_p - 2^-s ((w_d g_d + w_c g_c) + w_sc g_sc) / (2 w_d diag(R_pp)),
 *   with optimize_times the time ladder on (w_d dJ_d/dT + w_t) + w_sc dsoft/dT.
 * The candidates go through minsnap_free_objective_soft and the same selection; with w_sc = 0 the call returns the
 * bits of minsnap_optimize_free_constraints.  Shapes the recovery kernel refuses return MINSNAP_ERR_UNSUPPORTED before
 * any device work.  The workspace is one cudaMallocAsync of, with S = n_steps, n_fd = n_free D, n_c = n_constraints,
 *   that of minsnap_optimize_free_constraints, 8 B (K D N + 2 n_fd + n_free + K + 3) + 8 B S (n_fd + K + K D N + 3)
 *   + 4 B (S + 1) (+ alignment), plus 8 B (n_fd + S) + 32 B S K n_c bytes:
 * 2.06 GB + 0.40 GB at B = 65,536, K = 10, S = 8, standard mask, two constraints (computed from the shapes).
 * d_max_value (optional) [B][n_constraints]: the maxima at the returned state. */
MINSNAP_API int minsnap_optimize_free_constraints_soft(long B, int K, int D, int N, int derivative,
                                                       const uint8_t* h_fixed_mask, const double* d_fixed_values,
                                                       double* d_free_values, double* d_times, int optimize_times,
                                                       double w_d, double w_c, double w_t, const double* d_sdf,
                                                       const int32_t* h_dims, const double* h_origin,
                                                       double resolution, double oob_value,
                                                       const double* h_min_bound, const double* h_max_bound,
                                                       int use_continuous_distance, double dt,
                                                       double map_resolution, double epsilon, double robot_radius,
                                                       double coll_pot_multiplier, int n_constraints,
                                                       const int32_t* h_derivatives, const double* h_limits,
                                                       double weight, double maximum_cost, int extrema_flags,
                                                       double w_sc, int iterations, int n_steps,
                                                       double max_relative_step, double min_time,
                                                       double gradient_increment, double* d_history,
                                                       int32_t* d_is_collision, double* d_max_value,
                                                       minsnap_stream_t stream);

/* ---- host-buffer entry points (synchronous; copies inside) -------------------------------
 * The calls a host program makes when its data lives in host memory.  Work is cut into
 * chunks that are copied and solved on alternating streams so that PCIe and the SMs overlap.
 * Pinned host buffers (minsnap_host_alloc) make the copies asynchronous.  Calls whose buffers total at most
 * 4 MB (one trajectory from the C++ classes) are staged through a per-thread pinned block: one copy each way.
 * In MINSNAP_EXTREMA_OPTIMIZATION mode minsnap_extrema_host leaves h_min_* untouched. */
MINSNAP_API int minsnap_host_alloc(void** h_ptr, size_t bytes);
MINSNAP_API int minsnap_host_free(void* h_ptr);
MINSNAP_API int minsnap_reorder_host(int N, int K, long n_masks, const uint8_t* h_mask,
                                     int32_t* h_col_of_row, int32_t* h_counts);
MINSNAP_API int minsnap_solve_host(long B, int K, int D, int N, int derivative,
                                   const uint8_t* h_fixed_mask, const double* h_fixed_values,
                                   const double* h_times, double* h_coeffs, double* h_free_values,
                                   double* h_cost, int32_t* h_status, int32_t* h_col_of_row);
MINSNAP_API int minsnap_solve_standard_host(long B, int K, int D, int N, int derivative,
                                            const double* h_positions,
                                            const double* h_end_derivatives, const double* h_times,
                                            double v_max, double a_max, double magic,
                                            double* h_times_out, double* h_coeffs,
                                            double* h_free_values, double* h_cost,
                                            int32_t* h_status);
MINSNAP_API int minsnap_sample_at_host(long B, int K, int D, int N, const double* h_coeffs,
                                       const double* h_times, int M, const double* h_t,
                                       long t_stride, int n_deriv, double* h_out,
                                       int32_t* h_segment);
MINSNAP_API int minsnap_evaluate_range_host(int K, int D, int N, const double* h_coeffs,
                                            const double* h_times, double t_start, double t_end,
                                            double dt, int derivative, int max_samples,
                                            double* h_out, double* h_t_out, int32_t* h_count);
MINSNAP_API int minsnap_segment_matrices_host(long n, int N, int derivative, const double* h_T,
                                              double* h_A, double* h_Ainv, double* h_Q, double* h_H);
MINSNAP_API int minsnap_estimate_segment_times_host(long B, int K, int D, const double* h_positions,
                                                    double v_max, double a_max, double magic,
                                                    double* h_times);
MINSNAP_API int minsnap_coeffs_from_constraints_host(long B, int K, int D, int N,
                                                     const uint8_t* h_fixed_mask,
                                                     const double* h_fixed_values,
                                                     const double* h_free_values,
                                                     const double* h_times, double* h_coeffs);
MINSNAP_API int minsnap_derivative_gradient_host(long B, int K, int D, int N, int derivative,
                                                 const uint8_t* h_fixed_mask,
                                                 const double* h_fixed_values,
                                                 const double* h_free_values, const double* h_times,
                                                 double* h_coeffs, double* h_cost_Jd,
                                                 double* h_grad_free, double* h_diag_free);
MINSNAP_API int minsnap_cost_host(long B, int K, int D, int N, int derivative,
                                  const double* h_coeffs, const double* h_times, double* h_cost);

MINSNAP_API int minsnap_sample_uniform_host(long B, int K, int D, int N, const double* h_coeffs,
                                            const double* h_times, int M, int n_deriv, double* h_out,
                                            double* h_t_out);
MINSNAP_API int minsnap_cost_sweep_host(long B, int S, int K, int D, int N, int derivative,
                                        const double* h_positions, const double* h_end_derivatives,
                                        const double* h_times, double* h_cost, int32_t* h_status);
MINSNAP_API int minsnap_time_objective_host(long B, int S, int K, int D, int N, int derivative,
                                            const double* h_positions, const double* h_end_derivatives,
                                            const double* h_times, double time_penalty,
                                            double* h_objective, double* h_cost, int32_t* h_status);
MINSNAP_API int minsnap_time_gradient_host(long B, int K, int D, int N, int derivative,
                                           const double* h_coeffs, const double* h_times,
                                           double increment, double w_d, double w_t,
                                           double* h_gradient, double* h_segment_cost);
MINSNAP_API int minsnap_collision_cost_host(long B, int K, int D, int N, const double* h_coeffs,
                                            const double* h_times, const double* h_sdf,
                                            const int32_t* h_dims, const double* h_origin,
                                            double resolution, double oob_value,
                                            const double* h_min_bound, const double* h_max_bound,
                                            int use_continuous_distance, double dt,
                                            double map_resolution, double epsilon, double robot_radius,
                                            double coll_pot_multiplier, double* h_cost,
                                            int32_t* h_is_collision, int32_t* h_charged);

MINSNAP_API int minsnap_collision_gradient_host(long B, int K, int D, int N, const double* h_coeffs,
                                                const double* h_times, const double* h_sdf,
                                                const int32_t* h_dims, const double* h_origin,
                                                double resolution, double oob_value,
                                                const double* h_min_bound, const double* h_max_bound,
                                                int use_continuous_distance, double dt,
                                                double map_resolution, double epsilon, double robot_radius,
                                                double coll_pot_multiplier, const int32_t* h_col_of_row,
                                                int n_fixed, int n_free, double* h_cost, double* h_grad_free,
                                                int32_t* h_is_collision, int32_t* h_charged);

MINSNAP_API int minsnap_extrema_host(long B, int K, int D, int N, const double* h_coeffs,
                                     const double* h_times, int derivative, int mode,
                                     uint32_t dim_mask, double* h_max_time, double* h_max_value,
                                     int32_t* h_max_segment, double* h_min_time,
                                     double* h_min_value, int32_t* h_min_segment,
                                     double* h_cand_times, double* h_cand_values,
                                     int32_t* h_root_count);

/* ---- SURVEY 8(f)4: interchange formats -- HOST ONLY except for the sampling inside the table ---------
 * NumPy .npy files (format 1.0, little-endian float64, C order) for the batched arrays of this header --
 * coefficients [B][K][D][N], samples [B][M][n_deriv][D], times [B][K] -- readable by numpy.load and writable by
 * numpy.save.  minsnap_npy_read_f64: h_data == NULL reads only ndim / shape (shape has room for 8 entries);
 * MINSNAP_ERR_WORKSPACE when capacity (in elements) is too small, MINSNAP_ERR_UNSUPPORTED for other dtypes.
 * minsnap_sampled_table_host: the table of ref printMatlabSampledTrajectory (NL.i:2567-2662) for one trajectory,
 * rows [t, pos(D), vel(D), acc(D), jerk(D), snap(D), t_vertex], rows = sum_i (ceil(T_i / dt) + 1)
 * (minsnap_sampled_table_rows; the reference uses dt = 0.01), cols = 5 D + 2, sampled on the GPU;
 * minsnap_table_write_text writes it as whitespace-separated text with 17 significant digits. */
MINSNAP_API int minsnap_npy_write_f64(const char* path, const double* h_data, int ndim, const int64_t* shape);
MINSNAP_API int minsnap_npy_read_f64(const char* path, double* h_data, size_t capacity, int* ndim,
                                     int64_t* shape);
MINSNAP_API int minsnap_sampled_table_rows(int K, const double* h_times, double dt);
MINSNAP_API int minsnap_sampled_table_host(int K, int D, int N, const double* h_coeffs,
                                           const double* h_times, double dt, double* h_table,
                                           int capacity_rows, int* rows_out, int* cols_out);
MINSNAP_API int minsnap_table_write_text(const char* path, const double* h_table, int rows, int cols);

/* ---- a3: synthetic inputs (ref: createRandomVertices, src/vertex.cpp:27-79) -- HOST ONLY ----
 * positions[b] = vertex positions of createRandomVertices(., K, pos_min, pos_max, base_seed + b):
 * std::mt19937 + one std::uniform_real_distribution<double> per axis, a vertex closer than 0.2
 * to its predecessor is redrawn.  The constraint structure (standard mask, zero end
 * derivatives) is implied.  No GPU involved: this only manufactures workloads. */
MINSNAP_API int minsnap_random_positions_host(long B, int K, int D, const double* h_pos_min,
                                              const double* h_pos_max, uint64_t base_seed,
                                              double* h_positions);

/* ---- measurement helper: dependency-free DFMA loop, reports achieved FP64 TFLOP/s --------- */
MINSNAP_API int minsnap_fp64_peak(int repeats, double* tflops);

#ifdef __cplusplus
}
#endif
#endif /* MINSNAP_B200_H_ */
