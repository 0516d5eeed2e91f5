// Internal launch interface between the C ABI (minsnap_capi.cu) and the kernel translation
// units.  Every function enqueues work on `stream` and returns the cudaError_t of the launch.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <optional>

namespace minsnap {

// Largest dynamic shared memory a CTA may request on sm_100 (227 KB).
constexpr size_t kMaxDynamicSmem = 227 * 1024;

// Multiprocessors of the current device (148 on B200), queried once per device: grid caps and the batch-size
// thresholds between kernels scale with it instead of carrying the number.
inline long sm_count() {
  static int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    cached[dev] = (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) == cudaSuccess && n > 0) ? n : 148;
  }
  return cached[dev];
}

bool supported_n(int N);

// Stream-ordered scratch memory, freed on `stream` when it goes out of scope (after the work enqueued so far).
struct AsyncBuffer {
  void* ptr = nullptr;
  cudaStream_t stream = nullptr;
  cudaError_t alloc(size_t bytes, cudaStream_t s) {
    stream = s;
    return cudaMallocAsync(&ptr, bytes ? bytes : 16, s);
  }
  ~AsyncBuffer() {
    if (ptr) cudaFreeAsync(ptr, stream);
  }
};

// ---- minsnap_general.cu ----------------------------------------------------------------
cudaError_t launch_reorder(int N, int K, long n_masks, const uint8_t* d_mask, int32_t* d_col_of_row,
                           int32_t* d_counts, cudaStream_t stream);
cudaError_t launch_estimate_times(long B, int K, int D, const double* d_positions, double v_max,
                                  double a_max, double magic, double* d_times, cudaStream_t stream);
cudaError_t launch_segment_matrices(long n, int N, int derivative, const double* d_T, double* d_A,
                                    double* d_Ainv, double* d_Q, double* d_H, cudaStream_t stream);

struct GeneralSolveArgs {
  long B;
  int K, D, N, derivative, n_fixed, n_free;
  int fixed_div = 1;            // problem b uses fixed-value record b / fixed_div
  const int32_t* d_col_of_row;  // [N*K]
  const double* d_fixed_values; // [B][n_fixed][D]
  const double* d_free_in;      // [B][n_free][D]; only for coefficient recovery
  const double* d_times;        // [B][K]
  double* d_coeffs;             // [B][K][D][N] (optional for cost-only runs)
  double* d_free_out;           // optional
  double* d_cost;               // optional; J_d = d^T R d instead of computeCost in launch_derivative_gradient
  int32_t* d_status;            // optional
  double* d_grad_free = nullptr;  // [B][n_free][D], launch_derivative_gradient only: dJ_d/dd_p
  double* d_diag_free = nullptr;  // [B][n_free], launch_derivative_gradient only (optional): diag(R_pp)
};
// Returns cudaErrorInvalidConfiguration when one problem does not fit shared memory.
cudaError_t launch_solve_general(const GeneralSolveArgs& a, cudaStream_t stream);
// cudaErrorInvalidConfiguration where launch_solve_general would refuse the shape, without launching anything
cudaError_t general_fits(int N, int K, int D, int n_fixed, int n_free);
cudaError_t launch_coeffs_from_constraints(const GeneralSolveArgs& a, cudaStream_t stream);
// coefficient recovery plus J_d, its gradient in d_p and diag(R_pp) (d_grad_free and d_cost required)
cudaError_t launch_derivative_gradient(const GeneralSolveArgs& a, cudaStream_t stream);

// A (K+1) x h mask packed into bits, passed by value to the kernel that unpacks it on the device.
struct MaskBits {
  static constexpr int kWords = 512;   // 16,384 constraints, beyond what the general kernel's shared memory takes
  uint32_t words[kWords];
};
// launch_reorder of one HOST mask, without a host-to-device copy (capturable into a CUDA graph); d_mask receives the
// unpacked mask.  cudaErrorInvalidConfiguration when the mask has more than 32 * MaskBits::kWords entries.
cudaError_t launch_reorder_host_mask(int N, int K, const uint8_t* h_mask, uint8_t* d_mask, int32_t* d_col_of_row,
                                     int32_t* d_counts, cudaStream_t stream);
cudaError_t launch_cost(long B, int K, int D, int N, int derivative, const double* d_coeffs,
                        const double* d_times, double* d_cost, cudaStream_t stream);

// SURVEY 8(f)2 (ref getCostAndGradientTime NL.i:2155-2243, objectiveFunctionTime NL.i:765-832)
cudaError_t launch_time_gradient(long B, int K, int D, int N, int derivative, const double* d_coeffs,
                                 const double* d_times, double increment, double w_d, double w_t, double* d_gradient,
                                 double* d_segment_cost, cudaStream_t stream);
cudaError_t launch_add_time_penalty(long n, int K, const double* d_times, const double* d_cost, double time_penalty,
                                    double* d_objective, cudaStream_t stream);

// device-side glue of the batched time descent (SURVEY 8(f)2)
cudaError_t launch_time_candidates(long B, int S, int K, const double* d_times, const double* d_grad_cost,
                                   double time_penalty, double max_relative_step, double min_time, double* d_cand,
                                   cudaStream_t stream);
cudaError_t launch_time_select(long B, int S, int K, const double* d_cand, const double* d_cost, double time_penalty,
                               double* d_times, double* d_incumbent, double* d_history_row, cudaStream_t stream);

// device-side glue of the batched descent on the free derivatives (minsnap_optimize_free_constraints)
cudaError_t launch_free_candidates(long B, int S, int n_free, int D, int K, const double* d_free, const double* d_grad_d,
                                   const double* d_grad_c, const double* d_diag, double w_d, double w_c,
                                   const double* d_times, double* d_cand_free, double* d_cand_times,
                                   cudaStream_t stream, const double* d_grad_sc = nullptr, double w_sc = 0.0);
cudaError_t launch_free_combine(long n, int K, const double* d_cost, const double* d_jc, const double* d_times,
                                double w_d, double w_c, double w_t, double* d_objective, double* d_jd,
                                cudaStream_t stream);
// objective[i] += w_sc soft[i] (minsnap_free_objective_soft: the soft term added last)
cudaError_t launch_free_soft_add(long n, const double* d_soft, double w_sc, double* d_objective, cudaStream_t stream);
cudaError_t launch_free_select(long B, int S, int n_fd, int K, const double* d_cand_obj, const double* d_cand_free,
                               const double* d_cand_times, const int32_t* d_cand_hit, double* d_free, double* d_times,
                               double* d_incumbent, int32_t* d_hit, double* d_history_row, cudaStream_t stream);

// device-side glue of the time descent with soft limits (minsnap_optimize_segment_times_soft)
// out_p[b R + r] = positions[b] (row_p doubles each), out_e likewise when d_end is set
cudaError_t launch_replicate_rows(long B, int R, int row_p, const double* d_positions, double* d_out_p, int row_e,
                                  const double* d_end, double* d_out_e, cudaStream_t stream);
// cand[(b K + n) 2 + j] = times[b] with segment n moved by -/+ increment (j = 0 / 1); a time <= 0.1 moves to 0.1
cudaError_t launch_soft_gradient_candidates(long B, int K, const double* d_times, double increment, double* d_cand,
                                            cudaStream_t stream);
// gradient[b K + n] += (soft[(b K + n) 2 + 1] - soft[(b K + n) 2]) / (2 increment)
cudaError_t launch_soft_gradient_add(long B, int K, const double* d_soft, double increment, double* d_gradient,
                                     cudaStream_t stream);

// ---- minsnap_standard.cu ---------------------------------------------------------------
// The kernels behind minsnap_solve_standard; choose_standard_route (minsnap_standard_route.cuh) picks one.
enum class StandardRoute { Tm, Pair, PairLong, Bcr, Chunked, General, Unsupported };

// The names MINSNAP_STANDARD_ROUTE takes.
inline const char* standard_route_name(StandardRoute r) {
  static const char* const names[] = {"tm", "pair", "pair_long", "bcr", "chunked", "general", "unsupported"};
  return names[static_cast<int>(r)];
}

struct StandardSolveArgs {
  long B;
  int K, D, N, derivative;
  const double* d_positions;       // [B][K+1][D]
  const double* d_end_derivatives; // [B][2][h-1][D] or NULL
  const double* d_times;           // [B][K] or NULL
  double v_max, a_max, magic;
  double* d_times_out;             // optional
  double* d_coeffs;                // [B][K][D][N]
  double* d_free_out;              // optional [B][n_free][D]
  double* d_cost;                  // optional
  int32_t* d_status;               // optional
  std::optional<StandardRoute> forced;  // this route or cudaErrorNotSupported, never a fallback
};
bool standard_supported(int K, int D, int N, int derivative);
cudaError_t launch_solve_standard(const StandardSolveArgs& a, cudaStream_t stream);

struct SweepArgs {
  long B;
  int S, K, D, N, derivative;
  const double* d_positions;
  const double* d_end_derivatives;
  const double* d_times; // [B][S][K]
  double* d_cost;        // [B][S]
  int32_t* d_status;     // optional [B][S]
};
cudaError_t launch_cost_sweep(const SweepArgs& a, cudaStream_t stream);

// ---- minsnap_sample.cu -----------------------------------------------------------------
struct SampleArgs {
  long B;
  int K, D, N, M, n_deriv;
  const double* d_coeffs;
  const double* d_times;
  const double* d_t;   // NULL => uniform grid
  long t_stride;       // 0 => shared row
  double* d_out;       // [B][M][n_deriv][D]
  double* d_t_out;     // optional [B][M]
  int32_t* d_segment;  // optional [B][M]
};
cudaError_t launch_sample(const SampleArgs& a, cudaStream_t stream);
cudaError_t launch_evaluate_range(long B, int K, int D, int N, const double* d_coeffs,
                                  const double* d_times, double t_start, double t_end, double dt,
                                  int derivative, int max_samples, double* d_out, double* d_t_out,
                                  int32_t* d_count, cudaStream_t stream);

// ---- minsnap_extrema.cu ----------------------------------------------------------------
struct ExtremaArgs {
  long B;
  int K, D, N, derivative;
  int mode;            // 0: computeMaximumOfMagnitude (LIN.i:470-503), 1: Trajectory::computeMinMaxMagnitude
  bool keep_small;     // false: drop trailing coefficients below machine epsilon like the reference
  uint32_t dim_mask;   // dimensions that take part (never 0 here)
  const double* d_coeffs;
  const double* d_times;
  double* d_max_time;      // [B] each, optional
  double* d_max_value;
  int32_t* d_max_segment;
  double* d_min_time;      // mode 1 only
  double* d_min_value;
  int32_t* d_min_segment;
  double* d_cand_times;    // optional [B][K][max_roots + 2]: start, end, roots (ascending)
  double* d_cand_values;   // optional, same shape
  int32_t* d_root_count;   // optional [B][K]
  int max_roots;
};
int extrema_max_roots(int N, int derivative, int n_dims);
cudaError_t launch_extrema(const ExtremaArgs& a, cudaStream_t stream);

// Soft limits on max |p^(k)| over all dimensions (ref evaluateMaximumMagnitudeAsSoftConstraint NL.i:2396-2426 over
// computeMaximumOfMagnitude, mode 0): soft = sum_c min(maximum_cost, exp((max_c - limit_c) / limit_c * weight)).
// The constraints travel by value in the kernels' parameters.
constexpr int kMaxSoftConstraints = 4;
struct SoftConstraintArgs {
  long B;
  int K, D, N;
  int n_constraints;
  int derivative[kMaxSoftConstraints];
  double limit[kMaxSoftConstraints];
  double weight, maximum_cost;
  bool keep_small;
  const double* d_coeffs;   // [B][K][D][N]
  const double* d_times;    // [B][K]
  void* d_scratch;          // soft_constraint_scratch_bytes(B, K, n_constraints)
  double* d_soft;           // optional [B]
  double* d_terms;          // optional [B][n_constraints]
  double* d_max_value;      // optional [B][n_constraints]
  // objective epilogue, on when d_objective is set: cost + time_penalty (sum_k times)^2 + soft, NaN where status != 0
  double* d_objective = nullptr;  // [B]
  const double* d_cost = nullptr; // [B] computeCost
  const int32_t* d_status = nullptr;  // optional [B]
  double time_penalty = 0.0;
};
size_t soft_constraint_scratch_bytes(long B, int K, int n_constraints);
cudaError_t launch_soft_constraint_cost(const SoftConstraintArgs& a, cudaStream_t stream);

// The soft cost's gradient in the free derivatives and in the segment times (d held fixed), from the per-segment
// maxima launch_soft_constraint_cost left in soft.d_scratch for the same coefficients and times.
struct SoftGradientArgs {
  SoftConstraintArgs soft;
  const int32_t* d_col_of_row;   // [N K] constraint index map
  int n_fixed, n_free;
  double* d_grad_free;           // [B][n_free][D]
  double* d_grad_times;          // optional [B][K]
  bool add_times = false;        // d_grad_times += times_weight g_T instead of d_grad_times = g_T
  double times_weight = 1.0;
  double* d_max_time = nullptr;  // optional [B][n_constraints]
  int32_t* d_max_segment = nullptr;
};
cudaError_t launch_soft_constraint_gradient(const SoftGradientArgs& a, cudaStream_t stream);

// ---- minsnap_collision.cu ---------------------------------------------------------------
// SURVEY 8(f)3 (ref getCostAndGradientCollision NL.i:1523-1709): collision cost against a dense distance grid
struct CollisionArgs {
  long B;
  int K, N;                 // D = 3
  const double* d_coeffs;   // [B][K][3][N]
  const double* d_times;    // [B][K]
  const double* d_sdf;      // [nx][ny][nz], distance at the cell centres
  int nx, ny, nz;
  double origin[3], resolution, oob_value;
  double min_bound[3], max_bound[3];
  int use_continuous_distance;
  double dt, map_resolution, epsilon, robot_radius, coll_pot_multiplier;
  double* d_cost;           // [B]
  int32_t* d_is_collision;  // optional [B]
  int32_t* d_charged;       // optional [B]: number of samples that were charged
  // gradient w.r.t. the free derivatives (NL.i:1666-1686); all unused when d_grad_free is null
  double* d_grad_free;          // [B][n_free][3], ZERO on entry
  const int32_t* d_col_of_row;  // [N K] constraint index map, or null = the standard mask
  int n_fixed, n_free;
};
cudaError_t launch_collision_cost(const CollisionArgs& a, cudaStream_t stream);

// ---- minsnap_peak.cu -------------------------------------------------------------------
cudaError_t run_fp64_peak(int repeats, double* tflops);

}  // namespace minsnap
