// General-mask kernels: any fixed/free pattern, any K that fits shared memory, any D.
// One warp owns one trajectory; R_pp lives in shared memory as a symmetric band.
//
// Reference rows (SURVEY.md section 8a): a2 estimateSegmentTimes, a5-a9 segment matrices,
// a10 constraint reordering, a11 constructR, a12 solveLinear, a13 coefficient recovery,
// a16 computeCost.  Citations: LIN.i = impl/polynomial_optimization_linear_impl.h.
#include "minsnap_device.cuh"
#include "minsnap_launch.h"

namespace minsnap {

bool supported_n(int N) { return N == 4 || N == 6 || N == 8 || N == 10 || N == 12; }

// =========================================================================================
// a10. Constraint reordering (ref: setupConstraintReorderingMatrix, LIN.i:171-250).
// Column order = fixed constraints sorted by (vertex, derivative), then free ones sorted the
// same way (the reference's two std::set<Constraint>); row order = per segment
// [start vertex: derivative 0..h-1 ; end vertex: derivative 0..h-1].  A warp scans the mask
// 32 entries at a time with ballot/popc prefix counts.  Integer-only, bit-exact.
// =========================================================================================
__global__ void __launch_bounds__(32) reorder_kernel(int N, int K, long n_masks,
                                                     const uint8_t* __restrict__ mask,
                                                     int32_t* __restrict__ col_of_row,
                                                     int32_t* __restrict__ counts) {
  extern __shared__ int32_t col_of_constraint[];  // [(K+1)*h]
  const int lane = threadIdx.x;
  const int h = N / 2;
  const int nc = (K + 1) * h;
  const unsigned lt = (1u << lane) - 1u;
  for (long m = blockIdx.x; m < n_masks; m += gridDim.x) {
    const uint8_t* mk = mask + m * nc;
    int n_fixed = 0;
    for (int base = 0; base < nc; base += kWarp) {
      const int idx = base + lane;
      const bool f = idx < nc && mk[idx] != 0;
      n_fixed += __popc(__ballot_sync(0xffffffffu, f));
    }
    int cf = 0, cp = n_fixed;
    for (int base = 0; base < nc; base += kWarp) {
      const int idx = base + lane;
      const bool valid = idx < nc;
      const bool f = valid && mk[idx] != 0;
      const unsigned bf = __ballot_sync(0xffffffffu, f);
      const unsigned bp = __ballot_sync(0xffffffffu, valid && !f);
      if (valid) col_of_constraint[idx] = f ? cf + __popc(bf & lt) : cp + __popc(bp & lt);
      cf += __popc(bf);
      cp += __popc(bp);
    }
    __syncwarp();
    for (int row = lane; row < N * K; row += kWarp) {
      const int seg = row / N, r = row - seg * N;
      const int at_end = r >= h;
      col_of_row[m * (long)(N * K) + row] = col_of_constraint[(seg + at_end) * h + (r - at_end * h)];
    }
    if (lane == 0) {
      counts[2 * m] = n_fixed;
      counts[2 * m + 1] = nc - n_fixed;
    }
    __syncwarp();
  }
}

cudaError_t launch_reorder(int N, int K, long n_masks, const uint8_t* d_mask, int32_t* d_col_of_row,
                           int32_t* d_counts, cudaStream_t stream) {
  const size_t smem = sizeof(int32_t) * (size_t)(K + 1) * (N / 2);
  if (smem > kMaxDynamicSmem) return cudaErrorInvalidConfiguration;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(reorder_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  const int grid = (int)(n_masks < sm_count() * 32 ? n_masks : sm_count() * 32);
  reorder_kernel<<<grid, 32, smem, stream>>>(N, K, n_masks, d_mask, d_col_of_row, d_counts);
  return cudaGetLastError();
}

// =========================================================================================
// a2. estimateSegmentTimes (ref: src/vertex.cpp:162-178), one thread per segment.
// =========================================================================================
__device__ inline double estimate_time(const double* __restrict__ p0, const double* __restrict__ p1, int D,
                                       double v_max, double a_max, double magic) {
  double s = 0.0;
  for (int d = 0; d < D; ++d) {
    const double diff = p1[d] - p0[d];
    s += diff * diff;
  }
  const double distance = sqrt(s);
  return distance / v_max * 2 * (1.0 + magic * v_max / a_max * exp(-distance / v_max * 2));
}

__global__ void estimate_times_kernel(long n_segments_total, int K, int D, const double* __restrict__ positions,
                                      double v_max, double a_max, double magic, double* __restrict__ times) {
  for (long t = blockIdx.x * (long)blockDim.x + threadIdx.x; t < n_segments_total;
       t += (long)gridDim.x * blockDim.x) {
    const long b = t / K;
    const int i = (int)(t - b * K);
    const double* p0 = positions + (b * (K + 1) + i) * D;
    times[t] = estimate_time(p0, p0 + D, D, v_max, a_max, magic);
  }
}

cudaError_t launch_estimate_times(long B, int K, int D, const double* d_positions, double v_max, double a_max,
                                  double magic, double* d_times, cudaStream_t stream) {
  const long total = B * K;
  if (total == 0) return cudaSuccess;
  const int block = 256;
  long grid = (total + block - 1) / block;
  if (grid > sm_count() * 16) grid = sm_count() * 16;
  estimate_times_kernel<<<(int)grid, block, 0, stream>>>(total, K, D, d_positions, v_max, a_max, magic, d_times);
  return cudaGetLastError();
}

// =========================================================================================
// a5-a9, a11. Per-segment matrices through the closed forms; one warp per segment time.
// =========================================================================================
template <int N>
__global__ void segment_matrices_kernel(long n, int delta, const double* __restrict__ T_in, double* __restrict__ A,
                                        double* __restrict__ Ainv, double* __restrict__ Q, double* __restrict__ H) {
  constexpr int h = N / 2;
  const int lane = threadIdx.x & 31;
  const long warp = blockIdx.x * (long)(blockDim.x >> 5) + uniform_warp_index();
  const long n_warps = ((long)gridDim.x * blockDim.x) >> 5;
  const double* a1 = UnitTables<N>::a1inv();
  const double* h1 = UnitTables<N>::h1(delta);
  for (long s = warp; s < n; s += n_warps) {
    const double T = T_in[s];
    for (int e = lane; e < N * N; e += kWarp) {
      const int r = e / N, c = e - r * N;
      const int kr = r % h, kc = c % h;
      if (A) {
        double v;
        if (r < h) v = (c == r) ? falling_factorial(r, r) : 0.0;            // row at t = 0
        else v = (c >= kr) ? falling_factorial(kr, c) * int_power(T, c - kr) : 0.0;  // row at t = T
        A[s * N * N + e] = v;
      }
      if (Ainv) Ainv[s * N * N + e] = a1[e] * int_power(T, kc - r);
      if (Q) {
        double v = 0.0;
        if (r >= delta && c >= delta) {
          const int ex = r + c - 2 * delta + 1;
          v = 2.0 * falling_factorial(delta, r) * falling_factorial(delta, c) / (double)ex * int_power(T, ex);
        }
        Q[s * N * N + e] = v;
      }
      if (H) H[s * N * N + e] = h1[e] * int_power(T, kr + kc + 1 - 2 * delta);
    }
  }
}

template <int N>
static cudaError_t launch_segment_matrices_n(long n, int delta, const double* d_T, double* d_A, double* d_Ainv,
                                             double* d_Q, double* d_H, cudaStream_t stream) {
  const int block = 128;
  long grid = (n * 32 + block - 1) / block;
  if (grid > sm_count() * 16) grid = sm_count() * 16;
  if (grid < 1) grid = 1;
  segment_matrices_kernel<N><<<(int)grid, block, 0, stream>>>(n, delta, d_T, d_A, d_Ainv, d_Q, d_H);
  return cudaGetLastError();
}

#define MINSNAP_DISPATCH_N(N_, CALL)                 \
  switch (N_) {                                      \
    case 4: { constexpr int kN = 4; CALL; } break;   \
    case 6: { constexpr int kN = 6; CALL; } break;   \
    case 8: { constexpr int kN = 8; CALL; } break;   \
    case 10: { constexpr int kN = 10; CALL; } break; \
    case 12: { constexpr int kN = 12; CALL; } break; \
    default: return cudaErrorInvalidValue;           \
  }

cudaError_t launch_segment_matrices(long n, int N, int derivative, const double* d_T, double* d_A, double* d_Ainv,
                                    double* d_Q, double* d_H, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  MINSNAP_DISPATCH_N(N, return launch_segment_matrices_n<kN>(n, derivative, d_T, d_A, d_Ainv, d_Q, d_H, stream));
  return cudaSuccess;
}

// =========================================================================================
// a11-a13 + a16. General solve: warp per trajectory.
//
// Shared memory per CTA : H1[N*N], A1inv[N*N], col_of_row[N*K] (int32)
// Shared memory per warp: tpow[K][2N-1]   T_i^e for e = -(N-1) .. N-1
//                         band[n_free][N]  lower band of R_pp: band[c][j] = R_pp[c+j][c];
//                                          overwritten by the unit-lower LDL^T factor, with the
//                                          reciprocal pivot in band[c][0]
//                         rhs[n_free][D]   -R_pf d_f, overwritten by y, then by d_p
//                         df[n_fixed][D]   fixed values in column order
//                         acol[N]          the un-scaled pivot column of the current step
// The free columns are ordered by (vertex, derivative), so two free columns that share a
// segment are at most N-1 apart: the half bandwidth is N-1 for every mask.
// =========================================================================================
template <int N>
struct GeneralLayout {
  static constexpr int PW = 2 * N - 1;
  __host__ __device__ static size_t per_warp_doubles(int K, int D, int n_fixed, int n_free) {
    return (size_t)K * PW + (size_t)n_free * N + (size_t)n_free * D + (size_t)n_fixed * D + N;
  }
  __host__ __device__ static size_t cta_bytes(int warps, int K, int D, int n_fixed, int n_free) {
    size_t doubles = 2 * N * N + warps * per_warp_doubles(K, D, n_fixed, n_free);
    return doubles * sizeof(double) + sizeof(int32_t) * (size_t)N * K;
  }
};

struct GeneralKernelParams {
  long B;
  int K, D, delta, n_fixed, n_free, warps;
  int fixed_div;  // problem b reads fixed values of record b / fixed_div (time sweeps share them)
  const int32_t* col_of_row;
  const double* fixed_values;
  const double* free_in;
  const double* times;
  double* coeffs;
  double* free_out;
  double* cost;
  int32_t* status;
  // kGrad only (appended so that the other instantiations see the same parameter offsets)
  double* grad_free;  // [B][n_free][D]: dJ_d/dd_p = 2 (R_pf d_f + R_pp d_p)
  double* diag_free;  // [B][n_free]: diag(R_pp), optional
};

// d value of end-point row r of segment seg in dimension dim.
__device__ inline double dvalue(const int32_t* col, const double* df, const double* dp, int n_fixed, int D, int row,
                                int dim) {
  const int c = col[row];
  return c < n_fixed ? df[c * D + dim] : dp[(c - n_fixed) * D + dim];
}

// Coefficient recovery (a13) and optional cost (a16) for one trajectory held in shared memory.  kGrad adds the
// gradient of J_d = d^T R d in the free derivatives and diag(R_pp), and writes J_d (not 0.5 J_d) to p.cost.
template <int N, bool kGrad>
__device__ inline void recover_coefficients(const GeneralKernelParams& p, long b, int lane, const double* H1s,
                                            const double* A1s, const int32_t* col, const double* tpow,
                                            const double* df, const double* dp, int& nonfinite) {
  constexpr int h = N / 2;
  constexpr int PW = 2 * N - 1;
  const int total = p.K * p.D * N;
  double* out = p.coeffs + b * (long)total;
  double cost_acc = 0.0;
  for (int t = lane; t < total; t += kWarp) {
    const int n = t % N;
    const int dim = (t / N) % p.D;
    const int seg = t / (N * p.D);
    const double* tp = tpow + seg * PW + (N - 1);
    // coefficient n of (seg, dim): sum_r A1inv[n][r] T^(k_r - n) d_r
    double acc = 0.0;
#pragma unroll
    for (int r = 0; r < N; ++r) {
      const double a = A1s[n * N + r];
      if (a != 0.0) acc += a * tp[(r % h) - n] * dvalue(col, df, dp, p.n_fixed, p.D, seg * N + r, dim);
    }
    if (p.coeffs) out[t] = acc;
    if (!isfinite(acc)) nonfinite = 1;
    if (p.cost) {
      // row n of the per-segment quadratic form d^T H_T d (accurate route, SURVEY 8d)
      const int kn = n % h;
      double row = 0.0;
#pragma unroll
      for (int s = 0; s < N; ++s)
        row += H1s[n * N + s] * tp[kn + (s % h) + 1 - 2 * p.delta] *
               dvalue(col, df, dp, p.n_fixed, p.D, seg * N + s, dim);
      cost_acc += row * dvalue(col, df, dp, p.n_fixed, p.D, seg * N + n, dim);
    }
  }
  if (p.cost) {
    cost_acc = warp_sum(cost_acc);
    if (lane == 0) p.cost[b] = kGrad ? cost_acc : 0.5 * cost_acc;
  }
  if (kGrad) {
    // Free column c is the constraint (vertex v, derivative k).  Two rows map to it: row h+k of segment v-1 (its
    // end) and row k of segment v (its start), so (R d)_c = (H_{v-1} d_{v-1})_{h+k} + (H_v d_v)_k and
    // R_pp[c][c] = H_{v-1}[h+k][h+k] + H_v[k][k].  One lane owns each (v, k, dim) and adds the two rows in that
    // order: every output has one writer and a fixed summation order, so the result is bitwise reproducible.
    const int n_vk = (p.K + 1) * h;
    for (int t = lane; t < n_vk * p.D; t += kWarp) {
      const int dim = t % p.D;
      const int v = t / (p.D * h), k = (t / p.D) % h;
      const int c = (v < p.K ? col[v * N + k] : col[(v - 1) * N + h + k]) - p.n_fixed;
      if (c < 0) continue;
      double g = 0.0, diag = 0.0;
#pragma unroll
      for (int side = 0; side < 2; ++side) {   // 0: end of segment v-1, 1: start of segment v
        const int seg = v - 1 + side, n = side ? k : h + k;
        if (seg < 0 || seg >= p.K) continue;
        const double* tp = tpow + seg * PW + (N - 1) + 1 - 2 * p.delta;
        double row = 0.0;
#pragma unroll
        for (int s = 0; s < N; ++s)
          row += H1s[n * N + s] * tp[k + (s % h)] * dvalue(col, df, dp, p.n_fixed, p.D, seg * N + s, dim);
        g += row;
        diag += H1s[n * N + n] * tp[2 * k];
      }
      p.grad_free[(b * p.n_free + c) * p.D + dim] = 2.0 * g;
      if (p.diag_free && dim == 0) p.diag_free[b * p.n_free + c] = diag;
    }
  }
}

template <int N, bool kSolve, bool kGrad = false>
__global__ void __launch_bounds__(256) solve_general_kernel(GeneralKernelParams p) {
  constexpr int h = N / 2;
  constexpr int PW = 2 * N - 1;
  constexpr int HB = N - 1;               // half bandwidth
  constexpr int NP = HB * (HB + 1) / 2;   // (p, q) update pairs per pivot step
  constexpr int NPASS = (NP + kWarp - 1) / kWarp;

  extern __shared__ double smem[];
  const int lane = threadIdx.x & 31;
  const int warp = uniform_warp_index();
  const int K = p.K, D = p.D, n_fixed = p.n_fixed, n_free = p.n_free;
  const size_t per_warp = GeneralLayout<N>::per_warp_doubles(K, D, n_fixed, n_free);

  double* H1s = smem;
  double* A1s = H1s + N * N;
  double* wbase = A1s + N * N + warp * per_warp;
  double* tpow = wbase;
  double* band = tpow + (size_t)K * PW;
  double* rhs = band + (size_t)n_free * N;
  double* df = rhs + (size_t)n_free * D;
  double* acol = df + (size_t)n_fixed * D;
  int32_t* col = reinterpret_cast<int32_t*>(A1s + N * N + p.warps * per_warp);

  {
    const double* h1 = UnitTables<N>::h1(p.delta);
    const double* a1 = UnitTables<N>::a1inv();
    for (int i = threadIdx.x; i < N * N; i += blockDim.x) {
      H1s[i] = h1[i];
      A1s[i] = a1[i];
    }
    for (int i = threadIdx.x; i < N * K; i += blockDim.x) col[i] = p.col_of_row[i];
  }
  __syncthreads();

  // (p, q) pairs of the trailing update handled by this lane, 1 <= q <= p <= HB
  int pair_p[NPASS], pair_q[NPASS];
#pragma unroll
  for (int u = 0; u < NPASS; ++u) {
    const int t = lane + u * kWarp;
    int pp = 1;
    while (pp * (pp + 1) / 2 <= t) ++pp;  // pp(pp-1)/2 <= t < pp(pp+1)/2
    pair_p[u] = pp;
    pair_q[u] = t - pp * (pp - 1) / 2 + 1;
  }

  for (long b = (long)blockIdx.x * p.warps + warp; b < p.B; b += (long)gridDim.x * p.warps) {
    int status = 0;
    // ---- a9: powers of the segment times ------------------------------------------------
    const double* Tb = p.times + b * K;
    for (int t = lane; t < K * PW; t += kWarp) {
      const int seg = t / PW;
      const double T = Tb[seg];
      if (!(T > 0.0)) status |= 2;  // MINSNAP_STATUS_BAD_TIME (ref: CHECK_GT, LIN.i:287)
      tpow[t] = int_power(T, t - seg * PW - (N - 1));
    }
    for (int t = lane; t < n_fixed * D; t += kWarp)
      df[t] = p.fixed_values[(b / p.fixed_div) * (long)(n_fixed * D) + t];

    if (kSolve) {
      for (int t = lane; t < n_free * N; t += kWarp) band[t] = 0.0;
      for (int t = lane; t < n_free * D; t += kWarp) rhs[t] = 0.0;
      __syncwarp();

      // ---- a11: R_pp (band) and -R_pf d_f, one segment at a time -----------------------
      for (int seg = 0; seg < K; ++seg) {
        const int32_t* cs = col + seg * N;
        const double* tp = tpow + seg * PW + (N - 1) + 1 - 2 * p.delta;
        for (int t = lane; t < N * N; t += kWarp) {
          const int r = t / N, s = t - r * N;
          const int cr = cs[r] - n_fixed, cc = cs[s] - n_fixed;
          if (cr >= 0 && cc >= 0 && cr >= cc) band[cc * N + (cr - cc)] += H1s[t] * tp[(r % h) + (s % h)];
        }
        for (int t = lane; t < N * D; t += kWarp) {
          const int r = t / D, dim = t - r * D;
          const int cr = cs[r] - n_fixed;
          if (cr >= 0) {
            double acc = 0.0;
            for (int s = 0; s < N; ++s) {
              const int c = cs[s];
              if (c < n_fixed) acc += H1s[r * N + s] * tp[(r % h) + (s % h)] * df[c * D + dim];
            }
            rhs[cr * D + dim] -= acc;
          }
        }
        __syncwarp();
      }

      // ---- a12: banded LDL^T with the forward substitution fused in ---------------------
      for (int j = 0; j < n_free; ++j) {
        const double d = band[j * N];
        const double inv = 1.0 / d;
        if (!(d > 0.0)) status |= 1;  // MINSNAP_STATUS_NONPOSITIVE_PIVOT
        const int nb = min(HB, n_free - 1 - j);
        __syncwarp();
        if (lane >= 1 && lane <= nb) {
          const double a = band[j * N + lane];
          acol[lane] = a;
          band[j * N + lane] = a * inv;
        }
        if (lane == 0) band[j * N] = inv;
        __syncwarp();
#pragma unroll
        for (int u = 0; u < NPASS; ++u) {
          const int pp = pair_p[u], qq = pair_q[u];
          if (pp <= nb) band[(j + qq) * N + (pp - qq)] -= band[j * N + pp] * acol[qq];
        }
        for (int t = lane; t < nb * D; t += kWarp) {
          const int pp = t / D + 1, dim = t - (pp - 1) * D;
          rhs[(j + pp) * D + dim] -= band[j * N + pp] * rhs[j * D + dim];
        }
        __syncwarp();
      }
      // y -> D^-1 y, then L^T x = z column by column
      for (int t = lane; t < n_free * D; t += kWarp) rhs[t] *= band[(t / D) * N];
      __syncwarp();
      for (int j = n_free - 1; j >= 1; --j) {
        const int nb = min(HB, j);
        for (int t = lane; t < nb * D; t += kWarp) {
          const int pp = t / D + 1, dim = t - (pp - 1) * D;
          rhs[(j - pp) * D + dim] -= band[(j - pp) * N + pp] * rhs[j * D + dim];
        }
        __syncwarp();
      }
      if (p.free_out)
        for (int t = lane; t < n_free * D; t += kWarp) p.free_out[b * (long)(n_free * D) + t] = rhs[t];
    } else {
      for (int t = lane; t < n_free * D; t += kWarp) rhs[t] = p.free_in[b * (long)(n_free * D) + t];
      __syncwarp();
    }

    // ---- a13 (+a16): coefficients, cost ---------------------------------------------------
    int nonfinite = 0;
    recover_coefficients<N, kGrad>(p, b, lane, H1s, A1s, col, tpow, df, rhs, nonfinite);
    if (nonfinite) status |= 4;
    status = __reduce_or_sync(0xffffffffu, status);
    if (p.status && lane == 0) p.status[b] = status;
    __syncwarp();
  }
}

template <int N, bool kSolve, bool kGrad = false>
static cudaError_t launch_general_n(const GeneralSolveArgs& a, cudaStream_t stream) {
  if (a.B == 0) return cudaSuccess;
  int warps = 8;
  while (warps > 1 && GeneralLayout<N>::cta_bytes(warps, a.K, a.D, a.n_fixed, a.n_free) > 100 * 1024) warps >>= 1;
  size_t smem = GeneralLayout<N>::cta_bytes(warps, a.K, a.D, a.n_fixed, a.n_free);
  if (smem > kMaxDynamicSmem) return cudaErrorInvalidConfiguration;
  auto kernel = solve_general_kernel<N, kSolve, kGrad>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  GeneralKernelParams p;
  p.B = a.B; p.K = a.K; p.D = a.D; p.delta = a.derivative; p.n_fixed = a.n_fixed; p.n_free = a.n_free;
  p.warps = warps;
  p.fixed_div = a.fixed_div > 0 ? a.fixed_div : 1;
  p.col_of_row = a.d_col_of_row; p.fixed_values = a.d_fixed_values; p.free_in = a.d_free_in;
  p.times = a.d_times; p.coeffs = a.d_coeffs; p.free_out = a.d_free_out; p.cost = a.d_cost;
  p.status = a.d_status;
  p.grad_free = a.d_grad_free; p.diag_free = a.d_diag_free;
  long grid = (a.B + warps - 1) / warps;
  const long max_grid = sm_count() * 32;
  if (grid > max_grid) grid = max_grid;
  kernel<<<(int)grid, warps * 32, smem, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_solve_general(const GeneralSolveArgs& a, cudaStream_t stream) {
  MINSNAP_DISPATCH_N(a.N, return (launch_general_n<kN, true>(a, stream)));
  return cudaSuccess;
}

cudaError_t general_fits(int N, int K, int D, int n_fixed, int n_free) {
  MINSNAP_DISPATCH_N(N, return GeneralLayout<kN>::cta_bytes(1, K, D, n_fixed, n_free) <= kMaxDynamicSmem
                                   ? cudaSuccess : cudaErrorInvalidConfiguration);
  return cudaSuccess;
}

cudaError_t launch_coeffs_from_constraints(const GeneralSolveArgs& a, cudaStream_t stream) {
  MINSNAP_DISPATCH_N(a.N, return (launch_general_n<kN, false>(a, stream)));
  return cudaSuccess;
}

cudaError_t launch_derivative_gradient(const GeneralSolveArgs& a, cudaStream_t stream) {
  if (!a.d_cost || (a.n_free > 0 && !a.d_grad_free)) return cudaErrorInvalidValue;
  MINSNAP_DISPATCH_N(a.N, return (launch_general_n<kN, false, true>(a, stream)));
  return cudaSuccess;
}

// The mask travels by value in the kernel's parameters, so that a caller can capture the whole call into a CUDA
// graph: a copy from pageable host memory cannot be captured.
__global__ void unpack_mask_kernel(MaskBits bits, int n, uint8_t* __restrict__ mask) {
  for (int i = threadIdx.x; i < n; i += blockDim.x) mask[i] = (bits.words[i >> 5] >> (i & 31)) & 1u;
}

cudaError_t launch_reorder_host_mask(int N, int K, const uint8_t* h_mask, uint8_t* d_mask, int32_t* d_col_of_row,
                                     int32_t* d_counts, cudaStream_t stream) {
  const int n = (K + 1) * (N / 2);
  if (n > 32 * MaskBits::kWords) return cudaErrorInvalidConfiguration;
  MaskBits bits = {};
  for (int i = 0; i < n; ++i)
    if (h_mask[i]) bits.words[i >> 5] |= 1u << (i & 31);
  unpack_mask_kernel<<<1, 256, 0, stream>>>(bits, n, d_mask);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  return launch_reorder(N, K, 1, d_mask, d_col_of_row, d_counts, stream);
}

// =========================================================================================
// a16 alone. computeCost from coefficients (ref: LIN.i:113-130): 0.5 sum_seg sum_dim c^T Q c.
// Warp per trajectory, lanes over (segment, dimension, row).
// =========================================================================================
template <int N>
__global__ void __launch_bounds__(256) cost_kernel(long B, int K, int D, int delta,
                                                   const double* __restrict__ coeffs,
                                                   const double* __restrict__ times, double* __restrict__ cost) {
  __shared__ double Q1[N * N];
  for (int e = threadIdx.x; e < N * N; e += blockDim.x) {
    const int r = e / N, c = e - r * N;
    double v = 0.0;
    if (r >= delta && c >= delta)
      v = 2.0 * falling_factorial(delta, r) * falling_factorial(delta, c) / (double)(r + c - 2 * delta + 1);
    Q1[e] = v;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long warp = blockIdx.x * (long)(blockDim.x >> 5) + uniform_warp_index();
  const long n_warps = ((long)gridDim.x * blockDim.x) >> 5;
  const int total = K * D * N;
  for (long b = warp; b < B; b += n_warps) {
    const double* cb = coeffs + b * (long)total;
    double acc = 0.0;
    for (int t = lane; t < total; t += kWarp) {
      const int r = t % N;
      const int seg = t / (N * D);
      if (r < delta) continue;
      const double T = times[b * K + seg];
      const double* c = cb + (t - r);
      // sum_s Q1[r][s] T^(r+s-2delta+1) c_s, Horner in T from the highest power down
      double row = 0.0;
      for (int s = N - 1; s >= delta; --s) row = row * T + Q1[r * N + s] * c[s];
      acc += c[r] * row * int_power(T, r - delta + 1);
    }
    acc = warp_sum(acc);
    if (lane == 0) cost[b] = 0.5 * acc;
  }
}

cudaError_t launch_cost(long B, int K, int D, int N, int derivative, const double* d_coeffs, const double* d_times,
                        double* d_cost, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const int block = 256;
  long grid = (B * 32 + block - 1) / block;
  if (grid > sm_count() * 16) grid = sm_count() * 16;
  MINSNAP_DISPATCH_N(N, (cost_kernel<kN><<<(int)grid, block, 0, stream>>>(B, K, D, derivative, d_coeffs, d_times, d_cost)));
  return cudaGetLastError();
}

// =========================================================================================
// SURVEY 8(f)2: numeric time gradient of the derivative cost (ref: getCostAndGradientTime,
// NL.i:2155-2243, with J_d = d^T R d from getCostAndGradientDerivative, NL.i:1452-1521).
// The reference moves ONE segment time by -/+ increment (a time <= 0.1 is set to 0.1 instead),
// rebuilds R and evaluates d^T R d with the end-point derivatives d of the last solve held
// fixed; only the moved segment's term q(T') = sum_dim d_seg^T H(T') d_seg changes, so
//   gradient[n] = w_d (q_n(T+) - q_n(T-)) / (2 increment) + w_t.
// One thread per (trajectory, segment): d_seg from the coefficients (derivatives at 0 and T),
// H(T') = H1 .* T'^(k_r + k_s + 1 - 2 delta) from the exact unit-time table.
// =========================================================================================
template <int N>
__global__ void __launch_bounds__(128) time_gradient_kernel(long B, int K, int D, int delta,
                                                            const double* __restrict__ coeffs,
                                                            const double* __restrict__ times, double increment,
                                                            double w_d, double w_t, double* __restrict__ gradient,
                                                            double* __restrict__ segment_cost) {
  constexpr int h = N / 2;
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * K) return;
  const double T = times[idx];
  const double T_minus = T <= 0.1 ? 0.1 : T - increment;
  const double T_plus = T <= 0.1 ? 0.1 : T + increment;
  // T'^(m + 1 - 2 delta) for m = k_r + k_s = 0 .. 2h-2
  double pw0[2 * h - 1], pwm[2 * h - 1], pwp[2 * h - 1];
#pragma unroll
  for (int m = 0; m < 2 * h - 1; ++m) {
    pw0[m] = int_power(T, m + 1 - 2 * delta);
    pwm[m] = int_power(T_minus, m + 1 - 2 * delta);
    pwp[m] = int_power(T_plus, m + 1 - 2 * delta);
  }
  const double* H1 = UnitTables<N>::h1(delta);
  double q0 = 0.0, qm = 0.0, qp = 0.0;
  for (int dim = 0; dim < D; ++dim) {
    const double* c = coeffs + (idx * D + dim) * N;
    double dv[N];
#pragma unroll
    for (int k = 0; k < h; ++k) {
      dv[k] = falling_factorial(k, k) * c[k];
      double r = falling_factorial(k, N - 1) * c[N - 1];
#pragma unroll
      for (int j = N - 2; j >= 0; --j)
        if (j >= k) r = fma(r, T, falling_factorial(k, j) * c[j]);
      dv[h + k] = r;
    }
#pragma unroll
    for (int r = 0; r < N; ++r) {
#pragma unroll
      for (int s = 0; s < N; ++s) {
        const int m = (r % h) + (s % h);
        const double term = dv[r] * dv[s] * H1[r * N + s];
        q0 = fma(term, pw0[m], q0);
        qm = fma(term, pwm[m], qm);
        qp = fma(term, pwp[m], qp);
      }
    }
  }
  if (gradient) gradient[idx] = w_d * ((qp - qm) / (2.0 * increment)) + w_t;
  if (segment_cost) segment_cost[idx] = q0;
}

cudaError_t launch_time_gradient(long B, int K, int D, int N, int derivative, const double* d_coeffs,
                                 const double* d_times, double increment, double w_d, double w_t, double* d_gradient,
                                 double* d_segment_cost, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const long n = B * K;
  const unsigned grid = (unsigned)((n + 127) / 128);
  MINSNAP_DISPATCH_N(N, (time_gradient_kernel<kN><<<grid, 128, 0, stream>>>(B, K, D, derivative, d_coeffs, d_times,
                                                                             increment, w_d, w_t, d_gradient,
                                                                             d_segment_cost)));
  return cudaGetLastError();
}

// objective[b][s] = cost[b][s] + time_penalty (sum_k times[b][s][k])^2  (ref objectiveFunctionTime,
// NL.i:778-784: cost_trajectory + total_time^2 * time_penalty)
// cost and objective may be the same array (minsnap_time_objective without a separate cost buffer): no __restrict__.
__global__ void __launch_bounds__(256) add_time_penalty_kernel(long n, int K, const double* __restrict__ times,
                                                               const double* cost, double time_penalty,
                                                               double* objective) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double total = 0.0;
  for (int k = 0; k < K; ++k) total += times[i * K + k];   // ref computeTotalTrajectoryTime: left to right
  objective[i] = cost[i] + total * total * time_penalty;
}

cudaError_t launch_add_time_penalty(long n, int K, const double* d_times, const double* d_cost, double time_penalty,
                                    double* d_objective, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  add_time_penalty_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(n, K, d_times, d_cost, time_penalty,
                                                                         d_objective);
  return cudaGetLastError();
}

// =========================================================================================
// SURVEY 8(f)2: the glue of a batched descent on the segment times, on the device.
// One optimiser iteration = solve (coefficients at the current times) -> time gradient -> the kernel below
// (step ladder: n_steps candidate allocations per trajectory along its own gradient) -> cost sweep over the
// candidates -> select kernel (penalty, first minimum, accept only an improvement): 5 launches, no host
// round trip, no temporaries beyond the workspace.
// =========================================================================================
// cand[b][s][k] = max(min_time, T_k - (max_relative_step / 2^s) scale_b g_k),  g = dJ/dT + 2 penalty sum(T),
// scale_b = min_k T_k / |g_k| (the step that would zero a segment time).
__global__ void __launch_bounds__(128) time_candidates_kernel(long B, int S, int K, const double* __restrict__ times,
                                                              const double* __restrict__ grad_cost, double time_penalty,
                                                              double max_relative_step, double min_time,
                                                              double* __restrict__ cand) {
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * S) return;
  const long b = idx / S;
  const int s = (int)(idx - b * S);
  const double* T = times + b * K;
  const double* gc = grad_cost + b * K;
  double total = 0.0;
  for (int k = 0; k < K; ++k) total += T[k];
  const double gp = 2.0 * time_penalty * total;
  double scale = 0.0;
  for (int k = 0; k < K; ++k) {
    const double g = fabs(gc[k] + gp);
    const double r = T[k] / (g < 1e-300 ? 1e-300 : g);
    scale = k == 0 ? r : fmin(scale, r);
  }
  double ladder = max_relative_step;
  for (int q = 0; q < s; ++q) ladder *= 0.5;
  double* out = cand + idx * K;
  for (int k = 0; k < K; ++k) {
    const double v = T[k] - (ladder * scale) * (gc[k] + gp);
    out[k] = v < min_time ? min_time : v;
  }
}

// objective[b][s] = cost[b][s] + penalty (sum_k cand[b][s][k])^2; the first minimum over s replaces the
// incumbent (times, objective) only when it is strictly smaller.  history_row (optional) receives the incumbent.
__global__ void __launch_bounds__(128) time_select_kernel(long B, int S, int K, const double* __restrict__ cand,
                                                          const double* __restrict__ cost, double time_penalty,
                                                          double* __restrict__ times, double* __restrict__ incumbent,
                                                          double* __restrict__ history_row) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double best = 0.0;
  int arg = -1;
  for (int s = 0; s < S; ++s) {
    const double* c = cand + (b * S + s) * K;
    double total = 0.0;
    for (int k = 0; k < K; ++k) total += c[k];
    const double obj = cost[b * S + s] + total * total * time_penalty;
    if (arg < 0 || obj < best) { best = obj; arg = s; }
  }
  double cur = incumbent[b];
  if (arg >= 0 && best < cur) {
    const double* c = cand + (b * S + arg) * K;
    for (int k = 0; k < K; ++k) times[b * K + k] = c[k];
    cur = best;
    incumbent[b] = cur;
  }
  if (history_row) history_row[b] = cur;
}

cudaError_t launch_time_candidates(long B, int S, int K, const double* d_times, const double* d_grad_cost,
                                   double time_penalty, double max_relative_step, double min_time, double* d_cand,
                                   cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const long n = B * S;
  time_candidates_kernel<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(B, S, K, d_times, d_grad_cost, time_penalty,
                                                                         max_relative_step, min_time, d_cand);
  return cudaGetLastError();
}

cudaError_t launch_time_select(long B, int S, int K, const double* d_cand, const double* d_cost, double time_penalty,
                               double* d_times, double* d_incumbent, double* d_history_row, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  time_select_kernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(B, S, K, d_cand, d_cost, time_penalty, d_times,
                                                                     d_incumbent, d_history_row);
  return cudaGetLastError();
}

// =========================================================================================
// The glue of the batched descent on the free derivatives (and optionally the segment times) against
// J = w_d J_d + w_c J_c + w_t sum(T), on the device.  See minsnap_optimize_free_constraints.
// =========================================================================================
// cand_free[b][s][j] = d_p[b][j] - 2^-s (w_d g_d[b][j] + w_c g_c[b][j]) / (2 w_d diag[b][j / D]): a Jacobi-scaled
// step, in the units of each free derivative.  Every operation is rounded on its own (no contraction), the sequence
// an elementwise torch version of the step performs.  cand_times (optional) [b][s] = times[b]: the times stay.
// kSoft: the numerator is (w_d g_d + w_c g_c) + w_sc g_sc, with the soft cost's gradient g_sc.
template <bool kSoft>
__global__ void __launch_bounds__(256) free_candidates_kernel(long B, int S, int n_fd, int D, int K,
                                                              const double* __restrict__ free_values,
                                                              const double* __restrict__ grad_d,
                                                              const double* __restrict__ grad_c,
                                                              const double* __restrict__ diag, double w_d, double w_c,
                                                              const double* __restrict__ times,
                                                              double* __restrict__ cand_free,
                                                              double* __restrict__ cand_times,
                                                              const double* __restrict__ grad_sc, double w_sc) {
  const long n_free_total = B * S * n_fd;
  const long total = n_free_total + (cand_times ? B * S * K : 0);
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    if (idx < n_free_total) {
      const long bs = idx / n_fd;
      const int j = (int)(idx - bs * n_fd);
      const long b = bs / S;
      const int s = (int)(bs - b * S);
      const long g = b * n_fd + j;
      double num = __dadd_rn(__dmul_rn(w_d, grad_d[g]), __dmul_rn(w_c, grad_c[g]));
      if constexpr (kSoft) num = __dadd_rn(num, __dmul_rn(w_sc, grad_sc[g]));
      const double step = __ddiv_rn(num, __dmul_rn(2.0 * w_d, diag[b * (n_fd / D) + j / D]));
      cand_free[idx] = __dsub_rn(free_values[g], __dmul_rn(ldexp(1.0, -s), step));
    } else {
      const long i = idx - n_free_total;
      const long bs = i / K;
      cand_times[i] = times[(bs / S) * K + (i - bs * K)];
    }
  }
}

// objective[i] = w_d J_d + w_c J_c + w_t sum_k times[i][k], J_d = 2 computeCost (the sum left to right, as
// computeTotalTrajectoryTime).  Jd (optional) receives J_d.
__global__ void __launch_bounds__(256) free_combine_kernel(long n, int K, const double* __restrict__ cost,
                                                           const double* __restrict__ jc,
                                                           const double* __restrict__ times, double w_d, double w_c,
                                                           double w_t, double* __restrict__ objective,
                                                           double* __restrict__ jd) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  double total = 0.0;
  for (int k = 0; k < K; ++k) total += times[i * K + k];
  const double j_d = 2.0 * cost[i];
  objective[i] = w_d * j_d + w_c * jc[i] + w_t * total;
  if (jd) jd[i] = j_d;
}

// The first minimum over the finite candidate objectives replaces the incumbent (free values, times, collision
// flag, objective) only when it is strictly smaller; history_row (optional) receives the incumbent.
__global__ void __launch_bounds__(128) free_select_kernel(long B, int S, int n_fd, int K,
                                                          const double* __restrict__ cand_obj,
                                                          const double* __restrict__ cand_free,
                                                          const double* __restrict__ cand_times,
                                                          const int32_t* __restrict__ cand_hit,
                                                          double* __restrict__ free_values, double* __restrict__ times,
                                                          double* __restrict__ incumbent, int32_t* __restrict__ hit,
                                                          double* __restrict__ history_row) {
  const long b = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double best = 0.0;
  int arg = -1;
  for (int s = 0; s < S; ++s) {
    const double obj = cand_obj[b * S + s];
    if (isfinite(obj) && (arg < 0 || obj < best)) { best = obj; arg = s; }
  }
  double cur = incumbent[b];
  if (arg >= 0 && best < cur) {
    const long c = b * S + arg;
    for (int j = 0; j < n_fd; ++j) free_values[b * n_fd + j] = cand_free[c * n_fd + j];
    for (int k = 0; k < K; ++k) times[b * K + k] = cand_times[c * K + k];
    if (hit) hit[b] = cand_hit[c];
    cur = best;
    incumbent[b] = cur;
  }
  if (history_row) history_row[b] = cur;
}

cudaError_t launch_free_candidates(long B, int S, int n_free, int D, int K, const double* d_free, const double* d_grad_d,
                                   const double* d_grad_c, const double* d_diag, double w_d, double w_c,
                                   const double* d_times, double* d_cand_free, double* d_cand_times,
                                   cudaStream_t stream, const double* d_grad_sc, double w_sc) {
  const long total = B * S * ((long)n_free * D + (d_cand_times ? K : 0));
  if (total == 0) return cudaSuccess;
  long grid = (total + 255) / 256;
  if (grid > sm_count() * 32) grid = sm_count() * 32;
  if (d_grad_sc)
    free_candidates_kernel<true><<<(int)grid, 256, 0, stream>>>(B, S, n_free * D, D, K, d_free, d_grad_d, d_grad_c,
                                                                d_diag, w_d, w_c, d_times, d_cand_free, d_cand_times,
                                                                d_grad_sc, w_sc);
  else
    free_candidates_kernel<false><<<(int)grid, 256, 0, stream>>>(B, S, n_free * D, D, K, d_free, d_grad_d, d_grad_c,
                                                                 d_diag, w_d, w_c, d_times, d_cand_free, d_cand_times,
                                                                 nullptr, 0.0);
  return cudaGetLastError();
}

// objective[i] += w_sc soft[i], rounded on its own: the soft term is added last
__global__ void __launch_bounds__(256) free_soft_add_kernel(long n, const double* __restrict__ soft, double w_sc,
                                                            double* __restrict__ objective) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  objective[i] = __dadd_rn(objective[i], __dmul_rn(w_sc, soft[i]));
}

cudaError_t launch_free_soft_add(long n, const double* d_soft, double w_sc, double* d_objective, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  free_soft_add_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(n, d_soft, w_sc, d_objective);
  return cudaGetLastError();
}

cudaError_t launch_free_combine(long n, int K, const double* d_cost, const double* d_jc, const double* d_times,
                                double w_d, double w_c, double w_t, double* d_objective, double* d_jd,
                                cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  free_combine_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(n, K, d_cost, d_jc, d_times, w_d, w_c, w_t,
                                                                       d_objective, d_jd);
  return cudaGetLastError();
}

cudaError_t launch_free_select(long B, int S, int n_fd, int K, const double* d_cand_obj, const double* d_cand_free,
                               const double* d_cand_times, const int32_t* d_cand_hit, double* d_free, double* d_times,
                               double* d_incumbent, int32_t* d_hit, double* d_history_row, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  free_select_kernel<<<(unsigned)((B + 127) / 128), 128, 0, stream>>>(B, S, n_fd, K, d_cand_obj, d_cand_free,
                                                                     d_cand_times, d_cand_hit, d_free, d_times,
                                                                     d_incumbent, d_hit, d_history_row);
  return cudaGetLastError();
}

// =========================================================================================
// The glue of the batched time descent with the reference's soft limits on max |p^(k)|, on the device.  See
// minsnap_optimize_segment_times_soft.  The maximum is not a fixed quadratic form in the end-point derivatives, so
// its gradient re-solves the 2K allocations T -/+ h e_n of every trajectory; they and the step ladder's candidates
// go through minsnap_solve_standard, which takes one row of positions per allocation.
// =========================================================================================
// out_p[i] = positions[i / R], out_e[i] = end[i / R] for i < B R (rows of row_p / row_e doubles)
__global__ void __launch_bounds__(256) replicate_rows_kernel(long B, int R, int row_p,
                                                             const double* __restrict__ positions,
                                                             double* __restrict__ out_p, int row_e,
                                                             const double* __restrict__ end,
                                                             double* __restrict__ out_e) {
  const long n_p = B * R * row_p;
  const long total = n_p + B * R * row_e;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    if (idx < n_p) {
      const long i = idx / row_p;
      out_p[idx] = positions[(i / R) * row_p + (idx - i * row_p)];
    } else {
      const long j = idx - n_p;
      const long i = j / row_e;
      out_e[j] = end[(i / R) * row_e + (j - i * row_e)];
    }
  }
}

// cand[(b K + n) 2 + j][k] = times[b][k], except k = n: T_n - increment (j = 0) or T_n + increment (j = 1), and
// 0.1 on both sides when T_n <= 0.1 (the clamp of getCostAndGradientTime, NL.i:2186-2187, 2207-2208).
__global__ void __launch_bounds__(256) soft_gradient_candidates_kernel(long B, int K, const double* __restrict__ times,
                                                                       double increment, double* __restrict__ cand) {
  const long total = B * K * 2 * K;
  for (long idx = (long)blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += (long)gridDim.x * blockDim.x) {
    const long row = idx / K;
    const int k = (int)(idx - row * K);
    const int j = (int)(row & 1);
    const long bn = row >> 1;
    const long b = bn / K;
    const int n = (int)(bn - b * K);
    const double T = times[b * K + k];
    double v = T;
    if (k == n) v = T <= 0.1 ? 0.1 : (j == 0 ? T - increment : T + increment);
    cand[idx] = v;
  }
}

__global__ void __launch_bounds__(256) soft_gradient_add_kernel(long n, const double* __restrict__ soft,
                                                                double increment, double* __restrict__ gradient) {
  const long i = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  gradient[i] = __dadd_rn(gradient[i], __ddiv_rn(__dsub_rn(soft[2 * i + 1], soft[2 * i]), 2.0 * increment));
}

static long glue_grid(long total) {
  long grid = (total + 255) / 256;
  if (grid > sm_count() * 32) grid = sm_count() * 32;
  return grid;
}

cudaError_t launch_replicate_rows(long B, int R, int row_p, const double* d_positions, double* d_out_p, int row_e,
                                  const double* d_end, double* d_out_e, cudaStream_t stream) {
  if (!d_end) row_e = 0;
  const long total = B * R * (long)(row_p + row_e);
  if (total == 0) return cudaSuccess;
  replicate_rows_kernel<<<(int)glue_grid(total), 256, 0, stream>>>(B, R, row_p, d_positions, d_out_p, row_e, d_end,
                                                                    d_out_e);
  return cudaGetLastError();
}

cudaError_t launch_soft_gradient_candidates(long B, int K, const double* d_times, double increment, double* d_cand,
                                            cudaStream_t stream) {
  const long total = B * K * 2 * K;
  if (total == 0) return cudaSuccess;
  soft_gradient_candidates_kernel<<<(int)glue_grid(total), 256, 0, stream>>>(B, K, d_times, increment, d_cand);
  return cudaGetLastError();
}

cudaError_t launch_soft_gradient_add(long B, int K, const double* d_soft, double increment, double* d_gradient,
                                     cudaStream_t stream) {
  const long n = B * K;
  if (n == 0) return cudaSuccess;
  soft_gradient_add_kernel<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>(n, d_soft, increment, d_gradient);
  return cudaGetLastError();
}

}  // namespace minsnap
