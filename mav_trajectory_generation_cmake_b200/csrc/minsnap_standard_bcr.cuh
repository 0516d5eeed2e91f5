// Long chains of the standard mask (N = 10, snap; BASELINE config 4: K = 256): one CTA per
// trajectory, block cyclic reduction of the block-tridiagonal system in shared memory.
//
// Reference rows (SURVEY.md section 8a): the same chain as minsnap_standard_fast.cuh -- a9 (closed
// forms instead of A, A^-1, Q), a10 (standard mask), a11 + a12 (R_pp is block tridiagonal with 4x4
// blocks, one per interior vertex; ref LIN.i:297-369), a13 (coefficients, ref LIN.i:252-273).
//
// Why another kernel: the two-lane kernel eliminates the K-1 blocks of a trajectory one after the
// other from both ends -- 127 dependent block steps per lane at K = 256, and a batch of 4,096
// trajectories occupies 256 warps, fewer than two per SM: pure dependency latency (0.61 ms).
// Cyclic reduction eliminates every second block of the current chain at once:
//   level l (stride s = 2^l) eliminates the blocks i = s (2 m + 1); with n = i - s, m = i + s the
//   surviving neighbours and R_j the coupling A_{j, next(j)},
//     P_i = D_i^-1 R_i,  Q_i = D_i^-1 R_n^T,  y_i = D_i^-1 b_i
//     D_m -= R_i^T P_i,  b_m -= R_i^T y_i                       (right neighbour)
//     D_n -= R_n Q_i,    b_n -= R_n y_i,    R_n <- -R_n P_i     (left neighbour, now coupled to m)
//   and after the last level x_i = y_i - Q_i x_{i-s} - P_i x_{i+s} from the top level down.
// 8 levels instead of 127 steps for about 2.6x the arithmetic; Schur complements of an SPD
// matrix stay SPD, so no pivoting is needed (the same property the sequential sweep relies on).
// One thread owns one eliminated block per level and keeps R_i, P_i, Q_i, y_i in registers across
// the two update phases (right neighbours first, then left ones: every surviving block has at most
// one eliminated neighbour on each side, so each phase is free of write conflicts).
//
// Shared memory per trajectory: 44 doubles per block (Q over D, P over R, y/x over b), stored
// level-major so that the threads of a level touch consecutive words, plus the staged inputs:
// K = 256 -> 107 KB, two CTAs per SM.  Coefficients: one thread per segment, 32-byte stores.
// Measured per trajectory (clock64, K = 256, one CTA per SM): inputs 3.5 k cycles (now prefetched with
// cp.async during the previous trajectory), assembly 2.8 k, reduction 22.6 k (35.5 k before the
// read-modify-writes of a phase were split into loads / arithmetic / stores), back substitution
// 7.5 k, coefficients 5.7 k.
#pragma once
#include <cuda_pipeline.h>
#include <cuda_runtime.h>

#include "minsnap_device.cuh"
#include "minsnap_launch.h"
#include "minsnap_standard_fast.cuh"

namespace minsnap {
namespace bcr {

using fast::FastParams;
using fast::kF;
using fast::kN;
using fast::TimePowers;
using fast::tri;

#define H1T(r, s) (minsnap_tables::kH1_N10_d4[(r) * 10 + (s)])
#define A1T(i, r) (minsnap_tables::kA1inv_N10[(i) * 10 + (r)])

constexpr int kMaxThreads = 256;
constexpr int kMaxLevels = 10;

// record fields (field f of the block at position pos lives at rec[pos * record_stride + f])
constexpr int kFieldDQ = 0;    // 16: D (packed lower triangle, first 10) before elimination, Q after
constexpr int kFieldRP = 16;   // 16: R before elimination, P after
constexpr int kFieldBY = 32;   // 4 D: b, then y, then x
template <int D>
__host__ __device__ constexpr int record_doubles() { return 32 + kF * D; }
// Records are stored one after the other (field offsets become immediate operands of LDS / STS instead
// of a multiply per access) with an odd stride in doubles, so that the threads of a level, which
// touch consecutive records, fall in different banks (ncu on the [field][block] layout it replaces:
// 21 % of the executed instructions were IMAD address arithmetic; this layout executes 22 % fewer
// instructions).
template <int D>
__host__ __device__ constexpr int record_stride() { return record_doubles<D>() | 1; }

template <int D>
__host__ __device__ inline size_t smem_doubles(int K) {
  const size_t nb = K - 1;
  // records + two input buffers (the next trajectory's inputs arrive while this one is solved)
  return nb * record_stride<D>() + 2 * ((size_t)(K + 1) * D + K + 2 * kF * D);
}

struct Levels {
  int n_levels;
  int offset[kMaxLevels + 1];   // first position of level l
  int count[kMaxLevels];        // blocks eliminated at level l
};

__device__ __forceinline__ Levels make_levels(int nb) {
  Levels L;
  L.n_levels = 0;
  int off = 0;
  for (int l = 0; l < kMaxLevels; ++l) {
    const int s = 1 << l;
    const int c = nb >= s ? (nb - s) / (2 * s) + 1 : 0;
    L.offset[l] = off;
    L.count[l] = c;
    off += c;
    if (c > 0) L.n_levels = l + 1;
  }
  L.offset[kMaxLevels] = off;
  return L;
}

// storage position of block i (1-based): blocks of one level are consecutive
__device__ __forceinline__ int position(const Levels& L, int i) {
  const int l = __ffs(i) - 1;
  return L.offset[l] + (i >> (l + 1));
}

// Coefficients of one segment (a13: c = A^-1 d with A^-1_T[i][r] = A1inv[i][r] T^(k_r - i)) from the
// derivative vectors at its two vertices; the D polynomials leave as 32-byte stores on sector
// boundaries.  Returns true when a coefficient is not finite.
template <int D>
__device__ __forceinline__ bool recover_segment(const double* pos_seg, double T, const double (&ds)[kF][D],
                                                const double (&de)[kF][D], double* dst, bool aligned16) {
  bool nonfinite = false;
  const double T2 = T * T, T3 = T2 * T, T4 = T2 * T2;
  const double tk[kF] = {T, T2, T3, T4};
  const double i1 = fast::fast_rcp(T);
  const double i2 = i1 * i1, i4 = i2 * i2, i5 = i4 * i1;
  const double ipow[5] = {i5, i5 * i1, i5 * i2, i4 * i4, i4 * i5};   // T^-5 .. T^-9
  double cf[D][kN];
#pragma unroll
  for (int d = 0; d < D; ++d) {
    const double dp = pos_seg[D + d] - pos_seg[d];
    cf[d][0] = pos_seg[d];
#pragma unroll
    for (int a = 0; a < kF; ++a) cf[d][1 + a] = A1T(1 + a, 1 + a) * ds[a][d];
#pragma unroll
    for (int i = 5; i < kN; ++i) {
      double acc = A1T(i, 5) * dp;
#pragma unroll
      for (int a = 0; a < kF; ++a) {
        acc = fma(A1T(i, 1 + a), tk[a] * ds[a][d], acc);
        acc = fma(A1T(i, 6 + a), tk[a] * de[a][d], acc);
      }
      cf[d][i] = acc * ipow[i - 5];
    }
    const int e9 = __double2hiint(cf[d][kN - 1]) & 0x7ff00000, e4 = __double2hiint(cf[d][kF]) & 0x7ff00000;
    if (e9 == 0x7ff00000 || e4 == 0x7ff00000) nonfinite = true;
  }
  constexpr int nn = D * kN;
#define MINSNAP_CF(e) cf[(e) / kN][(e) % kN]
  if (aligned16) {
    if ((reinterpret_cast<uintptr_t>(dst) & 16) == 0) {
#pragma unroll
      for (int e = 0; e + 4 <= nn; e += 4)
        fast::store_cs_v4(dst + e, MINSNAP_CF(e), MINSNAP_CF(e + 1), MINSNAP_CF(e + 2), MINSNAP_CF(e + 3));
      if (nn % 4 == 2) __stcs(reinterpret_cast<double2*>(dst + nn - 2), make_double2(MINSNAP_CF(nn - 2), MINSNAP_CF(nn - 1)));
    } else {
      __stcs(reinterpret_cast<double2*>(dst), make_double2(MINSNAP_CF(0), MINSNAP_CF(1)));
#pragma unroll
      for (int e = 2; e + 4 <= nn; e += 4)
        fast::store_cs_v4(dst + e, MINSNAP_CF(e), MINSNAP_CF(e + 1), MINSNAP_CF(e + 2), MINSNAP_CF(e + 3));
      if ((nn - 2) % 4 == 2)
        __stcs(reinterpret_cast<double2*>(dst + nn - 2), make_double2(MINSNAP_CF(nn - 2), MINSNAP_CF(nn - 1)));
    }
  } else {
#pragma unroll
    for (int e = 0; e < nn; ++e) __stcs(dst + e, MINSNAP_CF(e));
  }
#undef MINSNAP_CF
  return nonfinite;
}

// Coefficient recovery as a pass of its own, one thread per (trajectory, segment), for the long-chain
// mode of the two-lane kernel: its lanes would otherwise walk the K segments one after the other
// (a third of the chain latency at K = 256).  free_values [B][K-1][kF][D] as the solve wrote them.
template <int D>
__global__ void __launch_bounds__(128) recover_standard_kernel(FastParams p, const double* __restrict__ free_values,
                                                               const double* __restrict__ times) {
  const int K = p.K, nb = K - 1;
  const long idx = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= p.B * K) return;
  const long b = idx / K;
  const int seg = (int)(idx - b * K);
  double ds[kF][D], de[kF][D];
  const double* bd = p.end_derivatives ? p.end_derivatives + b * 2L * kF * D : nullptr;
  const double* fv = free_values + b * (long)nb * kF * D;
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int d = 0; d < D; ++d) {
      ds[a][d] = seg >= 1 ? fv[((seg - 1) * kF + a) * D + d] : (bd ? bd[a * D + d] : 0.0);
      de[a][d] = seg + 1 <= nb ? fv[(seg * kF + a) * D + d] : (bd ? bd[kF * D + a * D + d] : 0.0);
    }
  const bool bad = recover_segment<D>(p.positions + (b * (K + 1) + seg) * D, times[idx], ds, de,
                                      p.coeffs + idx * (D * kN), p.aligned16);
  if (bad && p.status) atomicOr(p.status + b, 4);
}

template <int D>
__global__ void __launch_bounds__(kMaxThreads) solve_standard_bcr_kernel(FastParams p) {
  extern __shared__ __align__(16) double smem[];
  const int K = p.K, nb = K - 1;
  const int tid = threadIdx.x;
  constexpr int kStride = record_stride<D>();                // odd number of doubles: consecutive blocks fall in different banks
  double* rec = smem;                                        // [nb][kStride]: one record per block
  const int in_doubles = (K + 1) * D + K + 2 * kF * D;       // positions, times, boundary derivatives
  double* in_base = rec + (size_t)nb * kStride;              // [2][in_doubles]
  __shared__ Levels sL;
  __shared__ int s_status;
  if (tid == 0) sL = make_levels(nb);
  const Levels& L = sL;

  // cp.async staging of one trajectory's inputs into buffer `which`
  auto issue_inputs = [&](long b, int which) {
    double* dst = in_base + (size_t)which * in_doubles;
    const double* src_p = p.positions + b * (long)(K + 1) * D;
    for (int e = tid; e < (K + 1) * D; e += blockDim.x) __pipeline_memcpy_async(dst + e, src_p + e, 8);
    if (p.times) {
      const double* src_t = p.times + b * (long)K;
      for (int e = tid; e < K; e += blockDim.x) __pipeline_memcpy_async(dst + (K + 1) * D + e, src_t + e, 8);
    }
    if (p.end_derivatives) {
      const double* src_b = p.end_derivatives + b * 2L * kF * D;
      for (int e = tid; e < 2 * kF * D; e += blockDim.x) __pipeline_memcpy_async(dst + (K + 1) * D + K + e, src_b + e, 8);
    }
    __pipeline_commit();
  };
  int cur = 0;
  if ((long)blockIdx.x < p.B) issue_inputs(blockIdx.x, 0);

  for (long b = blockIdx.x; b < p.B; b += gridDim.x) {
    // ---- inputs --------------------------------------------------------------------------------
    __pipeline_wait_prior(0);
    if (tid == 0) s_status = 0;
    __syncthreads();
    if (b + gridDim.x < p.B) issue_inputs(b + gridDim.x, cur ^ 1);   // lands during this trajectory's solve
    double* pos_s = in_base + (size_t)cur * in_doubles;     // [K+1][D]
    double* time_s = pos_s + (K + 1) * D;                    // [K]
    double* bd_s = time_s + K;                               // [2][kF][D] boundary derivatives
    cur ^= 1;
    if (!p.end_derivatives)
      for (int e = tid; e < 2 * kF * D; e += blockDim.x) bd_s[e] = 0.0;
    int status = 0;
    for (int e = tid; e < K; e += blockDim.x) {
      double T;
      if (p.times) {
        T = time_s[e];
      } else {
        // ref estimateSegmentTimes (src/vertex.cpp:162-178), same expression as minsnap_estimate_segment_times
        double s2 = 0.0;
        for (int d = 0; d < D; ++d) {
          const double diff = pos_s[(e + 1) * D + d] - pos_s[e * D + d];
          s2 += diff * diff;
        }
        const double distance = sqrt(s2);
        T = distance / p.v_max * 2 * (1.0 + p.magic * p.v_max / p.a_max * exp(-distance / p.v_max * 2));
        if (p.times_out) p.times_out[b * (long)K + e] = T;
        time_s[e] = T;
      }
      if (!(T > 0.0)) status |= 2;
    }
    __syncthreads();

    // ---- assembly: D_i, R_i, b_i of every interior vertex i = 1..nb ------------------------------
    for (int i = 1 + tid; i <= nb; i += blockDim.x) {
      const int at = position(L, i);
      TimePowers tp_prev, tp_next;
      tp_prev.set(time_s[i - 1]);
      tp_next.set(time_s[i]);
      double S[10];
      fast::diag_block(tp_prev, tp_next, S);
#pragma unroll
      for (int e = 0; e < 10; ++e) rec[(at) * kStride + kFieldDQ + e] = S[e];
      double E[kF][kF];
      fast::coupling_block(tp_next, E);   // A_{(i,a),(i+1,b)}
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int c = 0; c < kF; ++c) rec[(at) * kStride + kFieldRP + a * kF + c] = E[a][c];
      double g[kF][D];
#pragma unroll
      for (int a = 0; a < kF; ++a) {
        const double ce = H1T(6 + a, 5) * tp_prev.P[a + 1];   // end-free row of the previous segment
        const double cs = H1T(1 + a, 5) * tp_next.P[a + 1];   // start-free row of the next segment
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const double dprev = pos_s[i * D + d] - pos_s[(i - 1) * D + d];
          const double dnext = pos_s[(i + 1) * D + d] - pos_s[i * D + d];
          g[a][d] = -fma(ce, dprev, cs * dnext);
        }
      }
      if (p.end_derivatives) {
        // known boundary derivatives move to the right-hand side of the first / last block
        if (i == 1) {
          double E0[kF][kF];
          fast::coupling_block(tp_prev, E0);   // A_{(0,a),(1,c)}
#pragma unroll
          for (int c = 0; c < kF; ++c)
#pragma unroll
            for (int d = 0; d < D; ++d) {
              double acc = g[c][d];
#pragma unroll
              for (int a = 0; a < kF; ++a) acc = fma(-E0[a][c], bd_s[a * D + d], acc);
              g[c][d] = acc;
            }
        }
        if (i == nb) {
#pragma unroll
          for (int a = 0; a < kF; ++a)
#pragma unroll
            for (int d = 0; d < D; ++d) {
              double acc = g[a][d];
#pragma unroll
              for (int c = 0; c < kF; ++c) acc = fma(-E[a][c], bd_s[kF * D + c * D + d], acc);
              g[a][d] = acc;
            }
        }
      }
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) rec[(at) * kStride + kFieldBY + a * D + d] = g[a][d];
    }
    __syncthreads();

    // ---- reduction ---------------------------------------------------------------------------------
    for (int l = 0; l < L.n_levels; ++l) {
      const int s = 1 << l;
      const bool work = tid < L.count[l];
      const int i = s * (2 * tid + 1);
      const int n = i - s, m = i + s;
      const bool has_n = work && n >= 1, has_m = work && m <= nb;
      const int at = work ? L.offset[l] + tid : 0;
      const int at_n = has_n ? position(L, n) : 0, at_m = has_m ? position(L, m) : 0;
      double R[kF][kF], P[kF][kF], Q[kF][kF], y[kF][D], Rn[kF][kF];
      if (work) {
        double S[10], Si[10];
#pragma unroll
        for (int e = 0; e < 10; ++e) S[e] = rec[(at) * kStride + kFieldDQ + e];
        if (!fast::spd4_inverse(S, Si)) status |= 1;
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int c = 0; c < kF; ++c) {
            R[a][c] = has_m ? rec[(at) * kStride + kFieldRP + a * kF + c] : 0.0;
            Rn[a][c] = has_n ? rec[(at_n) * kStride + kFieldRP + a * kF + c] : 0.0;
          }
#pragma unroll
        for (int c = 0; c < kF; ++c) {
          const double in_p[4] = {R[0][c], R[1][c], R[2][c], R[3][c]};
          const double in_q[4] = {Rn[c][0], Rn[c][1], Rn[c][2], Rn[c][3]};   // column c of R_n^T
          double col[4];
          fast::sym4_apply(Si, in_p, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) P[a][c] = col[a];
          fast::sym4_apply(Si, in_q, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) Q[a][c] = col[a];
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const double in[4] = {rec[(at) * kStride + kFieldBY + 0 * D + d], rec[(at) * kStride + kFieldBY + 1 * D + d],
                                rec[(at) * kStride + kFieldBY + 2 * D + d], rec[(at) * kStride + kFieldBY + 3 * D + d]};
          double col[4];
          fast::sym4_apply(Si, in, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) y[a][d] = col[a];
        }
      }
      // phase 1: right neighbours (D_m -= R_i^T P_i, b_m -= R_i^T y_i).  All loads first, all stores
      // last: interleaved read-modify-writes of the same shared array would be kept in program order.
      if (has_m) {
        double Dm[10], bm[kF][D];
#pragma unroll
        for (int e = 0; e < 10; ++e) Dm[e] = rec[(at_m) * kStride + kFieldDQ + e];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) bm[a][d] = rec[(at_m) * kStride + kFieldBY + a * D + d];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int c = 0; c <= a; ++c) {
            double acc = Dm[tri(a, c)];
#pragma unroll
            for (int r = 0; r < kF; ++r) acc = fma(-R[r][a], P[r][c], acc);
            Dm[tri(a, c)] = acc;
          }
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double acc = bm[a][d];
#pragma unroll
            for (int r = 0; r < kF; ++r) acc = fma(-R[r][a], y[r][d], acc);
            bm[a][d] = acc;
          }
#pragma unroll
        for (int e = 0; e < 10; ++e) rec[(at_m) * kStride + kFieldDQ + e] = Dm[e];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) rec[(at_m) * kStride + kFieldBY + a * D + d] = bm[a][d];
      }
      __syncthreads();
      // phase 2: left neighbours (D_n -= R_n Q_i, b_n -= R_n y_i, R_n <- -R_n P_i), then the block's own record
      if (has_n) {
        double Dn[10], bn[kF][D];
#pragma unroll
        for (int e = 0; e < 10; ++e) Dn[e] = rec[(at_n) * kStride + kFieldDQ + e];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) bn[a][d] = rec[(at_n) * kStride + kFieldBY + a * D + d];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int c = 0; c <= a; ++c) {
            double acc = Dn[tri(a, c)];
#pragma unroll
            for (int r = 0; r < kF; ++r) acc = fma(-Rn[a][r], Q[r][c], acc);
            Dn[tri(a, c)] = acc;
          }
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double acc = bn[a][d];
#pragma unroll
            for (int r = 0; r < kF; ++r) acc = fma(-Rn[a][r], y[r][d], acc);
            bn[a][d] = acc;
          }
        double Rnew[kF][kF];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int c = 0; c < kF; ++c) {
            double acc = 0.0;
#pragma unroll
            for (int r = 0; r < kF; ++r) acc = fma(-Rn[a][r], P[r][c], acc);
            Rnew[a][c] = has_m ? acc : 0.0;
          }
#pragma unroll
        for (int e = 0; e < 10; ++e) rec[(at_n) * kStride + kFieldDQ + e] = Dn[e];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) rec[(at_n) * kStride + kFieldBY + a * D + d] = bn[a][d];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int c = 0; c < kF; ++c) rec[(at_n) * kStride + kFieldRP + a * kF + c] = Rnew[a][c];
      }
      if (work) {
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int c = 0; c < kF; ++c) {
            rec[(at) * kStride + kFieldDQ + a * kF + c] = Q[a][c];
            rec[(at) * kStride + kFieldRP + a * kF + c] = P[a][c];
          }
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) rec[(at) * kStride + kFieldBY + a * D + d] = y[a][d];
      }
      __syncthreads();
    }

    // ---- back substitution, top level down: x_i = y_i - Q_i x_{i-s} - P_i x_{i+s} --------------------
    for (int l = L.n_levels - 2; l >= 0; --l) {
      const int s = 1 << l;
      if (tid < L.count[l]) {
        const int i = s * (2 * tid + 1);
        const int n = i - s, m = i + s;
        const int at = L.offset[l] + tid;
        double x[kF][D];
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) x[a][d] = rec[(at) * kStride + kFieldBY + a * D + d];
        if (n >= 1) {
          const int at_n = position(L, n);
          double xn[kF][D];
#pragma unroll
          for (int c = 0; c < kF; ++c)
#pragma unroll
            for (int d = 0; d < D; ++d) xn[c][d] = rec[(at_n) * kStride + kFieldBY + c * D + d];
#pragma unroll
          for (int a = 0; a < kF; ++a)
#pragma unroll
            for (int c = 0; c < kF; ++c) {
              const double q = rec[(at) * kStride + kFieldDQ + a * kF + c];
#pragma unroll
              for (int d = 0; d < D; ++d) x[a][d] = fma(-q, xn[c][d], x[a][d]);
            }
        }
        if (m <= nb) {
          const int at_m = position(L, m);
          double xm[kF][D];
#pragma unroll
          for (int c = 0; c < kF; ++c)
#pragma unroll
            for (int d = 0; d < D; ++d) xm[c][d] = rec[(at_m) * kStride + kFieldBY + c * D + d];
#pragma unroll
          for (int a = 0; a < kF; ++a)
#pragma unroll
            for (int c = 0; c < kF; ++c) {
              const double pp = rec[(at) * kStride + kFieldRP + a * kF + c];
#pragma unroll
              for (int d = 0; d < D; ++d) x[a][d] = fma(-pp, xm[c][d], x[a][d]);
            }
        }
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) rec[(at) * kStride + kFieldBY + a * D + d] = x[a][d];
      }
      __syncthreads();
    }

    // ---- free derivatives (optional) and coefficients: one thread per segment ----------------------
    if (p.free_out) {
      for (int e = tid; e < nb * kF * D; e += blockDim.x) {
        const int v = e / (kF * D) + 1, r = e % (kF * D);
        p.free_out[b * (long)nb * kF * D + e] = rec[(position(L, v)) * kStride + kFieldBY + r];
      }
    }
    int nonfinite = 0;
    for (int seg = tid; seg < K; seg += blockDim.x) {
      const double T = time_s[seg];
      double ds[kF][D], de[kF][D];
      {
        const int at_s = seg >= 1 ? position(L, seg) : 0, at_e = seg + 1 <= nb ? position(L, seg + 1) : 0;
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            ds[a][d] = seg >= 1 ? rec[(at_s) * kStride + kFieldBY + a * D + d] : bd_s[a * D + d];
            de[a][d] = seg + 1 <= nb ? rec[(at_e) * kStride + kFieldBY + a * D + d] : bd_s[kF * D + a * D + d];
          }
      }
      if (recover_segment<D>(pos_s + seg * D, T, ds, de, p.coeffs + (b * (long)K + seg) * (D * kN), p.aligned16))
        nonfinite = 1;
    }
    if (nonfinite) status |= 4;
    if (p.status) {
      if (status) atomicOr(&s_status, status);
      __syncthreads();
      if (tid == 0) p.status[b] = s_status;
    }
    __syncthreads();   // the records are rewritten by the next trajectory
  }
}

inline bool supported(int K, int D) {
  const int nb = K - 1;
  if (nb < 1 || (nb + 1) / 2 > kMaxThreads) return false;
  const size_t bytes = (D == 1 ? smem_doubles<1>(K) : D == 2 ? smem_doubles<2>(K) : smem_doubles<3>(K)) * sizeof(double);
  return bytes <= kMaxDynamicSmem;
}

template <int D>
inline cudaError_t launch_d(const FastParams& p, cudaStream_t stream) {
  const int nb = p.K - 1;
  int threads = (((nb + 1) / 2 + 31) / 32) * 32;
  if (threads < 64) threads = 64;
  const size_t smem = smem_doubles<D>(p.K) * sizeof(double);
  cudaError_t e = cudaFuncSetAttribute(solve_standard_bcr_kernel<D>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  // persistent CTAs, as many as are resident at once: each walks its trajectories with the next
  // one's inputs in flight (a CTA per trajectory would leave the cp.async prefetch nothing to fetch)
  const long resident = sm_count() * (kMaxDynamicSmem + 1024 >= 2 * (smem + 1024) ? 2 : 1);
  long grid = p.B < resident ? p.B : resident;
  solve_standard_bcr_kernel<D><<<(int)grid, threads, smem, stream>>>(p);
  return cudaGetLastError();
}

template <int D>
inline cudaError_t launch_recover(const FastParams& p, const double* free_values, const double* times, cudaStream_t stream) {
  const long n = p.B * p.K;
  recover_standard_kernel<D><<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(p, free_values, times);
  return cudaGetLastError();
}

#undef H1T
#undef A1T

}  // namespace bcr
}  // namespace minsnap
