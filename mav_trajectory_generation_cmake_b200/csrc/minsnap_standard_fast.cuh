// Fast route for the standard mask (N = 10, snap): a THREAD PAIR per trajectory.
//
// Algebra (SURVEY.md section 8, notes A and B).  Unknowns are the free derivatives k = 1..4 at
// the interior vertices v = 1..K-1 (x_v in R^4 per dimension); R_pp is symmetric block
// tridiagonal with 4x4 blocks:
//     SE_{v-1}^T x_{v-1} + D_v x_v + SE_v x_{v+1} = b_v ,  x_0, x_K known (end derivatives)
//     D_v  = EE_{v-1} + SS_v          SS/EE/SE = start-free / end-free blocks of H_T
//     b_v  = -(ge_{v-1} dp_{v-1} + gs_v dp_v)   dp_i = p_{i+1} - p_i  (H annihilates constants,
//                                               so H[:,start pos] = -H[:,end pos])
// with H_T[r][s] = H1[r][s] T^(k_r + k_s - 7) taken from the exact unit-time table.
//
// Parallel scheme ("burn at both ends"): lane 2q eliminates the chain top-down from vertex 1,
// lane 2q+1 bottom-up from vertex K-1; they meet at the middle block, exchange their Schur
// contributions with one shuffle, solve the middle block (both lanes, identical arithmetic),
// then back-substitute outwards.  Time reversal maps derivative k to (-1)^k times itself and
// leaves the unit table invariant, so the bottom-up lane runs the SAME program on reversed
// inputs ("local coordinates") and flips the signs of odd derivatives when it leaves them.
// Each lane recovers the coefficients (ref: updateSegmentsFromCompactConstraints,
// LIN.i:252-273) of its half of the segments as soon as both end-point derivative vectors of a
// segment are known, through  c_i = T^-i sum_r A1inv[i][r] T^(k_r) d_r .
//
// Per block, per lane:  S^-1 explicitly through the 2x2 Schur blocks of the 4x4 SPD matrix (two
// reciprocals, shallow dependency depth), then Z = S^-1 SE and w = S^-1 g as mat-vec products
// (28 independent 4-FMA chains).  Z (16) and w -> x (4 D) of every eliminated block except the
// lane's last one (that stays in registers) live in shared memory as [slot][lane] rows of 256
// bytes (conflict-free); chains longer than kMaxK keep the same rows in a global scratch.
// Schur update S' = D' - SE^T Z, g' = b' - SE^T w;  back substitution x = w - Z x_next.
//
// HBM traffic is the algorithmic minimum: positions and times are read once (cp.async, all
// chunks in flight before the single wait), every polynomial is written once as 80 contiguous
// bytes with 16-byte streaming stores straight from registers.
#pragma once
#include <cuda_pipeline.h>

#include "minsnap_device.cuh"
#include "minsnap_launch.h"

namespace minsnap {
namespace fast {

constexpr int kN = 10;          // coefficients per polynomial
constexpr int kF = 4;           // free derivatives per interior vertex (k = 1..4)
constexpr int kPairsPerWarp = 16;
constexpr int kSlotStride = 32; // doubles between consecutive slots of one lane ([slot][lane])
constexpr int kBlockSlots = kF * kF;  // Z of one block
constexpr int kMaxK = 24;

#define H1T(r, s) (minsnap_tables::kH1_N10_d4[(r) * 10 + (s)])
#define A1T(i, r) (minsnap_tables::kA1inv_N10[(i) * 10 + (r)])
// 256-bit streaming store (PTX 8.8, sm_100+: STG.E.EF.ENL2.256); ptr must be 32-byte aligned.
__device__ __forceinline__ void store_cs_v4(double* ptr, double a, double b, double c, double d) {
  asm volatile("st.global.cs.v4.f64 [%0], {%1, %2, %3, %4};" ::"l"(ptr), "d"(a), "d"(b), "d"(c), "d"(d) : "memory");
}

// 1/x for a positive normal double: hardware seed (~20 bits) + two Newton steps.
__device__ __forceinline__ double fast_rcp(double x) {
  double r;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(x));
  double e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  e = fma(-x, r, 1.0);
  r = fma(r, e, r);
  return r;
}

// P[m] = T^(m-7) for m = 1..8 (P[0] unused).
struct TimePowers {
  double P[9];
  __device__ __forceinline__ void set(double T) {
    const double i1 = fast_rcp(T);
    const double i2 = i1 * i1;
    const double i3 = i2 * i1;
    const double i4 = i2 * i2;
    P[8] = T; P[7] = 1.0; P[6] = i1; P[5] = i2; P[4] = i3; P[3] = i4; P[2] = i4 * i1; P[1] = i3 * i3;
    P[0] = 0.0;
  }
};

// Lower triangle of a symmetric 4x4, packed row-wise: (0,0) (1,0) (1,1) (2,0) (2,1) (2,2) (3,0)...
__device__ __forceinline__ constexpr int tri(int a, int b) { return a * (a + 1) / 2 + b; }

// S = L D L^T.  On return l[tri(a,b)] (a > b) holds L, inv[a] = 1/D_a.  Returns false if a
// pivot is not positive.
__device__ __forceinline__ bool ldlt4(const double (&s)[10], double (&l)[10], double (&inv)[4]) {
  bool ok = true;
  const double d0 = s[tri(0, 0)];
  ok &= d0 > 0.0;
  inv[0] = fast_rcp(d0);
  l[tri(1, 0)] = s[tri(1, 0)] * inv[0];
  l[tri(2, 0)] = s[tri(2, 0)] * inv[0];
  l[tri(3, 0)] = s[tri(3, 0)] * inv[0];
  const double d1 = fma(-l[tri(1, 0)], s[tri(1, 0)], s[tri(1, 1)]);
  ok &= d1 > 0.0;
  inv[1] = fast_rcp(d1);
  const double t21 = fma(-l[tri(2, 0)], s[tri(1, 0)], s[tri(2, 1)]);
  const double t31 = fma(-l[tri(3, 0)], s[tri(1, 0)], s[tri(3, 1)]);
  l[tri(2, 1)] = t21 * inv[1];
  l[tri(3, 1)] = t31 * inv[1];
  const double d2 = fma(-l[tri(2, 1)], t21, fma(-l[tri(2, 0)], s[tri(2, 0)], s[tri(2, 2)]));
  ok &= d2 > 0.0;
  inv[2] = fast_rcp(d2);
  const double t32 = fma(-l[tri(3, 1)], t21, fma(-l[tri(3, 0)], s[tri(2, 0)], s[tri(3, 2)]));
  l[tri(3, 2)] = t32 * inv[2];
  const double d3 = fma(-l[tri(3, 2)], t32, fma(-l[tri(3, 1)], t31, fma(-l[tri(3, 0)], s[tri(3, 0)], s[tri(3, 3)])));
  ok &= d3 > 0.0;
  inv[3] = fast_rcp(d3);
  return ok;
}

// y <- S^-1 y with the factor above.
__device__ __forceinline__ void ldlt4_solve(const double (&l)[10], const double (&inv)[4], double (&y)[4]) {
  y[1] = fma(-l[tri(1, 0)], y[0], y[1]);
  y[2] = fma(-l[tri(2, 1)], y[1], fma(-l[tri(2, 0)], y[0], y[2]));
  y[3] = fma(-l[tri(3, 2)], y[2], fma(-l[tri(3, 1)], y[1], fma(-l[tri(3, 0)], y[0], y[3])));
  y[0] *= inv[0]; y[1] *= inv[1]; y[2] *= inv[2]; y[3] *= inv[3];
  y[2] = fma(-l[tri(3, 2)], y[3], y[2]);
  y[1] = fma(-l[tri(3, 1)], y[3], fma(-l[tri(2, 1)], y[2], y[1]));
  y[0] = fma(-l[tri(3, 0)], y[3], fma(-l[tri(2, 0)], y[2], fma(-l[tri(1, 0)], y[1], y[0])));
}

// Inverse of a symmetric positive definite 4x4 (packed lower triangles) through its 2x2 blocks:
//   S = [A B^T; B C],  Sigma = C - B A^-1 B^T,
//   S^-1 = [A^-1 + (B A^-1)^T Sigma^-1 (B A^-1),  -(B A^-1)^T Sigma^-1;  -Sigma^-1 B A^-1,  Sigma^-1].
// Two reciprocals and ~45 multiply-adds of depth ~12, against four serial pivots for L D L^T;
// the solves that follow become mat-vec products (independent 4-term chains).  Elimination
// without pivoting on an SPD matrix: the same subtractions L D L^T performs.  Returns false
// when a leading minor is not positive.
__device__ __forceinline__ bool spd4_inverse(const double (&s)[10], double (&si)[10]) {
  const double a00 = s[0], a10 = s[1], a11 = s[2];
  const double b00 = s[3], b01 = s[4], c00 = s[5];
  const double b10 = s[6], b11 = s[7], c10 = s[8], c11 = s[9];
  const double detA = fma(a00, a11, -(a10 * a10));
  bool ok = (a00 > 0.0) & (detA > 0.0);
  const double iA = fast_rcp(detA);
  const double A00 = a11 * iA, A10 = -a10 * iA, A11 = a00 * iA;
  const double BA00 = fma(b01, A10, b00 * A00), BA01 = fma(b01, A11, b00 * A10);
  const double BA10 = fma(b11, A10, b10 * A00), BA11 = fma(b11, A11, b10 * A10);
  const double g00 = fma(-BA01, b01, fma(-BA00, b00, c00));
  const double g10 = fma(-BA11, b01, fma(-BA10, b00, c10));
  const double g11 = fma(-BA11, b11, fma(-BA10, b10, c11));
  const double detG = fma(g00, g11, -(g10 * g10));
  ok &= (g00 > 0.0) & (detG > 0.0);
  const double iG = fast_rcp(detG);
  const double G00 = g11 * iG, G10 = -g10 * iG, G11 = g00 * iG;
  const double L00 = -fma(G10, BA10, G00 * BA00), L01 = -fma(G10, BA11, G00 * BA01);
  const double L10 = -fma(G11, BA10, G10 * BA00), L11 = -fma(G11, BA11, G10 * BA01);
  si[0] = fma(-BA10, L10, fma(-BA00, L00, A00));
  si[1] = fma(-BA11, L10, fma(-BA01, L00, A10));
  si[2] = fma(-BA11, L11, fma(-BA01, L01, A11));
  si[3] = L00; si[4] = L01; si[5] = G00;
  si[6] = L10; si[7] = L11; si[8] = G10; si[9] = G11;
  return ok;
}

// y = M x for a packed symmetric 4x4 M.
__device__ __forceinline__ void sym4_apply(const double (&m)[10], const double (&x)[4], double (&y)[4]) {
  y[0] = fma(m[6], x[3], fma(m[3], x[2], fma(m[1], x[1], m[0] * x[0])));
  y[1] = fma(m[7], x[3], fma(m[4], x[2], fma(m[2], x[1], m[1] * x[0])));
  y[2] = fma(m[8], x[3], fma(m[5], x[2], fma(m[4], x[1], m[3] * x[0])));
  y[3] = fma(m[9], x[3], fma(m[8], x[2], fma(m[7], x[1], m[6] * x[0])));
}

// Diagonal block D = EE(T_prev) + SS(T_next) in the coordinates of the lane (lower triangle).
__device__ __forceinline__ void diag_block(const TimePowers& prev, const TimePowers& next, double (&s)[10]) {
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int b = 0; b <= a; ++b) {
      const int m = a + b + 2;  // derivative orders (a+1) + (b+1)
      const double mix = ((a + b) & 1) ? next.P[m] - prev.P[m] : next.P[m] + prev.P[m];
      s[tri(a, b)] = H1T(a + 1, b + 1) * mix;
    }
}

// Coupling block SE(T)[a][b] = H1[a+1][6+b] T^(a+b+2-7).
__device__ __forceinline__ void coupling_block(const TimePowers& t, double (&e)[kF][kF]) {
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int b = 0; b < kF; ++b) e[a][b] = H1T(a + 1, 6 + b) * t.P[a + b + 2];
}

struct FastParams {
  long B;
  int K;
  const double* positions;
  const double* end_derivatives;
  const double* times;
  double v_max, a_max, magic;
  double* times_out;
  double* coeffs;
  double* free_out;
  double* cost;
  int32_t* status;
  int sweep_S;  // > 0: cost-only time sweep, times is [B][S][K]
  bool aligned16;  // positions / times pointers are 16-byte aligned (16-byte cp.async allowed)
  double* slot_scratch = nullptr;  // long chains: [warp][slot][lane] block storage in global memory
  // > 0 (headline kernel only): the problems are the chunks of longer trajectories, chunk_J per trajectory, and
  // `positions` is the trajectories' own array [B / chunk_J][chunk_J K + 1][D]: problem t reads its K + 1
  // vertices from vertex t K + t / chunk_J on (consecutive chunks share a vertex)
  int chunk_J = 0;
};

template <int D>
__host__ __device__ inline int lane_slots(int K) {
  const int mA = (K - 1) / 2;
  // The last eliminated block of a lane stays in registers; every other block stores Z (16)
  // and w/x (4 D).  During coefficient recovery the (dead) Z area holds three more vectors:
  // the boundary, the middle and the last block's x.
  const int stored = mA > 0 ? mA - 1 : 0;
  const int a = (kBlockSlots + kF * D) * stored;
  const int b = kF * D * stored + 3 * kF * D;
  return a > b ? a : b;
}

template <int D>
__host__ __device__ inline size_t warp_smem_doubles(int K, bool global_slots = false, bool direct = false) {
  // [slots][32] + positions [16][(K+1) D] + times [16][K]; every region a multiple of 16 bytes.
  // Long chains keep the slots in global memory (coalesced: one 256-byte row per slot).
  // Direct mode reads positions / times straight from global memory (no staging area).
  const size_t slots = global_slots ? 0 : ((size_t)lane_slots<D>(K) * kSlotStride + 1) & ~(size_t)1;
  if (direct) return slots;
  const size_t pos = ((size_t)kPairsPerWarp * (K + 1) * D + 1) & ~(size_t)1;
  const size_t tim = ((size_t)kPairsPerWarp * K + 1) & ~(size_t)1;
  return slots + pos + tim;
}

// Warp-cooperative asynchronous copy of n doubles, 16 bytes per cp.async when both pointers
// are 16-byte aligned.
__device__ __forceinline__ void async_copy_doubles(double* dst, const double* src, int n, int lane, bool aligned16) {
  if (aligned16) {
    const int n2 = n >> 1;
    for (int e = lane; e < n2; e += kWarp) __pipeline_memcpy_async(dst + 2 * e, src + 2 * e, 16);
    if ((n & 1) && lane == 0) __pipeline_memcpy_async(dst + n - 1, src + n - 1, 8);
  } else {
    for (int e = lane; e < n; e += kWarp) __pipeline_memcpy_async(dst + e, src + e, 8);
  }
}

// ------------------------------------------------------------------------------------------
// The kernel.  kCoeffs: recover and store coefficients; cost is computed when p.cost != NULL.
// ------------------------------------------------------------------------------------------
// kDirect: positions / times are read straight from global memory instead of being staged in
// shared memory.  Measured on B200: the cost sweep (64 time allocations share one set of
// positions, so the loads broadcast) gains 22 % (394 -> 308 us); the coefficient kernel loses 4 %
// and stays staged.  Capping registers at 168 for 10-12 resident warps was measured too: the
// spills and lost ILP cost 27 % per warp, more than the extra warps return.
template <int D, bool kCoeffs, bool kGlobalSlots = false, bool kCost = true, bool kDirect = false>
__global__ void __launch_bounds__(128) solve_standard_pair_kernel(FastParams p) {
  extern __shared__ __align__(16) double smem[];
  const int lane = threadIdx.x & 31;
  const int warp = uniform_warp_index();
  const int warps_per_cta = blockDim.x >> 5;
  const int K = p.K;
  const int pos_stride = (K + 1) * D;
  const int time_stride = K;
  double* wbase = smem + (size_t)warp * warp_smem_doubles<D>(K, kGlobalSlots, kDirect);
  double* slots = kGlobalSlots ? p.slot_scratch + ((size_t)blockIdx.x * warps_per_cta + warp) *
                                                      ((size_t)lane_slots<D>(K) * kSlotStride)
                               : wbase;                                  // [n_slots][32]
  double* pos_s = kGlobalSlots ? wbase
                               : slots + (((size_t)lane_slots<D>(K) * kSlotStride + 1) & ~(size_t)1);   // [16][pos_stride]
  double* time_s = pos_s + (((size_t)kPairsPerWarp * pos_stride + 1) & ~(size_t)1);      // [16][time_stride]

  const int side = lane & 1;   // 0: top-down lane, 1: bottom-up lane
  const int q = lane >> 1;     // pair index within the warp
  const int nb = K - 1;        // unknown blocks
  const int mA = nb / 2;       // blocks eliminated top-down; the middle block is vertex mA + 1
  const int nB = nb - mA - 1;  // blocks eliminated bottom-up
  const int my_n = side ? nB : mA;
  const int x_off = 0;                   // slot of w/x of block j (1-based): x_off + (j-1) * kF * D
  const int n_stored = mA > 0 ? mA - 1 : 0;   // blocks whose Z / w live in slots (the last one stays in registers)
  const int z_off = kF * D * n_stored;   // slot of Z of block j: z_off + (j-1) * 16
  const double flip[kF] = {side ? -1.0 : 1.0, 1.0, side ? -1.0 : 1.0, 1.0};  // (-1)^k, k = 1..4, for lane 1

  const long n_problems = p.sweep_S > 0 ? p.B * p.sweep_S : p.B;
  const long pairs_per_cta = (long)warps_per_cta * kPairsPerWarp;

  // Asynchronous global->shared input copies (cp.async): every chunk is in flight before the
  // first one is waited for.  Warps are persistent; the inputs of a warp's NEXT batch are
  // fetched while it recovers the coefficients of the current one, into the shared-memory
  // area of the (by then dead) Z blocks, so the DRAM latency is off the critical path.
  const int per_pos = (K + 1) * D;
  auto issue_inputs = [&](double* dst_pos, double* dst_time, long b0, int n) {
    if (p.sweep_S > 0) {
      for (int e = lane; e < n * per_pos; e += kWarp) {
        const int r = e / per_pos, o = e - r * per_pos;
        __pipeline_memcpy_async(dst_pos + e, p.positions + ((b0 + r) / p.sweep_S) * per_pos + o, 8);
      }
    } else {
      async_copy_doubles(dst_pos, p.positions + b0 * per_pos, n * per_pos, lane, p.aligned16);
    }
    if (p.times) async_copy_doubles(dst_time, p.times + b0 * K, n * K, lane, p.aligned16);
    __pipeline_commit();
  };
  const int pos_doubles = (kPairsPerWarp * per_pos + 1) & ~1;            // region sizes, even
  const int time_doubles = (kPairsPerWarp * K + 1) & ~1;
  // landing zone of the prefetch: the Z area minus its first 2*kF*D slots (those hold the
  // boundary / middle vectors during coefficient recovery)
  const int landing_slot = kF * D * n_stored + 3 * kF * D;
  double* landing = slots + (size_t)landing_slot * kSlotStride;
  const bool can_prefetch = !kGlobalSlots && !kDirect &&
                            (kBlockSlots * n_stored - 3 * kF * D) * kSlotStride >= pos_doubles + time_doubles &&
                            ((landing_slot * kSlotStride) & 1) == 0;
  const long stride = (long)gridDim.x * pairs_per_cta;
  const long first = (long)blockIdx.x * pairs_per_cta + (long)warp * kPairsPerWarp;
  bool landed = false;
  if (!kDirect && first < n_problems)
    issue_inputs(pos_s, time_s, first, (int)min((long)kPairsPerWarp, n_problems - first));

  for (long base = first; base < n_problems; base += stride) {
    const int n_here = (int)min((long)kPairsPerWarp, n_problems - base);
    const long next_base = base + stride;
    const int n_next = next_base < n_problems ? (int)min((long)kPairsPerWarp, n_problems - next_base) : 0;
    const long prob = base + q;          // problem of this pair
    const bool active = q < n_here;
    // ---- inputs of this batch ---------------------------------------------------------------
    if (!kDirect) {
      __pipeline_wait_prior(0);
      __syncwarp();
      if (landed) {
        for (int e = lane; e < n_here * per_pos; e += kWarp) pos_s[e] = landing[e];
        if (p.times)
          for (int e = lane; e < n_here * K; e += kWarp) time_s[e] = landing[pos_doubles + e];
        __syncwarp();
      }
      if (!p.times) {
        // ref estimateSegmentTimes (src/vertex.cpp:162-178), same expression as minsnap_estimate_segment_times
        for (int e = lane; e < n_here * K; e += kWarp) {
          const int r = e / K, o = e - r * K;
          const double* p0 = pos_s + r * pos_stride + o * D;
          double s2 = 0.0;
#pragma unroll
          for (int d = 0; d < D; ++d) {
            const double diff = p0[D + d] - p0[d];
            s2 += diff * diff;
          }
          const double distance = sqrt(s2);
          const double T = distance / p.v_max * 2 * (1.0 + p.magic * p.v_max / p.a_max * exp(-distance / p.v_max * 2));
          time_s[r * time_stride + o] = T;
          if (p.times_out) p.times_out[(base + r) * K + o] = T;
        }
        __syncwarp();
      }
    }

    // direct mode: idle lanes of a ragged last batch recompute the last problem (stores are masked)
    const long prob_in = active ? prob : n_problems - 1;
    const double* my_pos = kDirect ? p.positions + (p.sweep_S > 0 ? prob_in / p.sweep_S : prob_in) * per_pos
                                   : pos_s + q * pos_stride;
    const double* my_time = kDirect ? p.times + prob_in * K : time_s + q * time_stride;
    // local chain: vertex j <-> actual vertex (side ? K - j : j); segment j (between local
    // vertices j and j+1) <-> actual segment (side ? K-1-j : j)
    auto local_T = [&](int j) { return my_time[side ? K - 1 - j : j]; };
    auto local_p = [&](int j, int d) { return my_pos[(side ? K - j : j) * D + d]; };

    int status = 0;
    double* my_slots = slots + lane;     // slot s of this lane: my_slots[s * 33]

    // boundary derivatives of the local chain (vertex 0 of the lane), in local coordinates; read
    // on demand (zero when the caller passed no end derivatives) instead of living in registers
    const double* bd_src = nullptr;
    if (p.end_derivatives && active)
      bd_src = p.end_derivatives + ((p.sweep_S > 0 ? prob / p.sweep_S : prob) * 2 + side) * (kF * D);
    auto bd = [&](int a, int d) { return bd_src ? flip[a] * bd_src[a * D + d] : 0.0; };

    double xm[kF][D];   // middle block solution, local coordinates
    double Z[kF][kF], w[kF][D];   // after the forward sweep: the lane's LAST block, never written to slots
#pragma unroll
    for (int a = 0; a < kF; ++a) {
#pragma unroll
      for (int b = 0; b < kF; ++b) Z[a][b] = 0.0;
#pragma unroll
      for (int d = 0; d < D; ++d) w[a][d] = 0.0;
    }
    TimePowers tp_prev, tp_next;
    double dp_prev[D], dp_next[D];
    if (nb > 0) {
      // ---- forward sweep ------------------------------------------------------------------
      double S[10], g[kF][D];
      tp_prev.set(local_T(0));
      tp_next.set(local_T(1));
#pragma unroll
      for (int d = 0; d < D; ++d) {
        dp_prev[d] = local_p(1, d) - local_p(0, d);
        dp_next[d] = K >= 2 ? local_p(2, d) - local_p(1, d) : 0.0;
      }
      // block 1: D_1 and b_1 (with the known boundary derivatives moved to the right-hand side)
      auto rhs_block = [&](const TimePowers& tprev, const TimePowers& tnext, const double (&dprev)[D],
                           const double (&dnext)[D], double (&out)[kF][D]) {
#pragma unroll
        for (int a = 0; a < kF; ++a) {
          const double ce = H1T(6 + a, 5) * tprev.P[a + 1];   // ge: end-free row of the previous segment
          const double cs = H1T(1 + a, 5) * tnext.P[a + 1];   // gs: start-free row of the next segment
#pragma unroll
          for (int d = 0; d < D; ++d) out[a][d] = -fma(ce, dprev[d], cs * dnext[d]);
        }
      };
      diag_block(tp_prev, tp_next, S);
      rhs_block(tp_prev, tp_next, dp_prev, dp_next, g);
      if (bd_src) {
        double E0[kF][kF];
        coupling_block(tp_prev, E0);
#pragma unroll
        for (int b = 0; b < kF; ++b)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double acc = g[b][d];
#pragma unroll
            for (int a = 0; a < kF; ++a) acc = fma(-E0[a][b], bd(a, d), acc);
            g[b][d] = acc;
          }
      }

      for (int j = 1; j <= mA; ++j) {
        if (j <= my_n) {
          // here: tp_prev = segment j-1, tp_next = segment j, S/g = reduced block j
          double* zb = my_slots + (z_off + (j - 1) * kBlockSlots) * kSlotStride;
          double* wb = my_slots + (x_off + (j - 1) * kF * D) * kSlotStride;
          // inputs of block j+1 first: their shared-memory loads and the reciprocal chain of the
          // time powers overlap the arithmetic of block j (the compiler cannot hoist them over the
          // slot stores below on its own)
          const bool more = j < my_n;
          TimePowers tp_new;
          double dp_new[D];
          tp_new.set(local_T(more ? j + 1 : j));
#pragma unroll
          for (int d = 0; d < D; ++d) dp_new[d] = more ? local_p(j + 2, d) - local_p(j + 1, d) : 0.0;
          double Si[10];
          if (!spd4_inverse(S, Si)) status |= 1;
          double E[kF][kF];
          coupling_block(tp_next, E);
#pragma unroll
          for (int b = 0; b < kF; ++b) {
            const double in[4] = {E[0][b], E[1][b], E[2][b], E[3][b]};
            double col[4];
            sym4_apply(Si, in, col);
#pragma unroll
            for (int a = 0; a < kF; ++a) Z[a][b] = col[a];
          }
#pragma unroll
          for (int d = 0; d < D; ++d) {
            const double in[4] = {g[0][d], g[1][d], g[2][d], g[3][d]};
            double col[4];
            sym4_apply(Si, in, col);
#pragma unroll
            for (int a = 0; a < kF; ++a) w[a][d] = col[a];
          }
          if (j < my_n) {
#pragma unroll
            for (int a = 0; a < kF; ++a) {
#pragma unroll
              for (int b = 0; b < kF; ++b) zb[(a * kF + b) * kSlotStride] = Z[a][b];
#pragma unroll
              for (int d = 0; d < D; ++d) wb[(a * D + d) * kSlotStride] = w[a][d];
            }
            // advance to block j+1: D_{j+1} - E^T Z,  b_{j+1} - E^T w
            tp_prev = tp_next;
            tp_next = tp_new;
#pragma unroll
            for (int d = 0; d < D; ++d) {
              dp_prev[d] = dp_next[d];
              dp_next[d] = dp_new[d];
            }
            diag_block(tp_prev, tp_next, S);
            rhs_block(tp_prev, tp_next, dp_prev, dp_next, g);
#pragma unroll
            for (int a = 0; a < kF; ++a)
#pragma unroll
              for (int b = 0; b <= a; ++b) {
                double acc = S[tri(a, b)];
#pragma unroll
                for (int r = 0; r < kF; ++r) acc = fma(-E[r][a], Z[r][b], acc);
                S[tri(a, b)] = acc;
              }
#pragma unroll
            for (int a = 0; a < kF; ++a)
#pragma unroll
              for (int d = 0; d < D; ++d) {
                double acc = g[a][d];
#pragma unroll
                for (int r = 0; r < kF; ++r) acc = fma(-E[r][a], w[r][d], acc);
                g[a][d] = acc;
              }
          }
        }
      }

      // Schur contribution of this lane to the middle block, from its last eliminated block
      // (tp_next still holds the powers of the lane's last local segment): C = E^T Z, c = E^T w
      double C[10], c[kF][D];
#pragma unroll
      for (int i = 0; i < 10; ++i) C[i] = 0.0;
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) c[a][d] = 0.0;
      if (my_n >= 1) {
        double E[kF][kF];
        coupling_block(tp_next, E);
#pragma unroll
        for (int r = 0; r < kF; ++r)
#pragma unroll
          for (int a = 0; a < kF; ++a) {
#pragma unroll
            for (int b = 0; b <= a; ++b) C[tri(a, b)] = fma(E[r][a], Z[r][b], C[tri(a, b)]);
#pragma unroll
            for (int d = 0; d < D; ++d) c[a][d] = fma(E[r][a], w[r][d], c[a][d]);
          }
      }

      // ---- middle block, solved by both lanes in the coordinates of the top-down lane -------
      // own contribution -> top-down coordinates; a lane without blocks contributes the boundary
      // coupling instead (already part of b below), i.e. zeros here.
#pragma unroll
      for (int a = 0; a < kF; ++a) {
#pragma unroll
        for (int b = 0; b <= a; ++b)
          if ((a + b) & 1) C[tri(a, b)] = side ? -C[tri(a, b)] : C[tri(a, b)];
#pragma unroll
        for (int d = 0; d < D; ++d) c[a][d] *= flip[a];
      }
      double Sm[10], gm[kF][D];
      {
        const int m = mA + 1;                 // actual middle vertex
        const double Ta = my_time[m - 1], Tb = my_time[m];
        TimePowers ta, tb;
        ta.set(Ta);
        tb.set(Tb);
        double da[D], db[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
          da[d] = my_pos[m * D + d] - my_pos[(m - 1) * D + d];
          db[d] = my_pos[(m + 1) * D + d] - my_pos[m * D + d];
        }
        diag_block(ta, tb, Sm);
        rhs_block(ta, tb, da, db, gm);
        if (p.end_derivatives && active) {
          // boundary couplings that reach the middle block directly (K = 2, or K = 3 bottom side)
          const long rec = p.sweep_S > 0 ? prob / p.sweep_S : prob;
          if (m - 1 == 0) {
            const double* src = p.end_derivatives + (rec * 2 + 0) * (kF * D);
            double E0[kF][kF];
            coupling_block(ta, E0);
#pragma unroll
            for (int b = 0; b < kF; ++b)
#pragma unroll
              for (int d = 0; d < D; ++d)
#pragma unroll
                for (int a = 0; a < kF; ++a) gm[b][d] = fma(-E0[a][b], src[a * D + d], gm[b][d]);
          }
          if (m + 1 == K) {
            const double* src = p.end_derivatives + (rec * 2 + 1) * (kF * D);
            double E1[kF][kF];
            coupling_block(tb, E1);
#pragma unroll
            for (int a = 0; a < kF; ++a)
#pragma unroll
              for (int d = 0; d < D; ++d)
#pragma unroll
                for (int b = 0; b < kF; ++b) gm[a][d] = fma(-E1[a][b], src[b * D + d], gm[a][d]);
          }
        }
      }
      {
        // subtract the top-down contribution first, then the bottom-up one, on both lanes
#pragma unroll
        for (int i = 0; i < 10; ++i) {
          const double other = __shfl_xor_sync(0xffffffffu, C[i], 1);
          const double cA = side ? other : C[i];
          const double cB = side ? C[i] : other;
          Sm[i] = (Sm[i] - cA) - cB;
        }
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            const double other = __shfl_xor_sync(0xffffffffu, c[a][d], 1);
            const double cA = side ? other : c[a][d];
            const double cB = side ? c[a][d] : other;
            gm[a][d] = (gm[a][d] - cA) - cB;
          }
        double Si[10];
        if (!spd4_inverse(Sm, Si)) status |= 1;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const double in[4] = {gm[0][d], gm[1][d], gm[2][d], gm[3][d]};
          double col[4];
          sym4_apply(Si, in, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) xm[a][d] = flip[a] * col[a];   // -> local coordinates
        }
      }
      if (p.free_out && active && side == 0 && p.sweep_S == 0) {
        double* dst = p.free_out + (prob * (long)nb + mA) * (kF * D);
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) dst[a * D + d] = xm[a][d];
      }
    } else {
      // K == 1: no unknowns; the single segment has both ends fixed. Lane 0 recovers it with
      // the far end = the other boundary.
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) xm[a][d] = 0.0;
      if (p.end_derivatives && active) {
        const long rec = p.sweep_S > 0 ? prob / p.sweep_S : prob;
        const double* src = p.end_derivatives + (rec * 2 + 1) * (kF * D);
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) xm[a][d] = src[a * D + d];
      }
    }

    // ---- back substitution outwards: x_j = w_j - Z_j x_{j+1}, stored over w_j ----------------
    double xl[kF][D];   // x of the lane's last block (from the register copy of Z, w), local coordinates
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) xl[a][d] = 0.0;
    if (nb > 0) {
      double x_far[kF][D];
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) x_far[a][d] = xm[a][d];
      for (int j = mA; j >= 1; --j) {
        const int jj = side ? j - (mA - nB) : j;
        if (jj >= 1) {
          double x_near[kF][D];
          if (jj == my_n) {
            // the lane's last block: Z and w never left the registers
#pragma unroll
            for (int a = 0; a < kF; ++a)
#pragma unroll
              for (int d = 0; d < D; ++d) {
                double acc = w[a][d];
#pragma unroll
                for (int b = 0; b < kF; ++b) acc = fma(-Z[a][b], x_far[b][d], acc);
                x_near[a][d] = acc;
                xl[a][d] = acc;
              }
          } else {
            const double* zb = my_slots + (z_off + (jj - 1) * kBlockSlots) * kSlotStride;
            double* wb = my_slots + (x_off + (jj - 1) * kF * D) * kSlotStride;
#pragma unroll
            for (int a = 0; a < kF; ++a) {
              double zrow[kF];
#pragma unroll
              for (int b = 0; b < kF; ++b) zrow[b] = zb[(a * kF + b) * kSlotStride];
#pragma unroll
              for (int d = 0; d < D; ++d) {
                double acc = wb[(a * D + d) * kSlotStride];
#pragma unroll
                for (int b = 0; b < kF; ++b) acc = fma(-zrow[b], x_far[b][d], acc);
                x_near[a][d] = acc;
              }
            }
            // x is stored in ACTUAL coordinates (odd derivatives of the bottom-up lane flipped)
            // so that the recovery below reads start / end vectors without any sign logic
#pragma unroll
            for (int a = 0; a < kF; ++a)
#pragma unroll
              for (int d = 0; d < D; ++d) wb[(a * D + d) * kSlotStride] = flip[a] * x_near[a][d];
          }
#pragma unroll
          for (int a = 0; a < kF; ++a)
#pragma unroll
            for (int d = 0; d < D; ++d) x_far[a][d] = x_near[a][d];
          if (p.free_out && active && p.sweep_S == 0) {
            const int v = side ? K - jj : jj;    // actual vertex
            double* dst = p.free_out + (prob * (long)nb + (v - 1)) * (kF * D);
#pragma unroll
            for (int a = 0; a < kF; ++a)
#pragma unroll
              for (int d = 0; d < D; ++d) dst[a * D + d] = flip[a] * x_near[a][d];
          }
        }
      }
    }
    // boundary, middle and last-block vectors (actual coordinates) join the x's in three groups of
    // the now dead Z area, so every end-point vector is read the same way
    const int bd_slot = z_off, xm_slot = z_off + kF * D, xl_slot = z_off + 2 * kF * D;
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) {
        my_slots[(bd_slot + a * D + d) * kSlotStride] = bd_src ? bd_src[a * D + d] : 0.0;
        my_slots[(xm_slot + a * D + d) * kSlotStride] = flip[a] * xm[a][d];
        my_slots[(xl_slot + a * D + d) * kSlotStride] = flip[a] * xl[a][d];
      }
    __syncwarp();   // all Z blocks are dead from here on: their slots receive the next batch's inputs
    if (n_next > 0 && can_prefetch) {
      issue_inputs(landing, landing + pos_doubles, next_base, n_next);
      landed = true;
    }

    // ---- coefficient recovery / cost, one local segment per step ------------------------------
    // Local segment jj lies between local vertices jj (towards the boundary) and jj+1 (towards
    // the middle).  The top-down lane owns jj = mA..0, the bottom-up lane jj = nB..0 (its last
    // step is idle when nB < mA).
    double cost_acc = 0.0;
    int nonfinite = 0;
    const int top = nb > 0 ? mA : 0;
    const int n_steps = top + 1;
    for (int step = 0; step < n_steps; ++step) {
      const int j = top - step;
      const int jj = side ? j - (mA - nB) : j;
      const bool mine = active && jj >= 0 && (nb > 0 || side == 0);
      // end-point vectors of the segment in ACTUAL orientation (start = lower vertex index): the
      // vector of local vertex v lives at slot group  v == 0 ? boundary : v <= my_n ? x_v : middle
      const int jc = jj >= 0 ? jj : 0;
      //   v == 0 ? boundary : v < my_n ? x_v : v == my_n ? last block : middle
      const int near_slot = jc == 0 ? bd_slot : (jc < my_n ? x_off + (jc - 1) * kF * D : xl_slot);
      const int far_slot = jc + 1 < my_n ? x_off + jc * kF * D : (jc + 1 == my_n ? xl_slot : xm_slot);
      const double* start_ptr = my_slots + (side ? far_slot : near_slot) * kSlotStride;
      const double* end_ptr = my_slots + (side ? near_slot : far_slot) * kSlotStride;
      const int seg = side ? K - 1 - jc : jc;
      const double T = my_time[seg];
      if (!(T > 0.0)) status |= 2;   // MINSNAP_STATUS_BAD_TIME; the two lanes cover all K segments
      double u[2 * kF + 1][D];   // [dp, T^k start_k (k=1..4), T^k end_k (k=1..4)]
      double ds[kF][D];          // start derivatives (actual)
      {
        const double T2 = T * T, T3 = T2 * T, T4 = T2 * T2;
        const double tk[kF] = {T, T2, T3, T4};
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            const double s_val = start_ptr[(a * D + d) * kSlotStride];
            const double e_val = end_ptr[(a * D + d) * kSlotStride];
            ds[a][d] = s_val;
            u[1 + a][d] = tk[a] * s_val;
            u[1 + kF + a][d] = tk[a] * e_val;
          }
#pragma unroll
        for (int d = 0; d < D; ++d) u[0][d] = my_pos[(seg + 1) * D + d] - my_pos[seg * D + d];
      }
      const double i1 = fast_rcp(T);
      const double i2 = i1 * i1, i4 = i2 * i2, i5 = i4 * i1;
      if (kCoeffs) {
        const double ipow[5] = {i5, i5 * i1, i5 * i2, i4 * i4, i4 * i5};   // T^-5 .. T^-9
        // Row-outer, dimension-inner: the 9 table constants of an output row are live only while
        // they are applied to the D dimensions (short live ranges -> no constant-register hoarding).
        double cf[D][kN];
#pragma unroll
        for (int d = 0; d < D; ++d) cf[d][0] = my_pos[seg * D + d];
#pragma unroll
        for (int a = 0; a < kF; ++a) {
          const double ka = A1T(1 + a, 1 + a);
#pragma unroll
          for (int d = 0; d < D; ++d) cf[d][1 + a] = ka * ds[a][d];
        }
#pragma unroll
        for (int i = 5; i < kN; ++i) {
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double acc = A1T(i, 5) * u[0][d];
#pragma unroll
            for (int a = 0; a < kF; ++a) {
              acc = fma(A1T(i, 1 + a), u[1 + a][d], acc);
              acc = fma(A1T(i, 6 + a), u[1 + kF + a][d], acc);
            }
            cf[d][i] = acc * ipow[i - 5];
          }
        }
        // non-finite detection on the exponent fields of c_9 (scaled by T^-9: overflows first) and
        // c_4: integer tests instead of an FP64 reduction over all coefficients
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const int e9 = __double2hiint(cf[d][kN - 1]) & 0x7ff00000, e4 = __double2hiint(cf[d][kF]) & 0x7ff00000;
          if (e9 == 0x7ff00000 || e4 == 0x7ff00000) nonfinite = 1;
        }
        if (mine) {
          // the segment's D polynomials are 80 D contiguous, 16-byte aligned bytes of HBM
          double* dst = p.coeffs + (prob * K + seg) * (D * kN);
          if (p.aligned16) {
            // 32-byte stores (st.global.v4.f64, new with sm_100) on 32-byte boundaries, one 16-byte
            // store where the block starts or ends on a half sector: 8 store instructions per
            // 240-byte block instead of 15, and L2 receives whole sectors.  Measured: the per-lane
            // 16-byte stores (every lane in its own 128-byte line, half a sector each) were the
            // kernel's bottleneck -- 72 us with them, 41 us with the stores compiled out.
            constexpr int n = D * kN;
#define MINSNAP_CF(e) cf[(e) / kN][(e) % kN]
            if ((reinterpret_cast<uintptr_t>(dst) & 16) == 0) {
#pragma unroll
              for (int e = 0; e + 4 <= n; e += 4)
                store_cs_v4(dst + e, MINSNAP_CF(e), MINSNAP_CF(e + 1), MINSNAP_CF(e + 2), MINSNAP_CF(e + 3));
              if (n % 4 == 2)
                __stcs(reinterpret_cast<double2*>(dst + n - 2), make_double2(MINSNAP_CF(n - 2), MINSNAP_CF(n - 1)));
            } else {
              __stcs(reinterpret_cast<double2*>(dst), make_double2(MINSNAP_CF(0), MINSNAP_CF(1)));
#pragma unroll
              for (int e = 2; e + 4 <= n; e += 4)
                store_cs_v4(dst + e, MINSNAP_CF(e), MINSNAP_CF(e + 1), MINSNAP_CF(e + 2), MINSNAP_CF(e + 3));
              if ((n - 2) % 4 == 2)
                __stcs(reinterpret_cast<double2*>(dst + n - 2), make_double2(MINSNAP_CF(n - 2), MINSNAP_CF(n - 1)));
            }
#undef MINSNAP_CF
          } else {
#pragma unroll
            for (int d = 0; d < D; ++d)
#pragma unroll
              for (int i = 0; i < kN; ++i) __stcs(dst + d * kN + i, cf[d][i]);
          }
        }
      }
      if (kCost && p.cost && mine) {
        // u^T Hred1 u * T^-7: the per-segment quadratic form in scaled variables (SURVEY 8d), over the packed
        // lower triangle with doubled off-diagonal entries (tools/gen_tables.py): 54 multiply-adds per dimension
        const double i7 = i5 * i2;
        double qsum = 0.0;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          double qd = 0.0;
#pragma unroll
          for (int r = 0; r < 2 * kF + 1; ++r) {
            double row = minsnap_tables::kCostForm_N10_d4[tri(r, r)] * u[r][d];
#pragma unroll
            for (int s = 0; s < r; ++s) row = fma(minsnap_tables::kCostForm_N10_d4[tri(r, s)], u[s][d], row);
            qd = fma(row, u[r][d], qd);
          }
          qsum += qd;
        }
        cost_acc = fma(qsum, i7, cost_acc);
      }
    }

    if (kCost && p.cost) {
      cost_acc += __shfl_xor_sync(0xffffffffu, cost_acc, 1);
      if (active && side == 0) p.cost[prob] = 0.5 * cost_acc;
    }
    if (nonfinite) status |= 4;
    status |= __shfl_xor_sync(0xffffffffu, status, 1);
    if (p.status && active && side == 0) p.status[prob] = status;
    if (!kDirect && n_next > 0 && !can_prefetch) {
      __syncwarp();   // every lane is done with this batch's inputs
      issue_inputs(pos_s, time_s, next_base, n_next);
      landed = false;
    }
  }
}

#undef H1T
#undef A1T

// Chains up to kMaxK segments keep their block storage in shared memory; longer ones (config 4,
// K = 256) keep it in a global scratch and only stage the inputs in shared memory.
template <int D>
inline bool inputs_fit(int K) { return warp_smem_doubles<D>(K, true) * sizeof(double) <= kMaxDynamicSmem; }

inline bool supported(int K, int D, int N, int derivative) {
  if (!(N == 10 && derivative == 4 && K >= 1 && D >= 1 && D <= 3)) return false;
  if (K <= kMaxK) return true;
  return D == 1 ? inputs_fit<1>(K) : D == 2 ? inputs_fit<2>(K) : inputs_fit<3>(K);
}

template <int D, bool kCoeffs, bool kGlobalSlots, bool kDirect = false>
inline cudaError_t launch_mode(FastParams p, cudaStream_t stream) {
  const size_t per_warp = warp_smem_doubles<D>(p.K, kGlobalSlots, kDirect) * sizeof(double);
  // warps per CTA that maximise resident warps per SM (shared memory is the limiter; each CTA
  // also costs 1 KB of reserved shared memory)
  int warps = 1, best = 0;
  for (int w = 1; w <= 4; ++w) {
    const size_t cta = per_warp * w + 1024;
    if (per_warp * w > kMaxDynamicSmem) break;
    int resident = (int)((228 * 1024) / cta) * w;
    // 255 registers per thread: at most 8 warps per SM.  Measured on B200 (65,536 x K=10) with the 32-byte
    // coefficient stores: 6 warps 61.7 us, 7 warps 58.3 us, 8 warps 56.3 us; the cost-only kernel scales the same way.
    if (resident > 8) resident = 8;
    if (resident > best) { best = resident; warps = w; }
  }
  if (per_warp * warps > kMaxDynamicSmem) return cudaErrorInvalidConfiguration;
  const size_t smem = per_warp * warps;
  // the cost path is compiled out when no cost is requested (smaller hot loop, fewer registers)
  void (*kernel)(FastParams) = p.cost ? solve_standard_pair_kernel<D, kCoeffs, kGlobalSlots, true, kDirect>
                                      : solve_standard_pair_kernel<D, kCoeffs, kGlobalSlots, false, kDirect>;
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long n_problems = p.sweep_S > 0 ? p.B * p.sweep_S : p.B;
  const long per_cta = (long)warps * kPairsPerWarp;
  long grid = (n_problems + per_cta - 1) / per_cta;
  // One batch of 16 trajectories per warp while the grid stays modest: the hardware CTA scheduler
  // then balances the SMs dynamically (measured: a fixed persistent grid loses ~8% to the
  // 4.6-batches-per-slot tail at 65,536 problems).  Very large batches loop with prefetch.
  const long max_grid = sm_count() * 256;
  if (grid > max_grid) grid = max_grid;
  void* scratch = nullptr;
  if (kGlobalSlots) {
    const size_t bytes = (size_t)grid * warps * lane_slots<D>(p.K) * kSlotStride * sizeof(double);
    // keep the scratch in the device's stream-ordered pool between calls (no cudaMalloc per launch)
    int dev = 0;
    cudaMemPool_t pool;
    if (cudaGetDevice(&dev) == cudaSuccess && cudaDeviceGetDefaultMemPool(&pool, dev) == cudaSuccess) {
      uint64_t threshold = ~0ull;
      cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
    }
    if ((e = cudaMallocAsync(&scratch, bytes, stream)) != cudaSuccess) return e;
    p.slot_scratch = static_cast<double*>(scratch);
  }
  kernel<<<(int)grid, warps * 32, smem, stream>>>(p);
  e = cudaGetLastError();
  if (scratch) cudaFreeAsync(scratch, stream);
  return e;
}

template <int D, bool kCoeffs>
inline cudaError_t launch_d(const FastParams& p, cudaStream_t stream) {
  if (p.K <= kMaxK) {
    // direct reads for the cost sweep only (measured: see kDirect above)
    if (!kCoeffs && p.sweep_S > 0 && p.times) return launch_mode<D, kCoeffs, false, true>(p, stream);
    return launch_mode<D, kCoeffs, false>(p, stream);
  }
  return launch_mode<D, kCoeffs, true>(p, stream);
}

}  // namespace fast
}  // namespace minsnap
