// Long chains of the standard mask (N = 10, snap; BASELINE config 4: K = 256), partitioned: the chain is cut
// into J chunks of m segments at J - 1 separator vertices, and the work becomes three batch-parallel steps
// that each fill the machine, instead of one dependency chain of K - 1 block eliminations per trajectory.
//
// Reference rows (SURVEY.md section 8a): a9 (closed forms), a10 (standard mask), a11 + a12 (R_pp block tridiagonal,
// ref LIN.i:297-369), a13 (coefficients, ref LIN.i:252-273) -- the same system as minsnap_standard_fast.cuh:
//   E_{v-1}^T x_{v-1} + D_v x_v + E_v x_{v+1} = b_v      for the interior vertices v = 1 .. K-1.
//
//  1. chunk_schur_kernel: one THREAD per (chunk, side).  With L, R the chunk's end vertices, the side-0 thread
//     eliminates the chunk's interior blocks from L+1 up to R-1 carrying, next to the right-hand side, the four
//     columns that multiply the unknown x_L (the "spike"); nothing is stored -- what leaves is the chunk's Schur
//     complement on R:  E^T x_{R-1} = r_R + K x_L - C_RR x_R.  The side-1 thread runs the same program on the
//     reversed chunk (time reversal maps derivative k to (-1)^k and leaves the blocks invariant, as in the two-lane
//     kernel) without the spike and yields r_L, C_LL for L; the coupling of L to R is K^T by symmetry.
//  2. separator_solve_kernel: the J - 1 separators of a trajectory form a block-tridiagonal system again,
//       (D_s - C_RR[left chunk] - C_LL[right chunk]) y_j + K_{j-1} y_{j-1} + K_j^T y_{j+1} = b_s - r_R - r_L,
//     assembled by one thread per separator and solved by a thread pair per trajectory burning from both ends
//     (J/2 steps, the next block's values in flight during each).  It writes every chunk's two end-point
//     derivative vectors.
//  3. every chunk is now an independent standard problem of m segments with given end derivatives: the
//     headline kernel (minsnap_standard_tm.cuh) solves all B J of them in one launch, writing the coefficients
//     straight into [B][K][D][N] (a chunk's segments are contiguous there, as are its segment times).
//
// 4,096 x K = 256 (m = 8): 0.34 ms (cyclic reduction, one CTA per trajectory) -> see DESIGN.md section 4.5.
#pragma once
#include <cuda_runtime.h>

#include "minsnap_device.cuh"
#include "minsnap_launch.h"
#include "minsnap_standard_fast.cuh"
#include "minsnap_standard_tm.cuh"

namespace minsnap {
namespace chunked {

using fast::FastParams;
using fast::kF;
using fast::TimePowers;
using fast::tri;

#define H1T(r, s) (minsnap_tables::kH1_N10_d4[(r) * 10 + (s)])

// fields of the chunk records, stored [field][chunk j][trajectory b] (b fastest: both kernels coalesce)
template <int D>
struct Fields {
  static constexpr int kRR = 0;              // 10: C_RR, packed lower triangle
  static constexpr int kK = 10;              // 16: K[a][c], coefficient of x_L component c in row a of R's equation
  static constexpr int kRr = 26;             // 4 D: r_R
  static constexpr int kLL = 26 + kF * D;    // 10: C_LL
  static constexpr int kRl = 36 + kF * D;    // 4 D: r_L
  static constexpr int kCount = 36 + 2 * kF * D;
};

// chunk length: the headline kernel takes even K <= 12; the separator solve wants an odd number of separators
inline int chunk_segments(int K) {
  for (int m = 12; m >= 4; m -= 2)
    if (K % m == 0 && (K / m) % 2 == 0 && K / m >= 4) return m;
  return 0;
}
inline bool supported(int K, int D, int N, int derivative) {
  return N == 10 && derivative == 4 && D >= 1 && D <= 3 && K > fast::kMaxK && chunk_segments(K) > 0;
}

template <int D>
__device__ __forceinline__ void rhs_block(const TimePowers& tprev, const TimePowers& tnext, const double (&dprev)[D],
                                          const double (&dnext)[D], double (&out)[kF][D]) {
#pragma unroll
  for (int a = 0; a < kF; ++a) {
    const double ce = H1T(6 + a, 5) * tprev.P[a + 1];   // end-free row of the previous segment
    const double cs = H1T(1 + a, 5) * tnext.P[a + 1];   // start-free row of the next segment
#pragma unroll
    for (int d = 0; d < D; ++d) out[a][d] = -fma(ce, dprev[d], cs * dnext[d]);
  }
}

// ---- 1. Schur complement of every chunk on its two end vertices ------------------------------------------------
// grid.y = side.  Thread t of side s: trajectory b = t % B, chunk j = t / B.
template <int D>
__global__ void __launch_bounds__(128) chunk_schur_kernel(long B, int K, int m, const double* __restrict__ positions,
                                                          const double* __restrict__ times, double* __restrict__ rec,
                                                          int32_t* __restrict__ status) {
  const int J = K / m;
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * J) return;
  const int side = blockIdx.y;
  const long b = t % B;
  const int j = (int)(t / B);
  const double* tim = times + b * K + (long)j * m;                 // the chunk's m segment times
  const double* pos = positions + (b * (K + 1) + (long)j * m) * D;   // its m + 1 vertices
  // local chain: vertex i <-> actual (side ? m - i : i); segment i <-> actual (side ? m-1-i : i)
  auto local_T = [&](int i) { return __ldg(tim + (side ? m - 1 - i : i)); };
  auto local_p = [&](int i, int d) { return __ldg(pos + (side ? m - i : i) * D + d); };
  const int c = m - 1;   // interior blocks
  int bad = 0;

  TimePowers tp_prev, tp_next;
  double S[10], g[kF][D], V[kF][kF];
  double dp_prev[D], dp_next[D];
  {
    const double T0 = local_T(0), T1 = local_T(1);
    if (!(T0 > 0.0) || !(T1 > 0.0)) bad |= 2;
    tp_prev.set(T0);
    tp_next.set(T1);
  }
#pragma unroll
  for (int d = 0; d < D; ++d) {
    dp_prev[d] = local_p(1, d) - local_p(0, d);
    dp_next[d] = local_p(2, d) - local_p(1, d);
  }
  fast::diag_block(tp_prev, tp_next, S);
  rhs_block<D>(tp_prev, tp_next, dp_prev, dp_next, g);
  {
    // block 1's equation holds E_0^T x_0: as a right-hand side, the four columns -E_0^T
    double E0[kF][kF];
    fast::coupling_block(tp_prev, E0);
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int q = 0; q < kF; ++q) V[a][q] = -E0[q][a];
  }
  double CZ[10], cw[kF][D], CV[kF][kF];
  for (int i = 1; i <= c; ++i) {
    // here: tp_prev = segment i-1, tp_next = segment i, S / g / V = reduced block i
    const bool more = i < c;
    TimePowers tp_new;
    double dp_new[D];
    {
      const double Tn = local_T(more ? i + 1 : i);
      if (!(Tn > 0.0)) bad |= 2;
      tp_new.set(Tn);
    }
#pragma unroll
    for (int d = 0; d < D; ++d) dp_new[d] = more ? local_p(i + 2, d) - local_p(i + 1, d) : 0.0;
    double Si[10];
    if (!fast::spd4_inverse(S, Si)) bad |= 1;
    double E[kF][kF];
    fast::coupling_block(tp_next, E);
    // E^T S^-1 [E | g | V]: what block i hands to its right neighbour
    {
      double Z[kF][kF];
#pragma unroll
      for (int q = 0; q < kF; ++q) {
        const double in[4] = {E[0][q], E[1][q], E[2][q], E[3][q]};
        double col[4];
        fast::sym4_apply(Si, in, col);
#pragma unroll
        for (int a = 0; a < kF; ++a) Z[a][q] = col[a];
      }
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int q = 0; q <= a; ++q) {
          double acc = 0.0;
#pragma unroll
          for (int r = 0; r < kF; ++r) acc = fma(E[r][a], Z[r][q], acc);
          CZ[tri(a, q)] = acc;
        }
    }
    {
      double w[kF][D];
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const double in[4] = {g[0][d], g[1][d], g[2][d], g[3][d]};
        double col[4];
        fast::sym4_apply(Si, in, col);
#pragma unroll
        for (int a = 0; a < kF; ++a) w[a][d] = col[a];
      }
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) {
          double acc = 0.0;
#pragma unroll
          for (int r = 0; r < kF; ++r) acc = fma(E[r][a], w[r][d], acc);
          cw[a][d] = acc;
        }
    }
    if (side == 0) {
      double W[kF][kF];
#pragma unroll
      for (int q = 0; q < kF; ++q) {
        const double in[4] = {V[0][q], V[1][q], V[2][q], V[3][q]};
        double col[4];
        fast::sym4_apply(Si, in, col);
#pragma unroll
        for (int a = 0; a < kF; ++a) W[a][q] = col[a];
      }
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int q = 0; q < kF; ++q) {
          double acc = 0.0;
#pragma unroll
          for (int r = 0; r < kF; ++r) acc = fma(E[r][a], W[r][q], acc);
          CV[a][q] = acc;
        }
    }
    if (more) {
      tp_prev = tp_next;
      tp_next = tp_new;
#pragma unroll
      for (int d = 0; d < D; ++d) {
        dp_prev[d] = dp_next[d];
        dp_next[d] = dp_new[d];
      }
      fast::diag_block(tp_prev, tp_next, S);
      rhs_block<D>(tp_prev, tp_next, dp_prev, dp_next, g);
#pragma unroll
      for (int e = 0; e < 10; ++e) S[e] -= CZ[e];
#pragma unroll
      for (int a = 0; a < kF; ++a) {
#pragma unroll
        for (int d = 0; d < D; ++d) g[a][d] -= cw[a][d];
#pragma unroll
        for (int q = 0; q < kF; ++q) V[a][q] = -CV[a][q];
      }
    }
  }
  // results, in actual coordinates (the reversed side flips odd derivatives: k = a + 1)
  using F = Fields<D>;
  const long n_ch = B * J;
  double* out = rec + (long)j * B + b;
  if (side == 0) {
#pragma unroll
    for (int e = 0; e < 10; ++e) out[(F::kRR + e) * n_ch] = CZ[e];
#pragma unroll
    for (int a = 0; a < kF; ++a) {
#pragma unroll
      for (int q = 0; q < kF; ++q) out[(F::kK + a * kF + q) * n_ch] = CV[a][q];
#pragma unroll
      for (int d = 0; d < D; ++d) out[(F::kRr + a * D + d) * n_ch] = cw[a][d];
    }
  } else {
#pragma unroll
    for (int a = 0; a < kF; ++a) {
#pragma unroll
      for (int q = 0; q <= a; ++q) out[(F::kLL + tri(a, q)) * n_ch] = ((a + q) & 1) ? -CZ[tri(a, q)] : CZ[tri(a, q)];
#pragma unroll
      for (int d = 0; d < D; ++d) out[(F::kRl + a * D + d) * n_ch] = (a & 1) ? cw[a][d] : -cw[a][d];
    }
  }
  if (bad && status) atomicOr(status + b, bad);
}

// ---- 2a. the separator system, assembled for the lanes that will eliminate it -----------------------------------
// One thread per (trajectory, separator).  Separator j (1 .. J-1) in actual coordinates:
//   M = D_s - C_RR[chunk j-1] - C_LL[chunk j],   h = b_s - r_R[chunk j-1] - r_L[chunk j],   s = j m.
// The solve below burns the chain from both ends: the top-down lane owns separators 1 .. mA (local index i = j,
// coupling to the next one K_j^T), the bottom-up lane owns J-1 .. mA+2 (local index i = J - j, its own
// coordinates -- odd derivatives with the other sign -- and coupling flip K_{j-1} flip); the middle separator
// mA + 1 is kept in actual coordinates for both.  Records of kBlock doubles, [local index][entry][side][b].
template <int D>
struct SepLayout {
  static constexpr int kBlock = 10 + kF * D + kF * kF;   // M, h, coupling to the next separator
  static constexpr int kMid = 10 + kF * D;
};

// grid.y = part of the record a thread assembles (0: M, 1: h, 2: the coupling to the next separator and the couplings
// of the trajectory ends): the kernel is a gather of ~100 values per separator with next to no arithmetic, and one
// thread per (separator, part) keeps three times as many loads in flight as one thread per separator did.
template <int D>
__global__ void __launch_bounds__(128) assemble_separators_kernel(long B, int K, int m, const double* __restrict__ positions,
                                                                  const double* __restrict__ times,
                                                                  const double* __restrict__ rec,
                                                                  double* __restrict__ blocks,   // [mA][kBlock][2][B]
                                                                  double* __restrict__ edge,     // [16][2][B]: coupling of either trajectory end to its first separator
                                                                  double* __restrict__ middle) { // [kMid][B]
  using F = Fields<D>;
  using L = SepLayout<D>;
  const int J = K / m, ns = J - 1, mA = ns / 2;
  const long t = (long)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= B * ns) return;
  const int part = blockIdx.y;
  const long b = t % B;
  const int j = 1 + (int)(t / B);
  auto field = [&](int f, int chunk) { return __ldg(rec + ((long)f * J + chunk) * B + b); };
  const bool is_middle = j == mA + 1;
  const int side = j > mA + 1;
  const int i = side ? J - j : j;   // local index 1 .. mA
  double* out = blocks + ((long)(i - 1) * L::kBlock * 2 + side) * B + b;   // entry e at out[e 2 B]
  if (part < 2) {
    const int s = j * m;
    const double* tim = times + b * K;
    const double* pos = positions + b * (long)(K + 1) * D;
    TimePowers ta, tb;
    ta.set(__ldg(tim + s - 1));
    tb.set(__ldg(tim + s));
    if (part == 0) {
      double M[10];
      fast::diag_block(ta, tb, M);
#pragma unroll
      for (int e = 0; e < 10; ++e) M[e] = (M[e] - field(F::kRR + e, j - 1)) - field(F::kLL + e, j);
      if (is_middle) {
#pragma unroll
        for (int e = 0; e < 10; ++e) middle[(long)e * B + b] = M[e];
      } else {
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int q = 0; q <= a; ++q) out[(long)tri(a, q) * 2 * B] = (side && ((a + q) & 1)) ? -M[tri(a, q)] : M[tri(a, q)];
      }
    } else {
      double da[D], db[D], h[kF][D];
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const double p0 = __ldg(pos + s * D + d);
        da[d] = p0 - __ldg(pos + (s - 1) * D + d);
        db[d] = __ldg(pos + (s + 1) * D + d) - p0;
      }
      rhs_block<D>(ta, tb, da, db, h);
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d)
          h[a][d] = (h[a][d] - field(F::kRr + a * D + d, j - 1)) - field(F::kRl + a * D + d, j);
      if (is_middle) {
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) middle[(long)(10 + a * D + d) * B + b] = h[a][d];
      } else {
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) out[(long)(10 + a * D + d) * 2 * B] = (side && !(a & 1)) ? -h[a][d] : h[a][d];
      }
    }
    return;
  }
  if (!is_middle) {
    // coupling to the next local separator: top-down K_j^T (chunk j), bottom-up flip K_{j-1} flip (chunk j-1)
    const int chunk = side ? j - 1 : j;
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int q = 0; q < kF; ++q) {
        const double v = side ? (((a + q) & 1) ? -field(F::kK + a * kF + q, chunk) : field(F::kK + a * kF + q, chunk))
                              : field(F::kK + q * kF + a, chunk);
        out[(long)(10 + kF * D + a * kF + q) * 2 * B] = v;
      }
  }
  // the couplings of the two trajectory ends to their first separators (local form, as above with i = 0)
  if (j == 1 || j == ns) {
    for (int sd = (j == 1 ? 0 : 1); sd <= (j == ns ? 1 : 0); ++sd) {
      const int chunk = sd ? J - 1 : 0;
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int q = 0; q < kF; ++q) {
          const double v = sd ? (((a + q) & 1) ? -field(F::kK + a * kF + q, chunk) : field(F::kK + a * kF + q, chunk))
                              : field(F::kK + q * kF + a, chunk);
          edge[((long)(a * kF + q) * 2 + sd) * B + b] = v;
        }
    }
  }
}

// ---- 2b. thread pair per trajectory, burning the separator chain from both ends -------------------------------
// The blocks arrive assembled and in the lane's coordinates; the next block's 38 values are requested before the
// current one is eliminated, and the back substitution reads its stored blocks one step ahead likewise, so a step
// costs its arithmetic, not a round trip to L2.  Block storage of the lanes (Z and w of every eliminated
// separator but the last) lives in a global scratch, [warp][slot][entry][lane]: coalesced 256-byte rows.
template <int D>
__global__ void __launch_bounds__(32) separator_solve_kernel(long B, int K, int m, const double* __restrict__ boundary,   // [B][2][4][D] or null
                                                             const double* __restrict__ blocks, const double* __restrict__ edge,
                                                             const double* __restrict__ middle,
                                                             double* __restrict__ chunk_ends,       // [B J][2][4][D]
                                                             double* __restrict__ free_out,         // optional [B][K-1][4][D]
                                                             double* __restrict__ slots, int32_t* __restrict__ status) {
  using L = SepLayout<D>;
  constexpr int kVec = kF * D;
  constexpr int kSlot = kF * kF + kVec;
  const int J = K / m;
  const int ns = J - 1;            // separators (odd)
  const int mA = ns / 2;           // blocks eliminated by either lane (>= 1); the middle separator is mA + 1
  const int lane = threadIdx.x & 31;
  const int side = lane >> 4;
  const long b0 = (long)blockIdx.x * 16 + (lane & 15);
  const bool active = b0 < B;
  const long b = active ? b0 : 0;   // idle pairs of a ragged last warp run on trajectory 0 and write nothing
  const double flip[kF] = {side ? -1.0 : 1.0, 1.0, side ? -1.0 : 1.0, 1.0};
  int bad = 0;
  auto actual = [&](int i) { return side ? J - i : i; };   // local separator index -> actual

  const double* my_blocks = blocks + (long)side * B + b;   // entry e of local block i: my_blocks[((i-1) kBlock + e) 2 B]
  double nxt[L::kBlock];
  auto request = [&](int i) {
    const double* src = my_blocks + (long)(i - 1) * L::kBlock * 2 * B;
#pragma unroll
    for (int e = 0; e < L::kBlock; ++e) nxt[e] = __ldg(src + (long)e * 2 * B);
  };
  request(1);
  // the lane's end of the trajectory: known derivatives (actual coordinates), zero without a boundary array
  double xb[kF][D];
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int d = 0; d < D; ++d) xb[a][d] = boundary ? __ldg(boundary + (b * 2 + side) * kVec + a * D + d) : 0.0;
  double E[kF][kF];
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int q = 0; q < kF; ++q) E[a][q] = __ldg(edge + ((long)(a * kF + q) * 2 + side) * B + b);

  double* st = slots + (long)blockIdx.x * (mA > 1 ? mA - 1 : 0) * kSlot * 32 + lane;   // entry e of slot i: st[(i kSlot + e) 32]
  double Z[kF][kF], w[kF][D];
  double S[10], g[kF][D];
  // ---- forward sweep over local separators 1 .. mA ------------------------------------------
#pragma unroll
  for (int e = 0; e < 10; ++e) S[e] = nxt[e];
  // the known end vector moves to the right-hand side of the first separator
#pragma unroll
  for (int q = 0; q < kF; ++q)
#pragma unroll
    for (int d = 0; d < D; ++d) {
      double acc = nxt[10 + q * D + d];
#pragma unroll
      for (int a = 0; a < kF; ++a) acc = fma(-E[a][q], flip[a] * xb[a][d], acc);
      g[q][d] = acc;
    }
  for (int i = 1; i <= mA; ++i) {
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int q = 0; q < kF; ++q) E[a][q] = nxt[10 + kVec + a * kF + q];
    if (i < mA) request(i + 1);   // in flight during this block's elimination
    double Si[10];
    if (!fast::spd4_inverse(S, Si)) bad |= 1;
#pragma unroll
    for (int q = 0; q < kF; ++q) {
      const double in[4] = {E[0][q], E[1][q], E[2][q], E[3][q]};
      double col[4];
      fast::sym4_apply(Si, in, col);
#pragma unroll
      for (int a = 0; a < kF; ++a) Z[a][q] = col[a];
    }
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const double in[4] = {g[0][d], g[1][d], g[2][d], g[3][d]};
      double col[4];
      fast::sym4_apply(Si, in, col);
#pragma unroll
      for (int a = 0; a < kF; ++a) w[a][d] = col[a];
    }
    if (i < mA) {
      double* slot = st + (long)(i - 1) * kSlot * 32;
#pragma unroll
      for (int a = 0; a < kF; ++a) {
#pragma unroll
        for (int q = 0; q < kF; ++q) slot[(a * kF + q) * 32] = Z[a][q];
#pragma unroll
        for (int d = 0; d < D; ++d) slot[(kF * kF + a * D + d) * 32] = w[a][d];
      }
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int q = 0; q <= a; ++q) {
          double acc = nxt[tri(a, q)];
#pragma unroll
          for (int r = 0; r < kF; ++r) acc = fma(-E[r][a], Z[r][q], acc);
          S[tri(a, q)] = acc;
        }
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) {
          double acc = nxt[10 + a * D + d];
#pragma unroll
          for (int r = 0; r < kF; ++r) acc = fma(-E[r][a], w[r][d], acc);
          g[a][d] = acc;
        }
    }
  }
  // ---- middle separator, solved by both lanes in actual coordinates --------------------------
  double C[10], c[kF][D];
#pragma unroll
  for (int e = 0; e < 10; ++e) C[e] = 0.0;
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int d = 0; d < D; ++d) c[a][d] = 0.0;
  // E still couples the lane's last block to the middle one
#pragma unroll
  for (int r = 0; r < kF; ++r)
#pragma unroll
    for (int a = 0; a < kF; ++a) {
#pragma unroll
      for (int q = 0; q <= a; ++q) C[tri(a, q)] = fma(E[r][a], Z[r][q], C[tri(a, q)]);
#pragma unroll
      for (int d = 0; d < D; ++d) c[a][d] = fma(E[r][a], w[r][d], c[a][d]);
    }
#pragma unroll
  for (int a = 0; a < kF; ++a) {
#pragma unroll
    for (int q = 0; q <= a; ++q)
      if ((a + q) & 1) C[tri(a, q)] = side ? -C[tri(a, q)] : C[tri(a, q)];
#pragma unroll
    for (int d = 0; d < D; ++d) c[a][d] *= flip[a];
  }
  double xm[kF][D];   // the middle separator, then the far vector of each back-substitution step (local coordinates)
  {
    double Sm[10], gm[kF][D];
#pragma unroll
    for (int e = 0; e < 10; ++e) Sm[e] = __ldg(middle + (long)e * B + b);
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) gm[a][d] = __ldg(middle + (long)(10 + a * D + d) * B + b);
#pragma unroll
    for (int e = 0; e < 10; ++e) {
      const double other = __shfl_xor_sync(0xffffffffu, C[e], 16);
      const double cA = side ? other : C[e];
      const double cB = side ? C[e] : other;
      Sm[e] = (Sm[e] - cA) - cB;
    }
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const double other = __shfl_xor_sync(0xffffffffu, c[a][d], 16);
        const double cA = side ? other : c[a][d];
        const double cB = side ? c[a][d] : other;
        gm[a][d] = (gm[a][d] - cA) - cB;
      }
    double Si[10];
    if (!fast::spd4_inverse(Sm, Si)) bad |= 1;
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const double in[4] = {gm[0][d], gm[1][d], gm[2][d], gm[3][d]};
      double col[4];
      fast::sym4_apply(Si, in, col);
#pragma unroll
      for (int a = 0; a < kF; ++a) xm[a][d] = flip[a] * col[a];   // -> local coordinates
    }
  }
  // separator j's vector ends chunk j-1 (slot 1) and starts chunk j (slot 0), in actual coordinates
  auto emit = [&](int j, const double (&x)[kF][D]) {
    if (!active) return;
    double* e1 = chunk_ends + ((b * J + (j - 1)) * 2 + 1) * kVec;
    double* e0 = chunk_ends + ((b * J + j) * 2 + 0) * kVec;
    double* fo = free_out ? free_out + (b * (long)(K - 1) + ((long)j * m - 1)) * kVec : nullptr;
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const double v = flip[a] * x[a][d];
        e1[a * D + d] = v;
        e0[a * D + d] = v;
        if (fo) fo[a * D + d] = v;
      }
  };
  if (side == 0) emit(mA + 1, xm);
  // ---- back substitution outwards, the stored blocks read one step ahead ------------------------
  double Zn[kF][kF], wn[kF][D];
  auto fetch = [&](int i) {   // stored block of local separator i (i < mA)
    const double* slot = st + (long)(i - 1) * kSlot * 32;
#pragma unroll
    for (int a = 0; a < kF; ++a) {
#pragma unroll
      for (int q = 0; q < kF; ++q) Zn[a][q] = slot[(a * kF + q) * 32];
#pragma unroll
      for (int d = 0; d < D; ++d) wn[a][d] = slot[(kF * kF + a * D + d) * 32];
    }
  };
  if (mA >= 2) fetch(mA - 1);
  for (int i = mA; i >= 1; --i) {
    double x[kF][D];
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) {
        double acc = w[a][d];
#pragma unroll
        for (int q = 0; q < kF; ++q) acc = fma(-Z[a][q], xm[q][d], acc);
        x[a][d] = acc;
      }
    if (i >= 2) {
#pragma unroll
      for (int a = 0; a < kF; ++a) {
#pragma unroll
        for (int q = 0; q < kF; ++q) Z[a][q] = Zn[a][q];
#pragma unroll
        for (int d = 0; d < D; ++d) w[a][d] = wn[a][d];
      }
      if (i >= 3) fetch(i - 2);
    }
    emit(actual(i), x);
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) xm[a][d] = x[a][d];
  }
  // the trajectory's own ends: chunk 0 starts, chunk J-1 ends with the boundary vector
  if (active) {
    double* e = chunk_ends + ((b * J + (side ? J - 1 : 0)) * 2 + side) * kVec;
#pragma unroll
    for (int a = 0; a < kF; ++a)
#pragma unroll
      for (int d = 0; d < D; ++d) e[a * D + d] = xb[a][d];
  }
  bad |= __shfl_xor_sync(0xffffffffu, bad, 16);
  if (bad && status && active && side == 0) atomicOr(status + b, bad);
}

// ---- glue -------------------------------------------------------------------------------------------------------
// interior free derivatives of the chunks [B J][m-1][kVec] into the trajectory's array [B][K-1][kVec]:
// block i of chunk j is vertex j m + i + 1, row j m + i (the separators' rows are written by the separator solve)
__global__ void scatter_chunk_free_kernel(long B, int K, int m, int kvec, const double* __restrict__ chunk_free,
                                          double* __restrict__ free_out) {
  const int J = K / m;
  const long per = (long)(m - 1) * kvec;
  const long total = B * J * per;
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
    const long t = e / per;
    const long r = e - t * per;
    const long b = t / J;
    const int j = (int)(t - b * J);
    free_out[(b * (K - 1) + (long)j * m) * kvec + r] = chunk_free[e];
  }
}

// status of a trajectory = OR over its chunks' (and the two kernels above)
__global__ void fold_chunk_status_kernel(long B, int J, const int32_t* __restrict__ chunk_status, const int32_t* __restrict__ extra,
                                         int32_t* __restrict__ status) {
  const long b = blockIdx.x * (long)blockDim.x + threadIdx.x;
  if (b >= B) return;
  int s = extra[b];
  for (int j = 0; j < J; ++j) s |= chunk_status[b * J + j];
  status[b] = s;
}

// Two internal streams per host thread and device (created once, never destroyed before the thread ends): the
// sub-batches of a call run their kernel chains side by side, so that the latency-bound separator solve of one --
// a 31-block chain on one warp per 16 trajectories -- overlaps the throughput-bound kernels of the other.  The fork
// and the join are events on the caller's stream: stream order as the caller sees it is unchanged, and the whole
// thing is capturable into a CUDA graph.
struct SideStreams {
  static constexpr int kN = 2;
  int device = -1;
  cudaStream_t s[kN] = {};
  cudaEvent_t fork = nullptr, join[kN] = {};
  bool ready() {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return false;
    if (device == dev) return true;
    if (device >= 0) return false;   // one device per thread; another device takes the single-stream path
    for (int i = 0; i < kN; ++i) {
      if (cudaStreamCreateWithFlags(&s[i], cudaStreamNonBlocking) != cudaSuccess) return false;
      if (cudaEventCreateWithFlags(&join[i], cudaEventDisableTiming) != cudaSuccess) return false;
    }
    if (cudaEventCreateWithFlags(&fork, cudaEventDisableTiming) != cudaSuccess) return false;
    device = dev;
    return true;
  }
};
inline SideStreams& side_streams() {
  static thread_local SideStreams st;
  return st;
}

// One contiguous range of trajectories through the three steps on stream `s`; every scratch array was allocated by
// the caller (on the caller's stream, before the fork).
template <int D>
struct RangeScratch {
  double *rec, *ends, *slots, *sep_blocks, *sep_edge, *sep_middle, *chunk_free;
  int32_t *st_chunk, *st_extra;
};

template <int D>
inline cudaError_t run_range(const FastParams& p, const RangeScratch<D>& w, cudaStream_t s) {
  const int K = p.K, m = chunk_segments(K), J = K / m;
  const long n_ch = p.B * J;
  constexpr int kVec = kF * D;
  using L = SepLayout<D>;
  cudaError_t e;
  if ((e = cudaMemsetAsync(w.st_extra, 0, sizeof(int32_t) * (size_t)p.B, s)) != cudaSuccess) return e;
  {
    const dim3 grid((unsigned)((n_ch + 127) / 128), 2);
    chunk_schur_kernel<D><<<grid, 128, 0, s>>>(p.B, K, m, p.positions, p.times, w.rec, w.st_extra);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  {
    const int ns = J - 1;
    assemble_separators_kernel<D><<<dim3((unsigned)((p.B * ns + 127) / 128), 3), 128, 0, s>>>(p.B, K, m, p.positions, p.times, w.rec,
                                                                                     w.sep_blocks, w.sep_edge, w.sep_middle);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    separator_solve_kernel<D><<<(unsigned)((p.B + 15) / 16), 32, 0, s>>>(p.B, K, m, p.end_derivatives, w.sep_blocks, w.sep_edge,
                                                                         w.sep_middle, w.ends, p.free_out, w.slots, w.st_extra);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  FastParams q = p;
  q.B = n_ch;
  q.K = m;
  q.chunk_J = J;   // the headline kernel picks every chunk's vertices out of the trajectories' own array
  q.end_derivatives = w.ends;
  q.times_out = nullptr;
  q.cost = nullptr;
  q.status = p.status ? w.st_chunk : nullptr;
  q.sweep_S = 0;
  q.aligned16 = (reinterpret_cast<uintptr_t>(p.times) % 16 == 0) && (reinterpret_cast<uintptr_t>(p.coeffs) % 16 == 0);
  // the chunks' interior free derivatives land in [B J][m-1][4][D]; the trajectory's array interleaves the
  // separators, so a caller asking for them gets them through the scatter below
  q.free_out = p.free_out ? w.chunk_free : nullptr;
  if ((e = tm::launch_d<D>(q, s)) != cudaSuccess) return e;
  if (p.free_out) {
    const long total = n_ch * (m - 1) * kVec;
    long grid = (total + 255) / 256;
    if (grid > sm_count() * 32) grid = sm_count() * 32;
    scatter_chunk_free_kernel<<<(unsigned)grid, 256, 0, s>>>(p.B, K, m, kVec, w.chunk_free, p.free_out);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  if (p.status) {
    fold_chunk_status_kernel<<<(unsigned)((p.B + 127) / 128), 128, 0, s>>>(p.B, J, w.st_chunk, w.st_extra, p.status);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  (void)sizeof(L);
  return cudaSuccess;
}

// p.times must be set (the caller estimates them first when they are computed on the device); p.cost is handled by
// the caller from the coefficients.  cudaErrorNotSupported: the headline kernel could not take the chunks.
template <int D>
inline cudaError_t launch_d(const FastParams& p, cudaStream_t stream) {
  const int K = p.K, m = chunk_segments(K), J = K / m;
  constexpr int kVec = kF * D;
  using L = SepLayout<D>;
  const int ns = J - 1, mA = ns / 2;
  const int stored = mA > 1 ? mA - 1 : 0;
  // Sub-batches: two from 2,048 trajectories on (each still fills the machine in its Schur and chunk kernels); the
  // ranges are multiples of 16 trajectories so that every array of a range keeps its alignment.  Measured at
  // K = 256: 4,096 trajectories 247 -> 232 us, 16,384 848 -> 805 us; three and four sub-batches 237 / 812 us.
  const int lanes = p.B >= 2048 && side_streams().ready() ? SideStreams::kN : 1;
  long first[SideStreams::kN + 1];
  for (int i = 0; i <= lanes; ++i) first[i] = i == lanes ? p.B : ((p.B * i / lanes) + 15) / 16 * 16;

  cudaError_t e;
  AsyncBuffer rec, ends, st_chunk, st_extra, slots, sep_blocks, sep_edge, sep_middle, free_scratch;
  const long n_ch = p.B * J;
  const long warps16 = (p.B + 15) / 16 + lanes;   // every range rounds its warp count up
  if ((e = rec.alloc(sizeof(double) * (size_t)Fields<D>::kCount * n_ch, stream)) != cudaSuccess) return e;
  if ((e = ends.alloc(sizeof(double) * (size_t)n_ch * 2 * kVec, stream)) != cudaSuccess) return e;
  if ((e = st_chunk.alloc(sizeof(int32_t) * (size_t)n_ch, stream)) != cudaSuccess) return e;
  if ((e = st_extra.alloc(sizeof(int32_t) * (size_t)p.B, stream)) != cudaSuccess) return e;
  if ((e = sep_blocks.alloc(sizeof(double) * (size_t)mA * L::kBlock * 2 * p.B, stream)) != cudaSuccess) return e;
  if ((e = sep_edge.alloc(sizeof(double) * (size_t)16 * 2 * p.B, stream)) != cudaSuccess) return e;
  if ((e = sep_middle.alloc(sizeof(double) * (size_t)L::kMid * p.B, stream)) != cudaSuccess) return e;
  if ((e = slots.alloc(sizeof(double) * (size_t)warps16 * stored * (kF * kF + kVec) * 32, stream)) != cudaSuccess) return e;
  if (p.free_out && (e = free_scratch.alloc(sizeof(double) * (size_t)n_ch * (m - 1) * kVec, stream)) != cudaSuccess) return e;

  SideStreams& ss = side_streams();
  if (lanes > 1 && (e = cudaEventRecord(ss.fork, stream)) != cudaSuccess) return e;
  cudaError_t result = cudaSuccess;
  for (int i = 0; i < lanes; ++i) {
    const long b0 = first[i], nb = first[i + 1] - first[i];
    if (nb <= 0) continue;
    FastParams r = p;
    r.B = nb;
    r.positions = p.positions + b0 * (long)(K + 1) * D;
    r.times = p.times + b0 * K;
    r.coeffs = p.coeffs + b0 * (long)K * D * fast::kN;
    r.end_derivatives = p.end_derivatives ? p.end_derivatives + b0 * 2 * kVec : nullptr;
    r.free_out = p.free_out ? p.free_out + b0 * (long)(K - 1) * kVec : nullptr;
    r.status = p.status ? p.status + b0 : nullptr;
    // the record arrays are [field][chunk][trajectory of the range]: every range owns a contiguous slice of each
    RangeScratch<D> w;
    w.rec = static_cast<double*>(rec.ptr) + (size_t)Fields<D>::kCount * J * b0;
    w.ends = static_cast<double*>(ends.ptr) + (size_t)b0 * J * 2 * kVec;
    w.st_chunk = static_cast<int32_t*>(st_chunk.ptr) + (size_t)b0 * J;
    w.st_extra = static_cast<int32_t*>(st_extra.ptr) + b0;
    w.sep_blocks = static_cast<double*>(sep_blocks.ptr) + (size_t)mA * L::kBlock * 2 * b0;
    w.sep_edge = static_cast<double*>(sep_edge.ptr) + (size_t)16 * 2 * b0;
    w.sep_middle = static_cast<double*>(sep_middle.ptr) + (size_t)L::kMid * b0;
    w.slots = static_cast<double*>(slots.ptr) + (size_t)(b0 / 16 + i) * stored * (kF * kF + kVec) * 32;
    w.chunk_free = p.free_out ? static_cast<double*>(free_scratch.ptr) + (size_t)b0 * J * (m - 1) * kVec : nullptr;
    cudaStream_t s = lanes > 1 ? ss.s[i] : stream;
    if (lanes > 1 && (e = cudaStreamWaitEvent(s, ss.fork, 0)) != cudaSuccess) { result = e; break; }
    e = run_range<D>(r, w, s);
    if (lanes > 1) {
      // join whatever was enqueued, also after an error: the caller's stream must not run ahead of the side streams
      cudaEventRecord(ss.join[i], s);
      cudaStreamWaitEvent(stream, ss.join[i], 0);
    }
    if (e != cudaSuccess) { result = e; break; }
  }
  return result;
}

#undef H1T

}  // namespace chunked
}  // namespace minsnap
