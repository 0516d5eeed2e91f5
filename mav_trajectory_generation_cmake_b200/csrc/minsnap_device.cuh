// Device-side helpers shared by all minsnap kernels (sm_100a).
//
// The kernels never form A, A^-1, Q or H per segment.  They use the exact unit-time tables
// in minsnap_tables.h and the time-scaling identities (k_r = r mod N/2 is the derivative
// order of end-point row r, delta the derivative whose square is integrated):
//     Ainv_T[i][r] = A1inv[i][r] * T^(k_r - i)
//     H_T[r][s]    = H1[r][s]    * T^(k_r + k_s + 1 - 2 delta)
//     Q_T[i][j]    = 2 b(delta,i) b(delta,j) / e * T^e,  e = i + j - 2 delta + 1
// which restate ref setupMappingMatrix / invertMappingMatrix / computeQuadraticCostJacobian /
// constructR (LIN.i:101-111, 132-169, 573-589, 305-308) without any matrix inverse.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

// __constant__: kernels that index the tables with compile-time constants get c[bank][offset]
// operands straight into DFMA/DMUL (no loads, no immediate moves)
#define MINSNAP_TABLE_QUAL static __constant__
// tables a kernel reads with a per-lane index live in global memory (coalesced; a lane-indexed read of a
// __constant__ array is replayed once per distinct address)
#define MINSNAP_TABLE_GLOBAL_QUAL static __device__
#include "minsnap_tables.h"

namespace minsnap {

constexpr int kWarp = 32;

// threadIdx.x / 32 through a shuffle: the compiler then knows the value is the same in every lane, keeps what is
// derived from it (batch bases, shared-memory carve-outs, loop bounds) in uniform registers and branches on it
// without a vote
__device__ __forceinline__ int uniform_warp_index() { return __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0); }

template <int N>
struct UnitTables;

#define MINSNAP_H1_CASE(N, d) \
  case d:                     \
    return minsnap_tables::kH1_N##N##_d##d;

template <>
struct UnitTables<4> {
  __device__ static const double* a1inv() { return minsnap_tables::kA1inv_N4; }
  __device__ static const double* h1(int delta) {
    switch (delta) {
      MINSNAP_H1_CASE(4, 0)
      default:
        return minsnap_tables::kH1_N4_d1;
    }
  }
};
template <>
struct UnitTables<6> {
  __device__ static const double* a1inv() { return minsnap_tables::kA1inv_N6; }
  __device__ static const double* h1(int delta) {
    switch (delta) {
      MINSNAP_H1_CASE(6, 0)
      MINSNAP_H1_CASE(6, 1)
      default:
        return minsnap_tables::kH1_N6_d2;
    }
  }
};
template <>
struct UnitTables<8> {
  __device__ static const double* a1inv() { return minsnap_tables::kA1inv_N8; }
  __device__ static const double* h1(int delta) {
    switch (delta) {
      MINSNAP_H1_CASE(8, 0)
      MINSNAP_H1_CASE(8, 1)
      MINSNAP_H1_CASE(8, 2)
      default:
        return minsnap_tables::kH1_N8_d3;
    }
  }
};
template <>
struct UnitTables<10> {
  __device__ static const double* a1inv() { return minsnap_tables::kA1inv_N10; }
  __device__ static const double* h1(int delta) {
    switch (delta) {
      MINSNAP_H1_CASE(10, 0)
      MINSNAP_H1_CASE(10, 1)
      MINSNAP_H1_CASE(10, 2)
      MINSNAP_H1_CASE(10, 3)
      default:
        return minsnap_tables::kH1_N10_d4;
    }
  }
};
template <>
struct UnitTables<12> {
  __device__ static const double* a1inv() { return minsnap_tables::kA1inv_N12; }
  __device__ static const double* h1(int delta) {
    switch (delta) {
      MINSNAP_H1_CASE(12, 0)
      MINSNAP_H1_CASE(12, 1)
      MINSNAP_H1_CASE(12, 2)
      MINSNAP_H1_CASE(12, 3)
      MINSNAP_H1_CASE(12, 4)
      default:
        return minsnap_tables::kH1_N12_d5;
    }
  }
};
#undef MINSNAP_H1_CASE

// b(d, j) = j (j-1) ... (j-d+1): ref computeBaseCoefficients, src/polynomial.cpp:140-155.
// Exact in double for every (d, j) the library reaches (j < 22).
__host__ __device__ inline double falling_factorial(int d, int j) {
  if (j < d) return 0.0;
  double r = 1.0;
  for (int q = 0; q < d; ++q) r *= static_cast<double>(j - q);
  return r;
}

// T^e for a small signed integer e: |e| - 1 multiplications, then at most one division.
__device__ inline double int_power(double T, int e) {
  const int n = e < 0 ? -e : e;
  double p = 1.0;
  for (int q = 0; q < n; ++q) p *= T;
  return e < 0 ? 1.0 / p : p;
}

__device__ inline double warp_sum(double v) {
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) v += __shfl_xor_sync(0xffffffffu, v, off);
  return v;
}

// f(std::integral_constant<int, D>) for the dimension counts D = 1..3 the standard-mask kernels are compiled for.
template <class F>
inline cudaError_t with_dim(int D, F&& f) {
  switch (D) {
    case 1: return f(std::integral_constant<int, 1>{});
    case 2: return f(std::integral_constant<int, 2>{});
    case 3: return f(std::integral_constant<int, 3>{});
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace minsnap
