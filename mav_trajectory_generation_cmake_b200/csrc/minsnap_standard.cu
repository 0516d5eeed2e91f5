// Standard-mask path: the constraint structure createRandomVertices produces (ref:
// src/vertex.cpp:59,71-76) -- end vertices fix derivatives 0..h-1, interior vertices fix
// position only.  n_fixed = K + 2h - 1, n_free = (K-1)(h-1).
//
// N = 10, snap, D <= 3 runs one of the standard-mask kernels (minsnap_standard_route.cuh picks it); every other
// shape packs its inputs into the general layout and runs the general kernels.
#include "minsnap_device.cuh"
#include "minsnap_launch.h"
#include "minsnap_standard_route.cuh"

namespace minsnap {

// ---- generic route ------------------------------------------------------------------------
__global__ void standard_mask_kernel(int K, int h, uint8_t* __restrict__ mask) {
  const int nc = (K + 1) * h;
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < nc; e += gridDim.x * blockDim.x) {
    const int v = e / h, c = e - v * h;
    mask[e] = (c == 0 || v == 0 || v == K) ? 1 : 0;
  }
}

// fixed_values[b][col][dim] in the reference's column order: vertex 0 (derivatives 0..h-1),
// vertices 1..K-1 (position), vertex K (derivatives 0..h-1).
__global__ void pack_standard_kernel(long B, int K, int D, int h, const double* __restrict__ positions,
                                     const double* __restrict__ end_derivatives, double* __restrict__ fixed_values) {
  const int n_fixed = K + 2 * h - 1;
  const long total = B * (long)n_fixed * D;
  for (long e = blockIdx.x * (long)blockDim.x + threadIdx.x; e < total; e += (long)gridDim.x * blockDim.x) {
    const int dim = (int)(e % D);
    const int col = (int)((e / D) % n_fixed);
    const long b = e / ((long)D * n_fixed);
    int v, c;
    if (col < h) { v = 0; c = col; }
    else if (col < h + K - 1) { v = col - h + 1; c = 0; }
    else { v = K; c = col - (h + K - 1); }
    double val;
    if (c == 0) val = positions[(b * (K + 1) + v) * D + dim];
    else val = end_derivatives ? end_derivatives[((b * 2 + (v == K)) * (h - 1) + (c - 1)) * D + dim] : 0.0;
    fixed_values[e] = val;
  }
}

static cudaError_t generic_route(long B, int S, int K, int D, int N, int derivative, const double* d_positions,
                                 const double* d_end_derivatives, const double* d_times, double* d_coeffs,
                                 double* d_free_out, double* d_cost, int32_t* d_status, cudaStream_t stream) {
  const int h = N / 2;
  const int n_fixed = K + 2 * h - 1;
  const int n_free = (K - 1) * (h - 1);
  AsyncBuffer mask, col, counts, fixed;
  cudaError_t e;
  if ((e = mask.alloc((size_t)(K + 1) * h, stream)) != cudaSuccess) return e;
  if ((e = col.alloc(sizeof(int32_t) * (size_t)N * K, stream)) != cudaSuccess) return e;
  if ((e = counts.alloc(sizeof(int32_t) * 2, stream)) != cudaSuccess) return e;
  if ((e = fixed.alloc(sizeof(double) * (size_t)B * n_fixed * D, stream)) != cudaSuccess) return e;
  standard_mask_kernel<<<((K + 1) * h + 255) / 256, 256, 0, stream>>>(K, h, static_cast<uint8_t*>(mask.ptr));
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = launch_reorder(N, K, 1, static_cast<uint8_t*>(mask.ptr), static_cast<int32_t*>(col.ptr),
                          static_cast<int32_t*>(counts.ptr), stream)) != cudaSuccess)
    return e;
  {
    const long total = B * (long)n_fixed * D;
    long grid = (total + 255) / 256;
    if (grid > sm_count() * 16) grid = sm_count() * 16;
    pack_standard_kernel<<<(int)grid, 256, 0, stream>>>(B, K, D, h, d_positions, d_end_derivatives,
                                                        static_cast<double*>(fixed.ptr));
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  GeneralSolveArgs g;
  g.B = B * S; g.K = K; g.D = D; g.N = N; g.derivative = derivative; g.n_fixed = n_fixed; g.n_free = n_free;
  g.fixed_div = S;
  g.d_col_of_row = static_cast<int32_t*>(col.ptr);
  g.d_fixed_values = static_cast<double*>(fixed.ptr);
  g.d_free_in = nullptr;
  g.d_times = d_times; g.d_coeffs = d_coeffs; g.d_free_out = d_free_out; g.d_cost = d_cost; g.d_status = d_status;
  return launch_solve_general(g, stream);
}

bool standard_supported(int K, int D, int N, int derivative) {
  return choose_standard_route({1, K, D, N, derivative, sm_count(), true, true, {}}) != StandardRoute::General;
}

static bool aligned16(const void* ptr) { return reinterpret_cast<uintptr_t>(ptr) % 16 == 0; }

// The parameters of the standard-mask kernels common to a solve and a cost sweep.
static fast::FastParams fast_params(long B, int K, const double* positions, const double* end_derivatives,
                                    const double* times, double* cost, int32_t* status) {
  fast::FastParams p{};
  p.B = B; p.K = K; p.positions = positions; p.end_derivatives = end_derivatives; p.times = times;
  p.cost = cost; p.status = status;
  return p;
}

static cudaError_t run_route(StandardRoute route, const StandardSolveArgs& a, const StandardRouteQuery& q,
                             cudaStream_t stream) {
  fast::FastParams p = fast_params(a.B, a.K, a.d_positions, a.d_end_derivatives, a.d_times, a.d_cost, a.d_status);
  p.v_max = a.v_max; p.a_max = a.a_max; p.magic = a.magic; p.times_out = a.d_times_out;
  p.coeffs = a.d_coeffs; p.free_out = a.d_free_out;
  p.aligned16 = q.inputs_aligned16 && q.coeffs_aligned16;
  // Without given times, Tm and Pair compute them in registers.  Chunked and General read them from memory: they are
  // estimated first.  Bcr and PairLong compute them too, into a scratch times_out where a later pass reads them
  // (Bcr's cost, PairLong's recovery).
  AsyncBuffer times_scratch, free_scratch;
  const bool estimate = route == StandardRoute::Chunked || route == StandardRoute::General;
  const bool times_later = (route == StandardRoute::Bcr && p.cost) || route == StandardRoute::PairLong;
  cudaError_t e;
  // a shape the general kernel refuses is refused before the estimate below writes times_out
  if (route == StandardRoute::General &&
      (e = general_fits(a.N, a.K, a.D, a.K + a.N - 1, (a.K - 1) * (a.N / 2 - 1))) != cudaSuccess)
    return e;
  if (!p.times && !p.times_out && (estimate || times_later)) {
    if ((e = times_scratch.alloc(sizeof(double) * (size_t)a.B * a.K, stream)) != cudaSuccess) return e;
    p.times_out = static_cast<double*>(times_scratch.ptr);
  }
  if (!p.times && estimate) {
    if ((e = launch_estimate_times(a.B, a.K, a.D, a.d_positions, a.v_max, a.a_max, a.magic, p.times_out, stream)) !=
        cudaSuccess)
      return e;
    p.times = p.times_out;
  }
  const double* times = p.times ? p.times : p.times_out;
  if (route == StandardRoute::General)
    return generic_route(a.B, 1, a.K, a.D, a.N, a.derivative, a.d_positions, a.d_end_derivatives, times, a.d_coeffs,
                         a.d_free_out, a.d_cost, a.d_status, stream);
  // Bcr, Chunked and PairLong leave the cost to a pass over the coefficients (ref computeCost, LIN.i:113-130)
  double* cost = nullptr;
  if (route == StandardRoute::Bcr || route == StandardRoute::Chunked || route == StandardRoute::PairLong)
    std::swap(cost, p.cost);
  if (route == StandardRoute::PairLong && !p.free_out) {
    if ((e = free_scratch.alloc(sizeof(double) * (size_t)a.B * (a.K - 1) * fast::kF * a.D, stream)) != cudaSuccess)
      return e;
    p.free_out = static_cast<double*>(free_scratch.ptr);
  }
  e = with_dim(a.D, [&](auto dim) {
    constexpr int D = decltype(dim)::value;
    switch (route) {
      case StandardRoute::Tm: return tm::launch_d<D>(p, stream);
      case StandardRoute::Pair: return fast::launch_d<D, true>(p, stream);
      case StandardRoute::Bcr: return bcr::launch_d<D>(p, stream);
      case StandardRoute::Chunked: return chunked::launch_d<D>(p, stream);
      case StandardRoute::PairLong: {
        // the two-lane kernel in long-chain mode: forward and backward sweeps only (free derivatives out), then the
        // coefficients as a pass of their own with one thread per segment
        const cudaError_t r = fast::launch_d<D, false>(p, stream);
        return r != cudaSuccess ? r : bcr::launch_recover<D>(p, p.free_out, times, stream);
      }
      default: return cudaErrorInvalidValue;
    }
  });
  if (e != cudaSuccess || !cost) return e;
  return launch_cost(a.B, a.K, a.D, a.N, a.derivative, a.d_coeffs, times, cost, stream);
}

cudaError_t launch_solve_standard(const StandardSolveArgs& a, cudaStream_t stream) {
  if (a.B == 0) return cudaSuccess;
  const StandardRouteQuery q{a.B, a.K, a.D, a.N, a.derivative, sm_count(), aligned16(a.d_coeffs),
                             aligned16(a.d_positions) && aligned16(a.d_times), a.forced};
  const StandardRoute route = choose_standard_route(q);
  if (route == StandardRoute::Unsupported) return cudaErrorNotSupported;
  const cudaError_t e = run_route(route, a, q, stream);
  // cudaErrorNotSupported: the headline kernel could not be set up (no tensor map).  Unforced, Tm falls back to the
  // first-generation kernel and Chunked to the default decision without it.
  if (e != cudaErrorNotSupported || q.forced) return e;
  if (route == StandardRoute::Tm) return run_route(StandardRoute::Pair, a, q, stream);
  if (route == StandardRoute::Chunked) return run_route(route_after_chunked(q), a, q, stream);
  return e;
}

cudaError_t launch_cost_sweep(const SweepArgs& a, cudaStream_t stream) {
  if (a.B == 0) return cudaSuccess;
  if (fast::supported(a.K, a.D, a.N, a.derivative)) {
    fast::FastParams p = fast_params(a.B, a.K, a.d_positions, a.d_end_derivatives, a.d_times, a.d_cost, a.d_status);
    p.sweep_S = a.S;
    p.aligned16 = aligned16(a.d_times);
    return with_dim(a.D, [&](auto dim) { return fast::launch_d<decltype(dim)::value, false>(p, stream); });
  }
  return generic_route(a.B, a.S, a.K, a.D, a.N, a.derivative, a.d_positions, a.d_end_derivatives, a.d_times, nullptr,
                       nullptr, a.d_cost, a.d_status, stream);
}

}  // namespace minsnap
