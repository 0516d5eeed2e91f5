// Which kernel solves a call of minsnap_solve_standard: a pure function of the shape, the batch size, the
// device's multiprocessor count and the pointers' alignment, so that the whole table can be checked without a device
// (tests/cpp/standard_routes.cu).
#pragma once
#include <optional>

#include "minsnap_launch.h"
#include "minsnap_standard_bcr.cuh"
#include "minsnap_standard_chunked.cuh"
#include "minsnap_standard_fast.cuh"
#include "minsnap_standard_tm.cuh"

namespace minsnap {

struct StandardRouteQuery {
  long B;
  int K, D, N, derivative;
  long sms;                 // multiprocessors of the device (148 on B200)
  bool coeffs_aligned16;    // the coefficient array is 16-byte aligned
  bool inputs_aligned16;    // so are the positions and the times (no times counts as aligned)
  std::optional<StandardRoute> forced;
};

// the two-lane kernel (minsnap_standard_fast.cuh); K > 24 in long-chain mode
inline bool pair_fits(const StandardRouteQuery& q) { return fast::supported(q.K, q.D, q.N, q.derivative); }
// block cyclic reduction (minsnap_standard_bcr.cuh) also covers long chains whose staged inputs no longer fit the
// two-lane kernel
inline bool bcr_fits(const StandardRouteQuery& q) {
  return q.N == 10 && q.derivative == 4 && q.D >= 1 && q.D <= 3 && q.K > fast::kMaxK && bcr::supported(q.K, q.D);
}
inline bool chunked_fits(const StandardRouteQuery& q) {
  return chunked::supported(q.K, q.D, q.N, q.derivative) && q.inputs_aligned16 && q.coeffs_aligned16;
}

// The default decision after the partitioned route; also where an unforced Chunked call goes when the headline
// kernel cannot take its chunks.
inline StandardRoute route_after_chunked(const StandardRouteQuery& q) {
  // Long chains: block cyclic reduction, one CTA per trajectory, while the batch is too small to fill the machine
  // with two-lane warps.  Measured at K = 256: a trajectory takes ~25 us through the reduction and two CTAs fit an
  // SM, so B trajectories cost ceil(B / 296) x 25 us (64 -> 0.023 ms, 512 -> 0.052 ms, 4,096 -> 0.35 ms); the
  // two-lane kernel (sweeps, then a separate recovery pass) needs 0.17 ms however small the batch and 0.48 ms for
  // 4,096, and keeps that time up to ~19,000 trajectories (16 per warp, 8 warps per SM).
  if (bcr_fits(q) && (!pair_fits(q) || q.B <= 38 * q.sms)) return StandardRoute::Bcr;
  if (q.K > fast::kMaxK) return StandardRoute::PairLong;
  // the second-generation kernel (block storage in tensor memory, coefficients out through the TMA) where it applies
  if (tm::supported(q.K, q.D, q.N, q.derivative) && q.coeffs_aligned16) return StandardRoute::Tm;
  return StandardRoute::Pair;
}

inline bool route_fits(StandardRoute r, const StandardRouteQuery& q) {
  switch (r) {
    case StandardRoute::Tm: return tm::supported(q.K, q.D, q.N, q.derivative) && q.coeffs_aligned16;
    case StandardRoute::Pair: return pair_fits(q) && q.K <= fast::kMaxK;
    case StandardRoute::PairLong: return pair_fits(q) && q.K > fast::kMaxK;
    case StandardRoute::Bcr: return bcr_fits(q);
    case StandardRoute::Chunked: return chunked_fits(q);
    case StandardRoute::General: return true;
    default: return false;
  }
}

// The route of a call: the forced one when it can take the call, else Unsupported; unforced, the default decision.
inline StandardRoute choose_standard_route(const StandardRouteQuery& q) {
  if (q.forced) return route_fits(*q.forced, q) ? *q.forced : StandardRoute::Unsupported;
  if (!pair_fits(q) && !bcr_fits(q)) return StandardRoute::General;
  // Partitioned route (minsnap_standard_chunked.cuh): chunk Schur complements, separator solve, then every chunk
  // through the headline kernel.  Its four launches cost ~70 us however small the batch; the reduction kernel's
  // ceil(B / 296) x 25 us is below that up to four waves (K = 256: 1,024 -> 0.100 against 0.107 ms, 4,096 -> 0.348
  // against 0.267 ms, 16,384 -> 1.35 against 0.93 ms).
  if (chunked_fits(q) && q.B > 8 * q.sms) return StandardRoute::Chunked;
  return route_after_chunked(q);
}

}  // namespace minsnap
