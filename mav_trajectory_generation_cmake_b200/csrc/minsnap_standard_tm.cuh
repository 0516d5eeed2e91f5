// Standard-mask solve, second generation (N = 10, snap, K = 2 or 4 <= K <= 12): the thread-pair
// elimination of minsnap_standard_fast.cuh with the cost ncu attributed to its output removed --
// per-lane coefficient stores, every lane of a store instruction in its own 128-byte line.
//
//  * Block storage in TENSOR MEMORY.  The Z (4x4) and w (4xD) of every eliminated block are
//    lane-private scratch, written once in the forward sweep and read once in the back
//    substitution.  They live in TMEM (tcgen05.st / tcgen05.ld, shape 32x32b: thread i of a warp
//    owns TMEM lane 32 (warp % 4) + i, a block is 32 + 8 D consecutive 32-bit columns).  No MMA is
//    involved: TMEM is used as what it physically is, a 128-lane x 512-column register-file
//    extension next to the SM, and the 21.5 KB of shared memory per warp it replaces hold the
//    copy-out tiles instead.
//  * Coefficients leave through the TMA as TENSOR stores.  Lanes 0..15 of a warp are the top-down
//    lanes of 16 consecutive trajectories, lanes 16..31 the bottom-up lanes.  After back-substitution
//    step j the top-down lanes hold segment j of their trajectories and the bottom-up lanes segment
//    K-1-j: 16 pieces of 80 D bytes each, 2400 D... apart in the coefficient array [B][K][10 D] -- a
//    {10 D, 1, 16} box of that 3-D tensor.  Every lane recovers its segment one dimension at a time
//    (10 live coefficients), parks it in its row of a dense shared-memory tile, and ONE elected lane
//    issues two cp.async.bulk.tensor.3d stores per step (SASS UTMASTG); rows past the end of a ragged
//    batch are clipped by the tensor map.  Two tiles per side: a step never waits for the previous copy.
//  * Recovery is interleaved with the back substitution (segment j is recovered as soon as x_j is
//    known), so x never leaves the registers and the 15 independent dot-product chains of a
//    dimension fill the FP64 pipe while the next block's TMEM loads are in flight.
//
// The tcgen05.ld/st are warp-collective with one address, so both lanes of a pair use tensor-memory slot j - 1 in
// iteration j.  Even K: both eliminate the same number of blocks.  Odd K (template parameter): the bottom-up lane
// has one block less, sits out the first forward iteration and the last recovery step, and its half of that
// step's tile is not sent.  Other shapes (K = 1, K = 3, K > 12, the cost sweep, unaligned outputs) keep the
// first-generation kernel.
//
// Arithmetic is that of minsnap_standard_fast.cuh (same closed-form blocks, same 2x2-Schur inverse,
// same summation orders).
#pragma once
#include <cuda.h>
#include <algorithm>
#include <cstdlib>

#include "minsnap_standard_fast.cuh"

namespace minsnap {
namespace tm {

using fast::kF;
using fast::kN;
using fast::kPairsPerWarp;
using fast::FastParams;
using fast::TimePowers;
using fast::tri;

constexpr int kWarpsPerCta = 4;   // one warp per TMEM lane quarter
constexpr int kMaxK = 12;
constexpr int kRecTab = 54;   // doubles per lane role in the recovery table (53 used)

#define H1T(r, s) (minsnap_tables::kH1_N10_d4[(r) * 10 + (s)])
#define A1T(i, r) (minsnap_tables::kA1inv_N10[(i) * 10 + (r)])

// ---- tensor memory -----------------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t cols) {
  const uint32_t dst = static_cast<uint32_t>(__cvta_generic_to_shared(smem_slot));
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(dst), "r"(cols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols) : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_store(uint32_t taddr, const double (&v)[4]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               :: "r"(taddr), "r"(__double2loint(v[0])), "r"(__double2hiint(v[0])), "r"(__double2loint(v[1])), "r"(__double2hiint(v[1])), "r"(__double2loint(v[2])), "r"(__double2hiint(v[2])), "r"(__double2loint(v[3])), "r"(__double2hiint(v[3])) : "memory");
}
__device__ __forceinline__ void tmem_load(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_store(uint32_t taddr, const double (&v)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
               :: "r"(taddr), "r"(__double2loint(v[0])), "r"(__double2hiint(v[0])), "r"(__double2loint(v[1])), "r"(__double2hiint(v[1])), "r"(__double2loint(v[2])), "r"(__double2hiint(v[2])), "r"(__double2loint(v[3])), "r"(__double2hiint(v[3])), "r"(__double2loint(v[4])), "r"(__double2hiint(v[4])), "r"(__double2loint(v[5])), "r"(__double2hiint(v[5])), "r"(__double2loint(v[6])), "r"(__double2hiint(v[6])), "r"(__double2loint(v[7])), "r"(__double2hiint(v[7])) : "memory");
}
__device__ __forceinline__ void tmem_load(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]) : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_store(uint32_t taddr, const double (&v)[16]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
               :: "r"(taddr), "r"(__double2loint(v[0])), "r"(__double2hiint(v[0])), "r"(__double2loint(v[1])), "r"(__double2hiint(v[1])), "r"(__double2loint(v[2])), "r"(__double2hiint(v[2])), "r"(__double2loint(v[3])), "r"(__double2hiint(v[3])), "r"(__double2loint(v[4])), "r"(__double2hiint(v[4])), "r"(__double2loint(v[5])), "r"(__double2hiint(v[5])), "r"(__double2loint(v[6])), "r"(__double2hiint(v[6])), "r"(__double2loint(v[7])), "r"(__double2hiint(v[7])), "r"(__double2loint(v[8])), "r"(__double2hiint(v[8])), "r"(__double2loint(v[9])), "r"(__double2hiint(v[9])), "r"(__double2loint(v[10])), "r"(__double2hiint(v[10])), "r"(__double2loint(v[11])), "r"(__double2hiint(v[11])), "r"(__double2loint(v[12])), "r"(__double2hiint(v[12])), "r"(__double2loint(v[13])), "r"(__double2hiint(v[13])), "r"(__double2loint(v[14])), "r"(__double2hiint(v[14])), "r"(__double2loint(v[15])), "r"(__double2hiint(v[15])) : "memory");
}
__device__ __forceinline__ void tmem_load(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31]) : "r"(taddr) : "memory");
}

__device__ __forceinline__ double pair_to_double(uint32_t lo, uint32_t hi) { return __hiloint2double((int)hi, (int)lo); }

// A block is stored / loaded in pieces of 4 doubles (x8): an operand group of 8 consecutive registers
// is what the values' natural allocation provides (measured: the x32 / x16 forms cost 56 register
// moves per block on either side).
template <int D>
__device__ __forceinline__ void tmem_store_block(uint32_t taddr, const double (&Z)[kF][kF], const double (&w)[kF][D]) {
#pragma unroll
  for (int a = 0; a < kF; ++a) {
    const double v[4] = {Z[a][0], Z[a][1], Z[a][2], Z[a][3]};
    tmem_store(taddr + 8 * a, v);
  }
  double flat[kF * D + 3];
#pragma unroll
  for (int e = 0; e < kF * D; ++e) flat[e] = w[e / D][e % D];
#pragma unroll
  for (int e = kF * D; e < kF * D + 3; ++e) flat[e] = 0.0;
#pragma unroll
  for (int c = 0; c < D; ++c) {   // 4 D doubles = D pieces
    const double v[4] = {flat[4 * c], flat[4 * c + 1], flat[4 * c + 2], flat[4 * c + 3]};
    tmem_store(taddr + 32 + 8 * c, v);
  }
}

// Z and w of one stored block: issue the loads, wait, unpack.
template <int D>
__device__ __forceinline__ void tmem_load_block(uint32_t taddr, double (&Z)[kF][kF], double (&w)[kF][D]) {
  uint32_t z[kF][8], r[D][8];
#pragma unroll
  for (int a = 0; a < kF; ++a) tmem_load(taddr + 8 * a, z[a]);
#pragma unroll
  for (int c = 0; c < D; ++c) tmem_load(taddr + 32 + 8 * c, r[c]);
  tmem_wait_ld();
#pragma unroll
  for (int a = 0; a < kF; ++a)
#pragma unroll
    for (int b2 = 0; b2 < kF; ++b2) Z[a][b2] = pair_to_double(z[a][2 * b2], z[a][2 * b2 + 1]);
#pragma unroll
  for (int e = 0; e < kF * D; ++e) w[e / D][e % D] = pair_to_double(r[e / 4][2 * (e % 4)], r[e / 4][2 * (e % 4) + 1]);
}

// ---- TMA: tensor store shared -> global ----------------------------------------------------
// The coefficients are written once and not read again by this launch: the stores carry an evict-first L2 policy, so
// that the 157 MB of output leave the inputs (and the next wave's prefetched inputs) in L2 (41.4 -> 41.0 us per
// 65,536 solves).
__device__ __forceinline__ uint64_t l2_evict_first_policy() {
  uint64_t policy;
  asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(policy));
  return policy;
}
__device__ __forceinline__ void tensor_store_3d(const CUtensorMap* map, const double* ssrc, int c0, int c1, int c2,
                                                uint64_t policy) {
  const uint32_t s = static_cast<uint32_t>(__cvta_generic_to_shared(ssrc));
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group.L2::cache_hint [%0, {%2, %3, %4}], [%1], %5;"
               ::"l"(reinterpret_cast<uint64_t>(map)), "r"(s), "r"(c0), "r"(c1), "r"(c2), "l"(policy) : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const double* gsrc, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(gsrc), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int kPending>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(kPending) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__host__ __device__ inline int stored_blocks(int K) {
  const int mA = (K - 1) / 2;
  return mA > 0 ? mA - 1 : 0;
}
template <int D>
__host__ __device__ constexpr int block_columns() { return 32 + 8 * D; }
template <int D>
inline int tmem_columns(int K) {
  const int need = stored_blocks(K) * block_columns<D>();
  int cols = 32;
  while (cols < need) cols <<= 1;
  return cols;
}
// per-warp shared memory, in doubles, every region a multiple of 128 bytes (the TMA reads the tiles):
// two input buffers of positions [16][(K+1) D] + times [16][K] (a warp's next batch arrives during the current
// one), copy-out tiles [2 buffers][2 sides][16][10 D]
template <int D>
struct WarpSmem {
  size_t pos, tim, in_stride, tile, total;
  __host__ __device__ explicit WarpSmem(int K) {
    size_t o = 0;
    pos = o; o += ((size_t)kPairsPerWarp * (K + 1) * D + 15) & ~(size_t)15;
    tim = o; o += ((size_t)kPairsPerWarp * K + 15) & ~(size_t)15;
    in_stride = o;
    o += in_stride;   // the second input buffer
    tile = o; o += (size_t)2 * 2 * kPairsPerWarp * D * kN;   // 16 x 80 D bytes is a multiple of 128
    total = o;
  }
};

// ref estimateSegmentTimes (src/vertex.cpp:162-178), same expression as minsnap_estimate_segment_times.  Out of
// line: inlined, its loop-invariant division was hoisted to the top of the kernel and ran on every launch.
template <int D>
__device__ __noinline__ void estimate_times(int K, double v_max, double a_max, double magic, double* times_out,
                                            const double* pos_s, double* time_s, long base, int n_here, int lane) {
  const int per_pos = (K + 1) * D;
  for (int e = lane; e < n_here * K; e += kWarp) {
    const int r = e / K, o = e - r * K;
    const double* p0 = pos_s + r * per_pos + o * D;
    double s2 = 0.0;
#pragma unroll
    for (int d = 0; d < D; ++d) {
      const double diff = p0[D + d] - p0[d];
      s2 += diff * diff;
    }
    const double distance = sqrt(s2);
    const double T = distance / v_max * 2 * (1.0 + magic * v_max / a_max * exp(-distance / v_max * 2));
    time_s[r * K + o] = T;
    if (times_out) times_out[(base + r) * K + o] = T;
  }
}

template <int D, bool kCost, bool kExtras, bool kOdd = false>
__global__ void __launch_bounds__(kWarpsPerCta * 32, 2)
solve_standard_tm_kernel(FastParams p, int tmem_cols, int resident_warps, const __grid_constant__ CUtensorMap coeff_map,
                         int pdl) {
  extern __shared__ __align__(128) double smem[];
  __shared__ uint32_t tmem_base_slot;
  // Recovery constants per lane role.  A top-down lane's new vector x_j STARTS its segment and the previous one
  // ends it; for a bottom-up lane it is the other way round and odd derivatives change sign.  Instead of
  // selecting the 24 values of every step, the role is folded into the table a lane reads:
  //   rec_tab[side][(i-5) 9 + 0]     = A1inv[i][5]                                  (position difference)
  //   rec_tab[side][(i-5) 9 + 1 + a] = side ? (-1)^(a+1) A1inv[i][6+a] : A1inv[i][1+a]   (applied to T^k new_k)
  //   rec_tab[side][(i-5) 9 + 5 + a] = side ? (-1)^(a+1) A1inv[i][1+a] : A1inv[i][6+a]   (applied to T^k old_k)
  //   rec_tab[side][45 + a]          = side ? 0 : A1inv[1+a][1+a]                        (c_k from new_k)
  //   rec_tab[side][49 + a]          = side ? (-1)^(a+1) A1inv[1+a][1+a] : 0             (c_k from old_k)
  __shared__ __align__(16) double rec_tab[2][kRecTab];
  // packed lower triangle of the per-segment cost form (doubled off-diagonal entries, tools/gen_tables.py); read
  // from shared memory the 45 entries pass through vector registers for an instruction each -- as constant-bank
  // operands they filled the uniform registers of the recovery loop (57.4 -> 62.7 us with cost)
  __shared__ __align__(16) double cost_tab[kCost ? 46 : 2];
  const uint64_t store_policy = l2_evict_first_policy();
  const int lane = threadIdx.x & 31;
  // through a shuffle the compiler knows the warp index is warp-uniform: addresses and batch bases derived from
  // it stay in uniform registers, and the TMA operands need no per-lane vote loop
  const int warp = uniform_warp_index();
  const int K = p.K;
  const int per_pos = (K + 1) * D;
  constexpr int kVec = kF * D;    // doubles per vertex vector
  constexpr int kTile = D * kN;   // doubles per segment

  const WarpSmem<D> lay(K);
  double* wbase = smem + (size_t)warp * lay.total;
  double* pos_s = wbase + lay.pos;     // [16][per_pos]   (the current batch's buffer; the other one is
  double* time_s = wbase + lay.tim;    // [16][K]          lay.in_stride further on or back)
  double* tile_s = wbase + lay.tile;   // [2][2][16][kTile]

  const long pairs_per_cta = (long)kWarpsPerCta * kPairsPerWarp;
  const long stride = (long)gridDim.x * pairs_per_cta;
  long base = (long)blockIdx.x * pairs_per_cta + (long)warp * kPairsPerWarp;
  // inputs by cp.async: every chunk of a batch in flight before the single wait
  auto issue_inputs = [&](long b0, double* pos_s, double* time_s) {
    const int n = (int)min((long)kPairsPerWarp, p.B - b0);
    if (kExtras && p.chunk_J > 0) {
      // chunks of longer trajectories: every problem's K + 1 vertices from its own place in the trajectories'
      // array (vertex t K + t / chunk_J on).  The n per_pos elements of the batch are dealt to the lanes 32 at
      // a time; a lane advances its (problem, offset, chunk-in-trajectory) position incrementally.
      const long traj0 = b0 / p.chunk_J;
      const int in0 = (int)(b0 - traj0 * p.chunk_J);
      int r = lane / per_pos, o = lane - r * per_pos;   // lane < 32: a handful of problems at most
      int in_traj = in0 + r;
      long traj = traj0;
      while (in_traj >= p.chunk_J) { in_traj -= p.chunk_J; ++traj; }
      while (r < n) {
        __pipeline_memcpy_async(pos_s + r * per_pos + o, p.positions + ((b0 + r) * K + traj) * D + o, 8);
        o += kWarp;
        while (o >= per_pos) {
          o -= per_pos;
          ++r;
          if (++in_traj == p.chunk_J) { in_traj = 0; ++traj; }
        }
      }
    } else {
      fast::async_copy_doubles(pos_s, p.positions + b0 * per_pos, n * per_pos, lane, p.aligned16);
    }
    if (p.times) fast::async_copy_doubles(time_s, p.times + b0 * K, n * K, lane, p.aligned16);
    __pipeline_commit();
  };
  // Programmatic dependent launch (pdl): the next launch on the stream may start filling the SMs this
  // launch's last CTAs leave, and runs its prologue (recovery table, tensor-memory allocation) there; it reads
  // nothing a predecessor may have written before griddepcontrol.wait, which returns once the predecessor has
  // completed and flushed -- stream order as the caller sees it is unchanged.  Back-to-back launches: 49.3 ->
  // 46.5 us per 65,536 solves.  Without pdl the first batch's loads are in flight during the allocation.
  if (pdl) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // the recovery table is generated (tools/gen_tables.py) and arrives from global memory by cp.async: nobody
  // waits for it before the first batch's inputs are waited for
  static_assert(2 * kRecTab <= kWarpsPerCta * 32, "one table entry per thread");
  if (threadIdx.x < 2 * kRecTab)
    __pipeline_memcpy_async(&rec_tab[0][0] + threadIdx.x, minsnap_tables::kRecoveryRoles_N10 + threadIdx.x, 8);
  if (kCost && threadIdx.x < 46)
    __pipeline_memcpy_async(cost_tab + threadIdx.x, minsnap_tables::kCostFormGlobal_N10_d4 + threadIdx.x, 8);
  __pipeline_commit();
  if (lane == 0) asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(&coeff_map)) : "memory");
  // tensor memory: one allocation per CTA (warp 0), every warp works in its own lane quarter.  The warps meet
  // the allocation at a barrier BEFORE any of them waits for its inputs (a barrier one block into the sweep,
  // with the arithmetic under way, was measured 1.4 us slower per 65,536 solves).
  uint32_t taddr = 0;
  bool tmem_ready = false;
  auto tmem_meet = [&](bool inputs_in_flight) {
    // this thread's part of the recovery table has landed (the inputs, committed after it, may still be in flight)
    if (inputs_in_flight) __pipeline_wait_prior(1); else __pipeline_wait_prior(0);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    taddr = tmem_base_slot + ((uint32_t)(warp & 3) << 21);   // lane field (bits 31..16) = 32 (warp % 4)
    tmem_ready = true;
  };
  if (pdl) {
    // all of this runs while the predecessor's last CTAs drain
    if (warp == 0) tmem_alloc(&tmem_base_slot, (uint32_t)tmem_cols);
    tmem_meet(false);
    // L2 is the point of coherence: pulling this warp's first batch towards it before the predecessor has
    // completed cannot leave a stale copy anywhere, and the first wave's DRAM latency passes during the wait
    if (lane == 0 && base + kPairsPerWarp <= p.B && p.aligned16 && !(kExtras && p.chunk_J > 0)) {
      bulk_prefetch_l2(p.positions + base * per_pos, (uint32_t)(kPairsPerWarp * per_pos * sizeof(double)));
      if (p.times) bulk_prefetch_l2(p.times + base * K, (uint32_t)(kPairsPerWarp * K * sizeof(double)));
    }
    asm volatile("griddepcontrol.wait;" ::: "memory");
  }

  const int side = lane >> 4;   // 0: top-down lane, 1: bottom-up lane
  const int q = lane & 15;      // trajectory of the batch
  const int nb = K - 1;         // unknown blocks
  const int mA = nb / 2;        // blocks eliminated by the top-down lane; the middle block is vertex mA + 1
  // Odd K: the bottom-up lane has one block (and one segment) less.  It sits out the FIRST forward iteration and the
  // LAST recovery step (local index jj = j - late), so that both lanes store / load tensor memory slot j - 1 in
  // iteration j -- the tcgen05 operations are warp-collective with one address -- and both reach their last block
  // (the one that stays in registers) in the same iteration.
  constexpr int odd = kOdd ? 1 : 0;       // a template parameter: the even-K instantiations carry none of this
  const int late = kOdd ? side : 0;       // per lane
  const double flip[kF] = {side ? -1.0 : 1.0, 1.0, side ? -1.0 : 1.0, 1.0};   // (-1)^k, k = 1..4, bottom-up lane

  int buf = 0;
  bool first = true;
  int in_buf = 0;
  for (; base < p.B; base += stride) {
    const int n_here = (int)min((long)kPairsPerWarp, p.B - base);
    const long prob = base + q;
    const bool active = q < n_here;
    const long other_in = in_buf ? -(long)lay.in_stride : (long)lay.in_stride;
    if (first) {
      first = false;
      issue_inputs(base, pos_s, time_s);
      // the batch that will take this warp's place on the SM one wave from now is pulled into L2 (TMA
      // prefetch), so that only the first wave of a launch waits for DRAM
      if (lane == 0 && p.aligned16 && !(kExtras && p.chunk_J > 0)) {
        const long pf = base + (long)resident_warps * kPairsPerWarp;
        if (pf + kPairsPerWarp <= p.B) {
          bulk_prefetch_l2(p.positions + pf * per_pos, (uint32_t)(kPairsPerWarp * per_pos * sizeof(double)));
          if (p.times) bulk_prefetch_l2(p.times + pf * K, (uint32_t)(kPairsPerWarp * K * sizeof(double)));
        }
      }
      if (!pdl) {   // the loads are in flight during the allocation
        if (warp == 0) tmem_alloc(&tmem_base_slot, (uint32_t)tmem_cols);
        tmem_meet(true);
      }
    }
    // the boundary derivatives of the lane's end of the chain (actual coordinates) are requested before the
    // inputs are waited for: both latencies pass together
    const double* bd_src = nullptr;
    if (kExtras && p.end_derivatives && active) bd_src = p.end_derivatives + (prob * 2 + side) * kVec;
    double bd_first[kF][D];
    if (kExtras) {
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) bd_first[a][d] = bd_src ? __ldg(bd_src + a * D + d) : 0.0;
    }
    __pipeline_wait_prior(0);
    __syncwarp();
    if (base + stride < p.B) {
      // the warp's next batch arrives in the other buffer while this one is solved (every lane left that
      // buffer before the __syncwarp above)
      issue_inputs(base + stride, pos_s + other_in, time_s + other_in);
      if (kExtras && p.end_derivatives && prob + stride < p.B) {
        // and its boundary derivatives move towards L1 (the loads at the top of the next batch hit there)
        const double* nb_src = p.end_derivatives + ((prob + stride) * 2 + side) * kVec;
        asm volatile("prefetch.global.L1 [%0];" ::"l"(nb_src));
        asm volatile("prefetch.global.L1 [%0];" ::"l"(nb_src + kVec - 1));
      }
    }
    if (!p.times) {
      estimate_times<D>(K, p.v_max, p.a_max, p.magic, p.times_out, pos_s, time_s, base, n_here, lane);
      __syncwarp();
    }
    // idle pairs of a ragged last batch run on the first pair's inputs (nothing of theirs reaches memory)
    const int qi = active ? q : 0;
    const double* my_pos = pos_s + qi * per_pos;
    const double* my_time = time_s + qi * K;
    // local chain: vertex j <-> actual vertex (side ? K - j : j); segment j <-> actual (side ? K-1-j : j)
    auto local_T = [&](int j) { return my_time[side ? K - 1 - j : j]; };
    auto local_p = [&](int j, int d) { return my_pos[(side ? K - j : j) * D + d]; };

    int status = 0;
    auto bd = [&](int a, int d) { return (kExtras && bd_src) ? flip[a] * __ldg(bd_src + a * D + d) : 0.0; };

    double xm[kF][D];             // middle block solution, local coordinates; then the far vector of each step
    double Z[kF][kF], w[kF][D];   // after the forward sweep: the lane's LAST block (never leaves the registers)
#pragma unroll
    for (int a = 0; a < kF; ++a) {
#pragma unroll
      for (int b = 0; b < kF; ++b) Z[a][b] = 0.0;
#pragma unroll
      for (int d = 0; d < D; ++d) w[a][d] = 0.0;
    }
    {
      auto rhs_block = [&](const TimePowers& tprev, const TimePowers& tnext, const double (&dprev)[D],
                           const double (&dnext)[D], double (&out)[kF][D]) {
#pragma unroll
        for (int a = 0; a < kF; ++a) {
          const double ce = H1T(6 + a, 5) * tprev.P[a + 1];   // end-free row of the previous segment
          const double cs = H1T(1 + a, 5) * tnext.P[a + 1];   // start-free row of the next segment
#pragma unroll
          for (int d = 0; d < D; ++d) out[a][d] = -fma(ce, dprev[d], cs * dnext[d]);
        }
      };
      TimePowers tp_prev, tp_next;
      // ---- forward sweep ------------------------------------------------------------------
      double S[10], g[kF][D];
      double dp_prev[D], dp_next[D];
      tp_prev.set(local_T(0));
      tp_next.set(local_T(1));
#pragma unroll
      for (int d = 0; d < D; ++d) {
        dp_prev[d] = local_p(1, d) - local_p(0, d);
        dp_next[d] = local_p(2, d) - local_p(1, d);
      }
      fast::diag_block(tp_prev, tp_next, S);
      rhs_block(tp_prev, tp_next, dp_prev, dp_next, g);
      if (kExtras && bd_src) {
        double E0[kF][kF];
        fast::coupling_block(tp_prev, E0);
#pragma unroll
        for (int b = 0; b < kF; ++b)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double acc = g[b][d];
#pragma unroll
            for (int a = 0; a < kF; ++a) acc = fma(-E0[a][b], flip[a] * bd_first[a][d], acc);
            g[b][d] = acc;
          }
      }
      for (int j = 1; j <= mA; ++j) {
        // here (jj = j - late >= 1): tp_prev = segment jj-1, tp_next = segment jj, S/g = reduced block jj
        const bool more = j < mA;        // warp-uniform: the lane's own last block is jj = mA - late
        const int jj = j - late;
        const bool mine = jj >= 1;
        TimePowers tp_new;
        double dp_new[D];
        double E[kF][kF];
        if (mine) {
        tp_new.set(local_T(more ? jj + 1 : jj));
#pragma unroll
        for (int d = 0; d < D; ++d) dp_new[d] = more ? local_p(jj + 2, d) - local_p(jj + 1, d) : 0.0;
        double Si[10];
        if (!fast::spd4_inverse(S, Si)) status |= 1;
        fast::coupling_block(tp_next, E);
#pragma unroll
        for (int b = 0; b < kF; ++b) {
          const double in[4] = {E[0][b], E[1][b], E[2][b], E[3][b]};
          double col[4];
          fast::sym4_apply(Si, in, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) Z[a][b] = col[a];
        }
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const double in[4] = {g[0][d], g[1][d], g[2][d], g[3][d]};
          double col[4];
          fast::sym4_apply(Si, in, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) w[a][d] = col[a];
        }
        }
        // block jj goes to tensor memory slot j - 1: Z at column (j-1) pitch, w right behind it (every lane takes
        // part; a lane that sat this iteration out parks zeros it never reads)
        if (more) tmem_store_block<D>(taddr + (uint32_t)((j - 1) * block_columns<D>()), Z, w);
        if (more && mine) {
          // advance to block jj+1: D_{jj+1} - E^T Z,  b_{jj+1} - E^T w
          tp_prev = tp_next;
          tp_next = tp_new;
#pragma unroll
          for (int d = 0; d < D; ++d) {
            dp_prev[d] = dp_next[d];
            dp_next[d] = dp_new[d];
          }
          fast::diag_block(tp_prev, tp_next, S);
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
      if (mA > 1) tmem_wait_st();   // the stores are complete before the back substitution loads them

      // Schur contribution of this lane to the middle block, from its last eliminated block
      // (tp_next holds the powers of the lane's last local segment): C = E^T Z, c = E^T w
      double C[10], c[kF][D];
#pragma unroll
      for (int i = 0; i < 10; ++i) C[i] = 0.0;
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) c[a][d] = 0.0;
      if (mA >= 1) {
        double E[kF][kF];
        fast::coupling_block(tp_next, E);
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
        const int m = mA + 1;   // actual middle vertex
        TimePowers ta, tb;
        ta.set(my_time[m - 1]);
        tb.set(my_time[m]);
        double da[D], db[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
          da[d] = my_pos[m * D + d] - my_pos[(m - 1) * D + d];
          db[d] = my_pos[(m + 1) * D + d] - my_pos[m * D + d];
        }
        fast::diag_block(ta, tb, Sm);
        rhs_block(ta, tb, da, db, gm);
        if (kExtras && p.end_derivatives && active && K == 2) {
          // both boundary couplings reach the middle block directly
          const double* src = p.end_derivatives + (prob * 2 + 0) * kVec;
          double E0[kF][kF];
          fast::coupling_block(ta, E0);
#pragma unroll
          for (int b = 0; b < kF; ++b)
#pragma unroll
            for (int d = 0; d < D; ++d)
#pragma unroll
              for (int a = 0; a < kF; ++a) gm[b][d] = fma(-E0[a][b], src[a * D + d], gm[b][d]);
          src += kVec;
          double E1[kF][kF];
          fast::coupling_block(tb, E1);
#pragma unroll
          for (int a = 0; a < kF; ++a)
#pragma unroll
            for (int d = 0; d < D; ++d)
#pragma unroll
              for (int b = 0; b < kF; ++b) gm[a][d] = fma(-E1[a][b], src[b * D + d], gm[a][d]);
        }
      }
      {
        // subtract the top-down contribution first, then the bottom-up one, on both lanes
#pragma unroll
        for (int i = 0; i < 10; ++i) {
          const double other = __shfl_xor_sync(0xffffffffu, C[i], 16);
          const double cA = side ? other : C[i];
          const double cB = side ? C[i] : other;
          Sm[i] = (Sm[i] - cA) - cB;
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
        if (!fast::spd4_inverse(Sm, Si)) status |= 1;
#pragma unroll
        for (int d = 0; d < D; ++d) {
          const double in[4] = {gm[0][d], gm[1][d], gm[2][d], gm[3][d]};
          double col[4];
          fast::sym4_apply(Si, in, col);
#pragma unroll
          for (int a = 0; a < kF; ++a) xm[a][d] = flip[a] * col[a];   // -> local coordinates
        }
      }
      if (kExtras && p.free_out && active && side == 0) {
        double* dst = p.free_out + (prob * (long)nb + mA) * kVec;
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) dst[a * D + d] = xm[a][d];
      }
    }

    // ---- back substitution outwards, each step followed by the recovery of its segment --------
    // Step j (mA .. 0) produces x of local vertex j (x_j = w_j - Z_j x_{j+1}; the boundary values at
    // j = 0) and recovers local segment j, which lies between local vertices j (near) and j + 1 (far).
    double cost_acc = 0.0;
    int nonfinite = 0;
    int pending_j = -1;
    auto flush_tile = [&](int jj, int b) {
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        const double* t0 = tile_s + (size_t)(b * 2) * kPairsPerWarp * kTile;
        tensor_store_3d(&coeff_map, t0, 0, jj, (int)base, store_policy);
        // the bottom-up rows hold local segment jj - odd (odd K: none in the last step)
        if (jj - odd >= 0)
          tensor_store_3d(&coeff_map, t0 + kPairsPerWarp * kTile, 0, K - 1 - (jj - odd), (int)base, store_policy);
        // the group is committed where it is next waited for: committed here, the instruction sat ~2 % of
        // the kernel on the scoreboard of the two stores just issued
      }
    };
    for (int j = mA; j >= 0; --j) {
      const int jj = j - late;          // the lane's local vertex / segment of this step; -1: the lane sits it out
      const int jc = jj > 0 ? jj : 0;   // (it then repeats its step 0 into a tile row that is never sent)
      double x_near[kF][D];
      if (j >= 1 && j < mA) tmem_load_block<D>(taddr + (uint32_t)((j - 1) * block_columns<D>()), Z, w);
      if (jj >= 1) {
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) {
            double acc = w[a][d];
#pragma unroll
            for (int b = 0; b < kF; ++b) acc = fma(-Z[a][b], xm[b][d], acc);
            x_near[a][d] = acc;
          }
        if (kExtras && p.free_out && active) {
          const int v = side ? K - jj : jj;   // actual vertex
          double* dst = p.free_out + (prob * (long)nb + (v - 1)) * kVec;
#pragma unroll
          for (int a = 0; a < kF; ++a)
#pragma unroll
            for (int d = 0; d < D; ++d) dst[a * D + d] = flip[a] * x_near[a][d];
        }
      } else {
#pragma unroll
        for (int a = 0; a < kF; ++a)
#pragma unroll
          for (int d = 0; d < D; ++d) x_near[a][d] = bd(a, d);
      }

      if (pending_j >= 0) {
        // The tile of the previous step leaves now: its 16 top-down rows are segment j+1 of 16 consecutive
        // trajectories, its 16 bottom-up rows segment K-2-j -- two {10 D, 1, 16} boxes of the coefficient
        // tensor [B][K][10 D].  Issued here, one back-substitution later, the proxy fence finds the tile's
        // stores long complete.
        flush_tile(pending_j, buf ^ 1);
      }
      // recovery of local segment j (ref updateSegmentsFromCompactConstraints, LIN.i:252-273) in ACTUAL
      // orientation: the bottom-up lane's segment starts at its far vertex; odd derivatives change sign.
      const int seg = side ? K - 1 - jc : jc;
      const double T = my_time[seg];
      if (!(T > 0.0)) status |= 2;   // MINSNAP_STATUS_BAD_TIME; the two lanes cover all K segments
      const double T2 = T * T, T3 = T2 * T, T4 = T2 * T2;
      const double tk[kF] = {T, T2, T3, T4};
      const double i1 = fast::fast_rcp(T);
      const double i2 = i1 * i1, i4 = i2 * i2, i5 = i4 * i1;
      const double ipow[5] = {i5, i5 * i1, i5 * i2, i4 * i4, i4 * i5};   // T^-5 .. T^-9
      double* tile = tile_s + ((size_t)(buf * 2 + side) * kPairsPerWarp + q) * kTile;
      const double* tab = rec_tab[side];
      double u[2 * kF + 1][D];   // [dp, T^k new_k (k = 1..4), T^k old_k (k = 1..4)], new = x_j, old = x_{j+1} (local)
      double cf[D][kN];
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const double p0 = my_pos[seg * D + d];
        u[0][d] = my_pos[(seg + 1) * D + d] - p0;
        cf[d][0] = p0;
      }
#pragma unroll
      for (int a = 0; a < kF; ++a) {
        const double kn = tab[45 + a], ko = tab[49 + a];
#pragma unroll
        for (int d = 0; d < D; ++d) {
          u[1 + a][d] = tk[a] * x_near[a][d];
          u[1 + kF + a][d] = tk[a] * xm[a][d];
          cf[d][1 + a] = fma(kn, x_near[a][d], ko * xm[a][d]);
        }
      }
      // 5 rows x D dimensions = 15 independent accumulation chains, advanced together one table column at a
      // time (a row-by-row order leaves only D chains in flight against the 8-cycle FP64 latency)
      {
        double acc[kN - 5][D];
#pragma unroll
        for (int i = 0; i < kN - 5; ++i)
#pragma unroll
          for (int d = 0; d < D; ++d) acc[i][d] = tab[i * 9] * u[0][d];
#pragma unroll
        for (int c = 1; c < 9; ++c)
#pragma unroll
          for (int i = 0; i < kN - 5; ++i) {
            const double coef = tab[i * 9 + c];
#pragma unroll
            for (int d = 0; d < D; ++d) acc[i][d] = fma(coef, u[c][d], acc[i][d]);
          }
#pragma unroll
        for (int i = 0; i < kN - 5; ++i)
#pragma unroll
          for (int d = 0; d < D; ++d) cf[d][5 + i] = acc[i][d] * ipow[i];
      }
      // non-finite detection on the exponent fields of c_9 (scaled by T^-9: overflows first) and c_4
#pragma unroll
      for (int d = 0; d < D; ++d) {
        const int e9 = __double2hiint(cf[d][kN - 1]) & 0x7ff00000, e4 = __double2hiint(cf[d][kF]) & 0x7ff00000;
        if (e9 == 0x7ff00000 || e4 == 0x7ff00000) nonfinite = 1;
      }
      // the copies that read this buffer two steps ago are done with it
      if (lane == 0) {
        bulk_commit();   // the previous step's two stores
        bulk_wait_read<1>();
      }
      __syncwarp();
      {
        double2* t2 = reinterpret_cast<double2*>(tile);
#pragma unroll
        for (int e = 0; e < kTile; e += 2) t2[e / 2] = make_double2(cf[e / kN][e % kN], cf[(e + 1) / kN][(e + 1) % kN]);
      }
      double qsum = 0.0;
      if (kCost) {
        // u^T Hred1 u * T^-7: the per-segment quadratic form in scaled variables (SURVEY 8d) over the packed lower
        // triangle, every entry fetched once from shared memory and applied to the D dimensions.  The variables
        // are in the lane's local orientation: time reversal leaves the form invariant when the position
        // difference changes sign with the odd derivatives.
        double fu0[D], qd[D];
#pragma unroll
        for (int d = 0; d < D; ++d) {
          fu0[d] = flip[0] * u[0][d];
          qd[d] = (cost_tab[0] * fu0[d]) * fu0[d];
        }
#pragma unroll
        for (int r = 1; r < 2 * kF + 1; ++r) {
          double row[D];
          const double c0 = cost_tab[tri(r, 0)], cr = cost_tab[tri(r, r)];
#pragma unroll
          for (int d = 0; d < D; ++d) row[d] = fma(c0, fu0[d], cr * u[r][d]);
#pragma unroll
          for (int s2 = 1; s2 < r; ++s2) {
            const double c = cost_tab[tri(r, s2)];
#pragma unroll
            for (int d = 0; d < D; ++d) row[d] = fma(c, u[s2][d], row[d]);
          }
#pragma unroll
          for (int d = 0; d < D; ++d) qd[d] = fma(row[d], u[r][d], qd[d]);
        }
#pragma unroll
        for (int d = 0; d < D; ++d) qsum += qd[d];
      }
      if (kCost && jj >= 0) cost_acc = fma(qsum, i5 * i2, cost_acc);
      pending_j = j;   // this step's tile leaves during the next step (or after the loop)
      buf ^= 1;
#pragma unroll
      for (int a = 0; a < kF; ++a)
#pragma unroll
        for (int d = 0; d < D; ++d) xm[a][d] = x_near[a][d];
    }

    flush_tile(pending_j, buf ^ 1);   // the last step's tile
    if (kCost && p.cost) {
      cost_acc += __shfl_xor_sync(0xffffffffu, cost_acc, 16);
      if (active && side == 0) p.cost[prob] = 0.5 * cost_acc;
    }
    if (nonfinite) status |= 4;
    status |= __shfl_xor_sync(0xffffffffu, status, 16);
    if (p.status && active && side == 0) p.status[prob] = status;
    // the next batch is in the other input buffer
    pos_s += other_in;
    time_s += other_in;
    in_buf ^= 1;
  }
  if (!tmem_ready) tmem_meet(false);   // a warp without a batch (ragged last CTA)
  if (lane == 0) {
    bulk_commit();
    bulk_wait_read<0>();   // shared memory stays valid until the last copies have read it
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem_base_slot, (uint32_t)tmem_cols);
}

#undef H1T
#undef A1T

inline bool supported(int K, int D, int N, int derivative) {
  // even K from 2, odd K from 5 (K = 3 leaves the bottom-up lane without a block: first-generation kernel)
  return N == 10 && derivative == 4 && D >= 1 && D <= 3 && K >= 2 && K <= kMaxK && K != 3;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (no link against libcuda)
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
inline EncodeTiledFn encode_tiled() {
  static EncodeTiledFn fn = [] {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) != cudaSuccess ||
        qres != cudaDriverEntryPointSuccess)
      ptr = nullptr;
    return reinterpret_cast<EncodeTiledFn>(ptr);
  }();
  return fn;
}

// The coefficient array as a 3-D tensor [B][K][10 D] of doubles with a {10 D, 1, 16} box.
inline bool make_coeff_map(CUtensorMap* map, double* coeffs, long B, int K, int D) {
  EncodeTiledFn fn = encode_tiled();
  if (!fn || B > 0x7fffffffL) return false;
  const cuuint64_t dims[3] = {(cuuint64_t)(D * kN), (cuuint64_t)K, (cuuint64_t)B};
  const cuuint64_t strides[2] = {(cuuint64_t)(D * kN) * sizeof(double), (cuuint64_t)K * D * kN * sizeof(double)};
  const cuuint32_t box[3] = {(cuuint32_t)(D * kN), 1u, (cuuint32_t)kPairsPerWarp};
  const cuuint32_t estr[3] = {1u, 1u, 1u};
  return fn(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 3, coeffs, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// cudaErrorNotSupported: no tensor map could be made; the caller takes the first-generation kernel.
template <int D>
inline cudaError_t launch_d(FastParams p, cudaStream_t stream) {
  const size_t smem = WarpSmem<D>(p.K).total * sizeof(double) * kWarpsPerCta;
  if (smem > kMaxDynamicSmem) return cudaErrorNotSupported;
  CUtensorMap map;
  if (!make_coeff_map(&map, p.coeffs, p.B, p.K, D)) return cudaErrorNotSupported;
  const int cols = tmem_columns<D>(p.K);
  const bool extras = p.end_derivatives || p.free_out;
  void (*kernel)(FastParams, int, int, const CUtensorMap, int);
  if (p.K & 1)
    kernel = extras ? (p.cost ? solve_standard_tm_kernel<D, true, true, true> : solve_standard_tm_kernel<D, false, true, true>)
                    : (p.cost ? solve_standard_tm_kernel<D, true, false, true> : solve_standard_tm_kernel<D, false, false, true>);
  else
    kernel = extras ? (p.cost ? solve_standard_tm_kernel<D, true, true> : solve_standard_tm_kernel<D, false, true>)
                    : (p.cost ? solve_standard_tm_kernel<D, true, false> : solve_standard_tm_kernel<D, false, false>);
  cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  const long per_cta = (long)kWarpsPerCta * kPairsPerWarp;
  const long need = (p.B + per_cta - 1) / per_cta;   // CTAs at one batch of 16 trajectories per warp
  int dev = 0, sms = 148, ctas = 2;
  if (cudaGetDevice(&dev) == cudaSuccess) cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  {
    // resident CTAs per SM from the three resources themselves (the occupancy query answers for the current
    // shared-memory carve-out, not for the one the launch will get)
    cudaFuncAttributes fa;
    int regs_per_sm = 65536, smem_per_sm = 228 * 1024;
    cudaDeviceGetAttribute(&regs_per_sm, cudaDevAttrMaxRegistersPerMultiprocessor, dev);
    cudaDeviceGetAttribute(&smem_per_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
    ctas = 512 / cols;   // tensor memory: 512 columns per SM
    if (cudaFuncGetAttributes(&fa, kernel) == cudaSuccess && fa.numRegs > 0) {
      const int regs_per_cta = ((fa.numRegs + 7) / 8 * 8) * kWarpsPerCta * 32;
      ctas = std::min(ctas, regs_per_sm / regs_per_cta);
      ctas = std::min(ctas, (int)(smem_per_sm / (smem + fa.sharedSizeBytes + 1024)));
    }
    if (ctas < 1) ctas = 1;
  }
  // Above two waves of CTAs a warp takes kBatchesPerWarp batches (the second arrives in the other input
  // buffer during the first; allocation, table, barrier and the final drain are paid once), and the grid stays a
  // whole number of waves so that every resident slot ends up with the same number of batches, give or take
  // one, as under one-batch CTAs: 65,536 solves, grid 1,024 -> 592: 43.2 -> 42.2 us.  (Grids that are not a
  // multiple of the slots lose to quantisation: 512 CTAs 47.3 us, 342 CTAs 55.8 us.)
  constexpr long kBatchesPerWarp = 2;
  const long slots = (long)sms * ctas;
  long grid = need;
  if (need > 2 * slots) {
    const long waves = (need + slots - 1) / slots;
    grid = slots * ((waves + kBatchesPerWarp - 1) / kBatchesPerWarp);
    if (grid > need) grid = need;
  }
  // MINSNAP_TM_PDL=0 switches programmatic dependent launch off: back-to-back launches may deadlock under it while
  // launch_dependents precedes tcgen05.alloc (dependent CTAs can take the tensor memory a predecessor CTA waits for)
  static const int pdl = [] { const char* v = std::getenv("MINSNAP_TM_PDL"); return v ? std::atoi(v) : 1; }();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(kWarpsPerCta * 32);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = pdl ? 1 : 0;
  return cudaLaunchKernelEx(&cfg, kernel, p, cols, sms * ctas * kWarpsPerCta, map, pdl);
}

}  // namespace tm
}  // namespace minsnap
