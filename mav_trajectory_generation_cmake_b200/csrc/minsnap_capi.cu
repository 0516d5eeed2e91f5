// C ABI of libminsnap_b200.so (declared in include/minsnap_b200.h): argument checking,
// workspace carving, stream-ordered scratch memory and the host-buffer pipelines.  No
// arithmetic of the hot path happens here -- every number comes out of a CUDA kernel.
#include "../../include/minsnap_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "minsnap_launch.h"

namespace {

thread_local char g_last_cuda_error[256] = "";

int cuda_fail(cudaError_t e, const char* what) {
  std::snprintf(g_last_cuda_error, sizeof(g_last_cuda_error), "%s: %s (%s)", what, cudaGetErrorName(e),
                cudaGetErrorString(e));
  if (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) return MINSNAP_ERR_NO_DEVICE;
  if (e == cudaErrorInvalidConfiguration) return MINSNAP_ERR_UNSUPPORTED;
  return MINSNAP_ERR_CUDA;
}

#define CU(call)                                        \
  do {                                                  \
    cudaError_t e__ = (call);                           \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

inline cudaStream_t as_stream(minsnap_stream_t s) { return static_cast<cudaStream_t>(s); }

inline size_t align_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct SolveWorkspace {
  uint8_t* mask;
  int32_t* col_of_row;
  int32_t* counts;
  static size_t bytes(int N, int K) {
    return align_up((size_t)(K + 1) * (N / 2), 16) + align_up(sizeof(int32_t) * (size_t)N * K, 16) + 16;
  }
  SolveWorkspace(void* base, int N, int K) {
    char* p = static_cast<char*>(base);
    mask = reinterpret_cast<uint8_t*>(p);
    p += align_up((size_t)(K + 1) * (N / 2), 16);
    col_of_row = reinterpret_cast<int32_t*>(p);
    p += align_up(sizeof(int32_t) * (size_t)N * K, 16);
    counts = reinterpret_cast<int32_t*>(p);
  }
};

bool shape_ok(long B, int K, int D, int N, int derivative) {
  return B >= 0 && K >= 1 && D >= 1 && minsnap::supported_n(N) && derivative >= 0 && derivative <= N / 2 - 1;
}

void count_mask(const uint8_t* mask, int N, int K, int* n_fixed, int* n_free) {
  int f = 0;
  const int nc = (K + 1) * (N / 2);
  for (int i = 0; i < nc; ++i) f += mask[i] != 0;
  *n_fixed = f;
  *n_free = nc - f;
}

// Keep freed scratch memory in the device pool so that repeated host-API calls do not pay
// for cudaMalloc each time.  Side effect, on purpose and process-wide: the release threshold of the
// device's DEFAULT memory pool is raised to "never trim" (documented in INTEGRATION.md).
void retain_pool_memory() {
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return;
  // once per thread and device: the attribute call is not a capturable operation, and a caller that captures a
  // host-API-free entry point into a CUDA graph has run it eagerly before
  static thread_local int done_for = -1;
  if (done_for == dev) return;
  done_for = dev;
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, dev) != cudaSuccess) return;
  uint64_t threshold = ~0ull;
  cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &threshold);
}

// ---------------------------------------------------------------------------------------
// Small host calls (one trajectory from the C++ drop-in classes): a thread-local staging arena
// -- one pinned host block and one device block of equal size, grown on demand, released when
// the thread exits -- turns a call into: pack inputs -> ONE H2D copy -> kernels -> ONE D2H copy
// -> unpack.  No cudaMalloc, no stream creation, no pageable-memory copies on the way.
// (The only state kept between calls is this cache of CUDA resources, private to the thread.)
// ---------------------------------------------------------------------------------------
constexpr size_t kSmallCallBytes = 4u << 20;

struct HostArena {
  char* h = nullptr;
  char* d = nullptr;
  size_t cap = 0;
  int device = -1;
  ~HostArena() { release(); }
  void release() {
    if (h) cudaFreeHost(h);
    if (d) cudaFree(d);
    h = d = nullptr;
    cap = 0;
  }
  cudaError_t ensure(size_t bytes) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev == device && bytes <= cap) return cudaSuccess;
    release();
    size_t want = 64u << 10;
    while (want < bytes) want <<= 1;
    if ((e = cudaHostAlloc(reinterpret_cast<void**>(&h), want, cudaHostAllocDefault)) != cudaSuccess) return e;
    if ((e = cudaMalloc(reinterpret_cast<void**>(&d), want)) != cudaSuccess) return e;
    cap = want;
    device = dev;
    return cudaSuccess;
  }
};
thread_local HostArena g_arena;

// Large host calls (minsnap_solve_standard_host and friends): a thread-local copy/solve/copy pipeline
// of kDepth stages.  Each stage owns a non-blocking stream and one device block; chunk c runs
// H2D -> kernel -> D2H on stream c % kDepth, so that H2D(c+1), the kernel of chunk c and D2H(c-1)
// overlap on the two copy engines and the SMs, and a stage's block is reused in stream order.  The
// streams and blocks are created on first use and kept for the life of the thread (round 1 created
// two streams and fourteen pool allocations on every call).
struct HostPipeline {
  static constexpr int kDepth = 3;
  cudaStream_t stream[kDepth] = {nullptr, nullptr, nullptr};
  char* block[kDepth] = {nullptr, nullptr, nullptr};
  size_t cap = 0;
  int device = -1;
  ~HostPipeline() { release(); }
  void release() {
    for (int i = 0; i < kDepth; ++i) {
      if (block[i]) cudaFree(block[i]);
      if (stream[i]) cudaStreamDestroy(stream[i]);
      block[i] = nullptr;
      stream[i] = nullptr;
    }
    cap = 0;
    device = -1;
  }
  cudaError_t ensure(size_t bytes_per_stage) {
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev != device) release();
    for (int i = 0; i < kDepth; ++i)
      if (!stream[i] && (e = cudaStreamCreateWithFlags(&stream[i], cudaStreamNonBlocking)) != cudaSuccess) return e;
    device = dev;
    if (bytes_per_stage <= cap) return cudaSuccess;
    for (int i = 0; i < kDepth; ++i) {
      if (stream[i] && (e = cudaStreamSynchronize(stream[i])) != cudaSuccess) return e;
      if (block[i]) cudaFree(block[i]);
      block[i] = nullptr;
    }
    cap = 0;
    const size_t want = align_up(bytes_per_stage, 1u << 20);
    for (int i = 0; i < kDepth; ++i)
      if ((e = cudaMalloc(reinterpret_cast<void**>(&block[i]), want)) != cudaSuccess) return e;
    cap = want;
    return cudaSuccess;
  }
};
thread_local HostPipeline g_pipeline;

// One host-buffer call.  The buffers are declared first -- inputs with their host source, outputs with their
// host destination (NULL: device-only, not copied back), device-only scratch -- and run() stages them: through
// the thread's pinned arena with ONE copy each way when the call is small (a trajectory from the C++ drop-in
// classes), through stream-ordered allocations with one copy per buffer when it is large; it then invokes the
// device-pointer entry point on the thread's stream and waits.  Every *_host entry point is this pattern.
class HostCall {
 public:
  HostCall() : st_(cudaStreamPerThread) {}
  ~HostCall() {
    for (auto* v : {&ins_, &outs_, &tmps_})
      for (auto& b : *v)
        if (b.dptr) cudaFreeAsync(b.dptr, st_);
  }
  int in(const void* src, size_t bytes) { return add(ins_, const_cast<void*>(src), src ? bytes : 0); }
  int out(void* dst, size_t bytes) { return add(outs_, dst, bytes) + 1000; }
  int scratch(size_t bytes) { return add(tmps_, nullptr, bytes) + 2000; }
  template <typename T>
  T* dev(int id) const {
    const Buf& b = buf(id);
    return reinterpret_cast<T*>(small_ ? g_arena.d + b.off : static_cast<char*>(b.dptr));
  }
  // device pointer of an optional buffer: NULL when the caller passed no host pointer for it
  template <typename T>
  T* dev_if(int id, const void* host) const { return host ? dev<T>(id) : nullptr; }

  template <typename F>
  int run(F&& launch) {
    size_t off = 0;
    for (auto& b : ins_) { b.off = off; off += pad(b.bytes); }
    in_end_ = off;
    for (auto& b : outs_) { b.off = off; off += pad(b.bytes); }
    out_end_ = off;
    for (auto& b : tmps_) { b.off = off; off += pad(b.bytes); }
    small_ = off <= kSmallCallBytes;
    if (small_) {
      CU(g_arena.ensure(off ? off : 16));
      for (auto& b : ins_)
        if (b.host && b.bytes) std::memcpy(g_arena.h + b.off, b.host, b.bytes);
      if (in_end_ > 0) CU(cudaMemcpyAsync(g_arena.d, g_arena.h, in_end_, cudaMemcpyHostToDevice, st_));
      const int rc = launch(st_);
      if (rc != MINSNAP_OK) return rc;
      if (out_end_ > in_end_)
        CU(cudaMemcpyAsync(g_arena.h + in_end_, g_arena.d + in_end_, out_end_ - in_end_, cudaMemcpyDeviceToHost, st_));
      CU(cudaStreamSynchronize(st_));
      for (auto& b : outs_)
        if (b.host && b.bytes) std::memcpy(b.host, g_arena.h + b.off, b.bytes);
      return MINSNAP_OK;
    }
    retain_pool_memory();   // freed blocks stay in the device's default pool between calls (process-wide setting)
    int rc = MINSNAP_OK;
    for (auto* v : {&ins_, &outs_, &tmps_})
      for (auto& b : *v) {
        const cudaError_t e = cudaMallocAsync(&b.dptr, b.bytes ? b.bytes : 16, st_);
        if (e != cudaSuccess) return cuda_fail(e, "cudaMallocAsync");
      }
    for (auto& b : ins_)
      if (b.host && b.bytes) {
        const cudaError_t e = cudaMemcpyAsync(b.dptr, b.host, b.bytes, cudaMemcpyHostToDevice, st_);
        if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync(H2D)"); break; }
      }
    if (rc == MINSNAP_OK) rc = launch(st_);
    if (rc == MINSNAP_OK)
      for (auto& b : outs_)
        if (b.host && b.bytes) {
          const cudaError_t e = cudaMemcpyAsync(b.host, b.dptr, b.bytes, cudaMemcpyDeviceToHost, st_);
          if (e != cudaSuccess) { rc = cuda_fail(e, "cudaMemcpyAsync(D2H)"); break; }
        }
    const cudaError_t es = cudaStreamSynchronize(st_);
    if (rc == MINSNAP_OK && es != cudaSuccess) rc = cuda_fail(es, "cudaStreamSynchronize");
    return rc;
  }
  // after run(): the first `bytes` of a device-only output (an output declared with a NULL host pointer)
  int fetch(int id, void* dst, size_t bytes) const {
    if (bytes == 0) return MINSNAP_OK;
    const Buf& b = buf(id);
    if (small_) {
      std::memcpy(dst, g_arena.h + b.off, bytes);
      return MINSNAP_OK;
    }
    CU(cudaMemcpyAsync(dst, b.dptr, bytes, cudaMemcpyDeviceToHost, st_));
    CU(cudaStreamSynchronize(st_));
    return MINSNAP_OK;
  }

 private:
  struct Buf {
    void* host;
    size_t bytes, off;
    void* dptr;
  };
  static size_t pad(size_t b) { return (b + 255) & ~size_t(255); }
  static int add(std::vector<Buf>& v, void* host, size_t bytes) {
    v.push_back(Buf{host, bytes, 0, nullptr});
    return static_cast<int>(v.size()) - 1;
  }
  const Buf& buf(int id) const { return id >= 2000 ? tmps_[id - 2000] : id >= 1000 ? outs_[id - 1000] : ins_[id]; }
  cudaStream_t st_;
  std::vector<Buf> ins_, outs_, tmps_;
  size_t in_end_ = 0, out_end_ = 0;
  bool small_ = true;
};

}  // namespace

extern "C" {

int minsnap_abi_version(void) { return 1; }

const char* minsnap_error_string(int code) {
  switch (code) {
    case MINSNAP_OK: return "ok";
    case MINSNAP_ERR_ARG: return "invalid argument";
    case MINSNAP_ERR_CUDA: return "CUDA runtime error";
    case MINSNAP_ERR_UNSUPPORTED: return "unsupported shape";
    case MINSNAP_ERR_NO_DEVICE: return "no usable CUDA device";
    case MINSNAP_ERR_WORKSPACE: return "workspace missing or too small";
    default: return "unknown error";
  }
}

const char* minsnap_last_cuda_error(void) { return g_last_cuda_error; }

int minsnap_device_info(int* device, int* sm_count, int* cc_major, int* cc_minor, size_t* global_mem_bytes) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) return cuda_fail(e, "cudaGetDeviceCount");
  if (n == 0) return MINSNAP_ERR_NO_DEVICE;
  int dev = 0;
  CU(cudaGetDevice(&dev));
  cudaDeviceProp prop;
  CU(cudaGetDeviceProperties(&prop, dev));
  if (device) *device = dev;
  if (sm_count) *sm_count = prop.multiProcessorCount;
  if (cc_major) *cc_major = prop.major;
  if (cc_minor) *cc_minor = prop.minor;
  if (global_mem_bytes) *global_mem_bytes = prop.totalGlobalMem;
  return MINSNAP_OK;
}

int minsnap_reorder(int N, int K, long n_masks, const uint8_t* d_mask, int32_t* d_col_of_row, int32_t* d_counts,
                    minsnap_stream_t stream) {
  if (!minsnap::supported_n(N) || K < 1 || n_masks < 0 || !d_mask || !d_col_of_row || !d_counts)
    return MINSNAP_ERR_ARG;
  if (n_masks == 0) return MINSNAP_OK;
  CU(minsnap::launch_reorder(N, K, n_masks, d_mask, d_col_of_row, d_counts, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_estimate_segment_times(long B, int K, int D, const double* d_positions, double v_max, double a_max,
                                   double magic, double* d_times, minsnap_stream_t stream) {
  if (B < 0 || K < 1 || D < 1 || !d_positions || !d_times) return MINSNAP_ERR_ARG;
  CU(minsnap::launch_estimate_times(B, K, D, d_positions, v_max, a_max, magic, d_times, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_segment_matrices(long n, int N, int derivative, const double* d_T, double* d_A, double* d_Ainv,
                             double* d_Q, double* d_H, minsnap_stream_t stream) {
  if (n < 0 || !minsnap::supported_n(N) || derivative < 0 || derivative > N / 2 - 1 || !d_T) return MINSNAP_ERR_ARG;
  CU(minsnap::launch_segment_matrices(n, N, derivative, d_T, d_A, d_Ainv, d_Q, d_H, as_stream(stream)));
  return MINSNAP_OK;
}

size_t minsnap_solve_workspace_bytes(int N, int K) {
  if (!minsnap::supported_n(N) || K < 1) return 0;
  return SolveWorkspace::bytes(N, K);
}

static int general_common(bool solve, long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                          const double* d_fixed_values, const double* d_free_in, const double* d_times,
                          double* d_coeffs, double* d_free_out, double* d_cost, int32_t* d_status,
                          int32_t* d_col_of_row, void* d_workspace, size_t workspace_bytes, cudaStream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || !h_fixed_mask) return MINSNAP_ERR_ARG;
  if (B > 0 && (!d_times || !d_coeffs)) return MINSNAP_ERR_ARG;
  if (!d_workspace || workspace_bytes < SolveWorkspace::bytes(N, K)) return MINSNAP_ERR_WORKSPACE;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (B > 0 && n_fixed > 0 && !d_fixed_values) return MINSNAP_ERR_ARG;
  if (B > 0 && !solve && n_free > 0 && !d_free_in) return MINSNAP_ERR_ARG;
  SolveWorkspace ws(d_workspace, N, K);
  CU(cudaMemcpyAsync(ws.mask, h_fixed_mask, (size_t)(K + 1) * (N / 2), cudaMemcpyHostToDevice, stream));
  CU(minsnap::launch_reorder(N, K, 1, ws.mask, ws.col_of_row, ws.counts, stream));
  if (d_col_of_row)
    CU(cudaMemcpyAsync(d_col_of_row, ws.col_of_row, sizeof(int32_t) * (size_t)N * K, cudaMemcpyDeviceToDevice,
                       stream));
  minsnap::GeneralSolveArgs a;
  a.B = B; a.K = K; a.D = D; a.N = N; a.derivative = derivative; a.n_fixed = n_fixed; a.n_free = n_free;
  a.d_col_of_row = ws.col_of_row; a.d_fixed_values = d_fixed_values; a.d_free_in = d_free_in;
  a.d_times = d_times; a.d_coeffs = d_coeffs; a.d_free_out = d_free_out; a.d_cost = d_cost;
  a.d_status = d_status;
  if (solve) CU(minsnap::launch_solve_general(a, stream));
  else CU(minsnap::launch_coeffs_from_constraints(a, stream));
  return MINSNAP_OK;
}

int minsnap_solve(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                  const double* d_fixed_values, const double* d_times, double* d_coeffs, double* d_free_values,
                  double* d_cost, int32_t* d_status, int32_t* d_col_of_row, void* d_workspace,
                  size_t workspace_bytes, minsnap_stream_t stream) {
  return general_common(true, B, K, D, N, derivative, h_fixed_mask, d_fixed_values, nullptr, d_times, d_coeffs,
                        d_free_values, d_cost, d_status, d_col_of_row, d_workspace, workspace_bytes,
                        as_stream(stream));
}

int minsnap_coeffs_from_constraints(long B, int K, int D, int N, const uint8_t* h_fixed_mask,
                                    const double* d_fixed_values, const double* d_free_values,
                                    const double* d_times, double* d_coeffs, void* d_workspace,
                                    size_t workspace_bytes, minsnap_stream_t stream) {
  return general_common(false, B, K, D, N, 0, h_fixed_mask, d_fixed_values, d_free_values, d_times, d_coeffs,
                        nullptr, nullptr, nullptr, nullptr, d_workspace, workspace_bytes, as_stream(stream));
}

int minsnap_cost(long B, int K, int D, int N, int derivative, const double* d_coeffs, const double* d_times,
                 double* d_cost, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || !d_cost) return MINSNAP_ERR_ARG;
  CU(minsnap::launch_cost(B, K, D, N, derivative, d_coeffs, d_times, d_cost, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_solve_standard(long B, int K, int D, int N, int derivative, const double* d_positions,
                           const double* d_end_derivatives, const double* d_times, double v_max, double a_max,
                           double magic, double* d_times_out, double* d_coeffs, double* d_free_values,
                           double* d_cost, int32_t* d_status, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;   // empty batch: nothing to read or write
  if (!d_positions || !d_coeffs) return MINSNAP_ERR_ARG;
  if (!d_times && !(v_max > 0.0 && a_max > 0.0)) return MINSNAP_ERR_ARG;
  minsnap::StandardSolveArgs a;
  a.B = B; a.K = K; a.D = D; a.N = N; a.derivative = derivative;
  a.d_positions = d_positions; a.d_end_derivatives = d_end_derivatives; a.d_times = d_times;
  a.v_max = v_max; a.a_max = a_max; a.magic = magic; a.d_times_out = d_times_out;
  a.d_coeffs = d_coeffs; a.d_free_out = d_free_values; a.d_cost = d_cost; a.d_status = d_status;
  // MINSNAP_STANDARD_ROUTE=tm|pair|pair_long|bcr|chunked|general runs that kernel, so that tests can compare two
  // kernels on the same inputs: MINSNAP_ERR_UNSUPPORTED where it cannot take the call, never another kernel;
  // MINSNAP_ERR_ARG for an unknown name.
  if (const char* name = std::getenv("MINSNAP_STANDARD_ROUTE")) {
    for (int r = 0; r < static_cast<int>(minsnap::StandardRoute::Unsupported); ++r)
      if (std::strcmp(name, minsnap::standard_route_name(static_cast<minsnap::StandardRoute>(r))) == 0)
        a.forced = static_cast<minsnap::StandardRoute>(r);
    if (!a.forced) return MINSNAP_ERR_ARG;
  }
  const cudaError_t e = minsnap::launch_solve_standard(a, as_stream(stream));
  if (e == cudaErrorNotSupported && a.forced) return MINSNAP_ERR_UNSUPPORTED;
  CU(e);
  return MINSNAP_OK;
}

int minsnap_sample_uniform(long B, int K, int D, int N, const double* d_coeffs, const double* d_times, int M,
                           int n_deriv, double* d_out, double* d_t_out, minsnap_stream_t stream) {
  if (B < 0 || K < 1 || D < 1 || !minsnap::supported_n(N) || M < 0 || n_deriv < 1) return MINSNAP_ERR_ARG;
  if (B == 0 || M == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || !d_out) return MINSNAP_ERR_ARG;
  minsnap::SampleArgs a;
  a.B = B; a.K = K; a.D = D; a.N = N; a.M = M; a.n_deriv = n_deriv;
  a.d_coeffs = d_coeffs; a.d_times = d_times; a.d_t = nullptr; a.t_stride = 0;
  a.d_out = d_out; a.d_t_out = d_t_out; a.d_segment = nullptr;
  CU(minsnap::launch_sample(a, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_sample_at(long B, int K, int D, int N, const double* d_coeffs, const double* d_times, int M,
                      const double* d_t, long t_stride, int n_deriv, double* d_out, int32_t* d_segment,
                      minsnap_stream_t stream) {
  if (B < 0 || K < 1 || D < 1 || !minsnap::supported_n(N) || M < 0 || n_deriv < 1 || (t_stride != 0 && t_stride < M))
    return MINSNAP_ERR_ARG;
  if (B == 0 || M == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || !d_t || !d_out) return MINSNAP_ERR_ARG;
  minsnap::SampleArgs a;
  a.B = B; a.K = K; a.D = D; a.N = N; a.M = M; a.n_deriv = n_deriv;
  a.d_coeffs = d_coeffs; a.d_times = d_times; a.d_t = d_t; a.t_stride = t_stride;
  a.d_out = d_out; a.d_t_out = nullptr; a.d_segment = d_segment;
  CU(minsnap::launch_sample(a, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_evaluate_range(long B, int K, int D, int N, const double* d_coeffs, const double* d_times,
                           double t_start, double t_end, double dt, int derivative, int max_samples,
                           double* d_out, double* d_t_out, int32_t* d_count, minsnap_stream_t stream) {
  if (B < 0 || K < 1 || D < 1 || !minsnap::supported_n(N) || !(dt > 0.0) || derivative < 0 || max_samples < 0)
    return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;   // empty batch: nothing to read or write
  if (!d_coeffs || !d_times || !d_out) return MINSNAP_ERR_ARG;
  CU(minsnap::launch_evaluate_range(B, K, D, N, d_coeffs, d_times, t_start, t_end, dt, derivative, max_samples,
                                    d_out, d_t_out, d_count, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_cost_sweep(long B, int S, int K, int D, int N, int derivative, const double* d_positions,
                       const double* d_end_derivatives, const double* d_times, double* d_cost, int32_t* d_status,
                       minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || S < 1 || !d_positions || !d_times || !d_cost) return MINSNAP_ERR_ARG;
  minsnap::SweepArgs a;
  a.B = B; a.S = S; a.K = K; a.D = D; a.N = N; a.derivative = derivative;
  a.d_positions = d_positions; a.d_end_derivatives = d_end_derivatives; a.d_times = d_times;
  a.d_cost = d_cost; a.d_status = d_status;
  CU(minsnap::launch_cost_sweep(a, as_stream(stream)));
  return MINSNAP_OK;
}

// SURVEY 8(f)1: extrema of |p^(k)| (ref LIN.i:470-503, src/trajectory.cpp:181-217)
static bool extrema_args_ok(long B, int K, int D, int N, int derivative, int mode, uint32_t* dim_mask) {
  const int base = mode & ~MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS;
  if (B < 0 || K < 1 || D < 1 || D > 32 || !minsnap::supported_n(N) || derivative < 0 || derivative > N - 2 ||
      (base != MINSNAP_EXTREMA_OPTIMIZATION && base != MINSNAP_EXTREMA_TRAJECTORY))
    return false;
  const uint32_t all = D == 32 ? 0xffffffffu : ((1u << D) - 1u);
  if (*dim_mask == 0) *dim_mask = all;
  return (*dim_mask & ~all) == 0;
}

int minsnap_extrema_max_roots(int N, int derivative, int n_dims) {
  if (!minsnap::supported_n(N) || derivative < 0 || derivative > N - 2 || n_dims < 1) return 0;
  return minsnap::extrema_max_roots(N, derivative, n_dims);
}

int minsnap_extrema(long B, int K, int D, int N, const double* d_coeffs, const double* d_times, int derivative,
                    int mode, uint32_t dim_mask, double* d_max_time, double* d_max_value, int32_t* d_max_segment,
                    double* d_min_time, double* d_min_value, int32_t* d_min_segment, double* d_cand_times,
                    double* d_cand_values, int32_t* d_root_count, minsnap_stream_t stream) {
  if (!extrema_args_ok(B, K, D, N, derivative, mode, &dim_mask)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times) return MINSNAP_ERR_ARG;
  minsnap::ExtremaArgs a;
  a.B = B; a.K = K; a.D = D; a.N = N; a.derivative = derivative;
  a.mode = mode & ~MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS;
  a.keep_small = (mode & MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS) != 0;
  a.dim_mask = dim_mask;
  a.d_coeffs = d_coeffs; a.d_times = d_times;
  a.d_max_time = d_max_time; a.d_max_value = d_max_value; a.d_max_segment = d_max_segment;
  a.d_min_time = d_min_time; a.d_min_value = d_min_value; a.d_min_segment = d_min_segment;
  a.d_cand_times = d_cand_times; a.d_cand_values = d_cand_values; a.d_root_count = d_root_count;
  a.max_roots = minsnap::extrema_max_roots(N, derivative, __builtin_popcount(dim_mask));
  CU(minsnap::launch_extrema(a, as_stream(stream)));
  return MINSNAP_OK;
}

// SURVEY 8(f)2: time-only objective (ref NL.i:765-832) and numeric time gradient (ref NL.i:2155-2243)
int minsnap_time_objective(long B, int S, int K, int D, int N, int derivative, const double* d_positions,
                           const double* d_end_derivatives, const double* d_times, double time_penalty,
                           double* d_objective, double* d_cost, int32_t* d_status, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || S < 1) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!d_positions || !d_times || !d_objective) return MINSNAP_ERR_ARG;
  // the cost lands in d_cost when given, else in d_objective, and is completed in place
  double* cost = d_cost ? d_cost : d_objective;
  const int rc = minsnap_cost_sweep(B, S, K, D, N, derivative, d_positions, d_end_derivatives, d_times, cost, d_status,
                                    stream);
  if (rc != MINSNAP_OK) return rc;
  CU(minsnap::launch_add_time_penalty(B * S, K, d_times, cost, time_penalty, d_objective, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_time_gradient(long B, int K, int D, int N, int derivative, const double* d_coeffs, const double* d_times,
                          double increment, double w_d, double w_t, double* d_gradient, double* d_segment_cost,
                          minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || !(increment > 0.0)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || (!d_gradient && !d_segment_cost)) return MINSNAP_ERR_ARG;
  CU(minsnap::launch_time_gradient(B, K, D, N, derivative, d_coeffs, d_times, increment, w_d, w_t, d_gradient,
                                   d_segment_cost, as_stream(stream)));
  return MINSNAP_OK;
}

// SURVEY 8(f)2: a batched descent on the segment times that never leaves the device.  Every iteration is five
// launches on `stream` (solve, time gradient, step ladder, cost sweep over the ladder, select); the workspace is
// one stream-ordered allocation.
int minsnap_optimize_segment_times(long B, int K, int D, int N, int derivative, const double* d_positions,
                                   const double* d_end_derivatives, double* d_times, int iterations, double time_penalty,
                                   int n_steps, double max_relative_step, double min_time, double gradient_increment,
                                   double* d_history, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || iterations < 0 || n_steps < 1 || !(max_relative_step > 0.0) ||
      !(min_time > 0.0) || !(gradient_increment > 0.0))
    return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!d_positions || !d_times) return MINSNAP_ERR_ARG;
  if (!minsnap::standard_supported(K, D, N, derivative)) return MINSNAP_ERR_UNSUPPORTED;
  cudaStream_t st = as_stream(stream);
  const size_t nb = (size_t)B, S = (size_t)n_steps;
  const size_t n_coeffs = nb * K * D * N, n_grad = nb * K, n_cand = nb * S * K, n_cost = nb * S;
  double* ws = nullptr;
  retain_pool_memory();
  CU(cudaMallocAsync(reinterpret_cast<void**>(&ws), sizeof(double) * (n_coeffs + n_grad + n_cand + n_cost + nb), st));
  double* coeffs = ws;
  double* grad = coeffs + n_coeffs;
  double* cand = grad + n_grad;
  double* cost = cand + n_cand;
  double* incumbent = cost + n_cost;
  int rc = MINSNAP_OK;
  // the incumbent objective at the initial times: one allocation per trajectory through the same sweep + penalty
  rc = minsnap_time_objective(B, 1, K, D, N, derivative, d_positions, d_end_derivatives, d_times, time_penalty, incumbent,
                              nullptr, nullptr, st);
  if (rc == MINSNAP_OK && d_history)
    if (cudaMemcpyAsync(d_history, incumbent, sizeof(double) * nb, cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = MINSNAP_ERR_CUDA;
  for (int it = 0; it < iterations && rc == MINSNAP_OK; ++it) {
    rc = minsnap_solve_standard(B, K, D, N, derivative, d_positions, d_end_derivatives, d_times, 0.0, 0.0, 0.0, nullptr,
                                coeffs, nullptr, nullptr, nullptr, st);
    // d cost / dT = 0.5 dJ_d/dT (w_d = 0.5, w_t = 0); the penalty's gradient is added by the ladder kernel
    if (rc == MINSNAP_OK) rc = minsnap_time_gradient(B, K, D, N, derivative, coeffs, d_times, gradient_increment, 0.5, 0.0, grad, nullptr, st);
    cudaError_t e = cudaSuccess;
    if (rc == MINSNAP_OK) e = minsnap::launch_time_candidates(B, n_steps, K, d_times, grad, time_penalty, max_relative_step, min_time, cand, st);
    if (rc == MINSNAP_OK && e == cudaSuccess)
      rc = minsnap_cost_sweep(B, n_steps, K, D, N, derivative, d_positions, d_end_derivatives, cand, cost, nullptr, st);
    if (rc == MINSNAP_OK && e == cudaSuccess)
      e = minsnap::launch_time_select(B, n_steps, K, cand, cost, time_penalty, d_times, incumbent,
                                      d_history ? d_history + (size_t)(it + 1) * nb : nullptr, st);
    if (rc == MINSNAP_OK && e != cudaSuccess) rc = cuda_fail(e, "time descent glue");
  }
  cudaFreeAsync(ws, st);
  return rc;
}

// ---------------------------------------------------------------------------------------
// The time-only objective with the reference's soft limits on max |p^(k)| (ref objectiveFunctionTime with
// use_soft_constraints NL.i:765-832, evaluateMaximumMagnitudeAsSoftConstraint NL.i:2396-2426,
// evaluateMaximumMagnitudeConstraint NL.i:2346-2392)
// ---------------------------------------------------------------------------------------
namespace {

// The constraint arguments shared by the three entries, checked and copied into the launcher's arguments.
int soft_args(int N, int n_constraints, const int32_t* h_derivatives, const double* h_limits, double weight,
              double maximum_cost, int extrema_flags, minsnap::SoftConstraintArgs* a) {
  if (n_constraints < 1 || n_constraints > minsnap::kMaxSoftConstraints || !h_derivatives || !h_limits ||
      !(weight > 0.0 && std::isfinite(weight)) || !(maximum_cost > 0.0 && std::isfinite(maximum_cost)) ||
      (extrema_flags != 0 && extrema_flags != MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS))
    return MINSNAP_ERR_ARG;
  a->n_constraints = n_constraints;
  for (int c = 0; c < n_constraints; ++c) {
    if (h_derivatives[c] < 0 || h_derivatives[c] > N - 2 || !(h_limits[c] > 0.0 && std::isfinite(h_limits[c])))
      return MINSNAP_ERR_ARG;
    a->derivative[c] = h_derivatives[c];
    a->limit[c] = h_limits[c];
  }
  a->weight = weight;
  a->maximum_cost = maximum_cost;
  a->keep_small = extrema_flags == MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS;
  return MINSNAP_OK;
}

// Scratch of the objective pipeline for up to n allocations: positions (and end derivatives) replicated per
// allocation, coefficients, computeCost, solve status, per-segment maxima.
struct SoftScratch {
  double* positions;
  double* end;
  double* coeffs;
  double* cost;
  int32_t* status;
  void* extrema;
  static size_t bytes(size_t n, int K, int D, int N, bool with_end, int n_constraints) {
    const size_t doubles = n * ((size_t)(K + 1) * D + (with_end ? (size_t)(N - 2) * D : 0) + (size_t)K * D * N + 1);
    return align_up(sizeof(double) * doubles + sizeof(int32_t) * n, 256) +
           minsnap::soft_constraint_scratch_bytes((long)n, K, n_constraints);
  }
  SoftScratch(void* base, size_t n, int K, int D, int N, bool with_end) {
    positions = static_cast<double*>(base);
    end = positions + n * (K + 1) * D;
    coeffs = end + (with_end ? n * (N - 2) * D : 0);
    cost = coeffs + n * K * D * N;
    status = reinterpret_cast<int32_t*>(cost + n);
    extrema = static_cast<char*>(base) + align_up(sizeof(double) * (size_t)(cost + n - positions) + sizeof(int32_t) * n, 256);
  }
};

// Solves the R allocations d_times [B R][K] of every trajectory (coefficients, and computeCost and status when
// want_cost) from its positions replicated R times.
int solve_replicated(long B, int R, int K, int D, int N, int derivative, const double* d_positions,
                     const double* d_end_derivatives, const double* d_times, bool want_cost, const SoftScratch& s,
                     cudaStream_t st) {
  CU(minsnap::launch_replicate_rows(B, R, (K + 1) * D, d_positions, s.positions, (N - 2) * D, d_end_derivatives, s.end,
                                    st));
  return minsnap_solve_standard(B * R, K, D, N, derivative, s.positions, d_end_derivatives ? s.end : nullptr, d_times,
                                0.0, 0.0, 0.0, nullptr, s.coeffs, nullptr, want_cost ? s.cost : nullptr,
                                want_cost ? s.status : nullptr, st);
}

// minsnap_time_objective_soft on the device: replicate, solve with cost and status, soft cost with the objective
// epilogue.  d_cost (optional) receives computeCost; without it the scratch holds it.
int soft_objective_device(long B, int S, int K, int D, int N, int derivative, const double* d_positions,
                          const double* d_end_derivatives, const double* d_times, double time_penalty,
                          minsnap::SoftConstraintArgs a, double* d_objective, double* d_cost, double* d_soft,
                          double* d_terms, const SoftScratch& s, cudaStream_t st) {
  SoftScratch sc = s;
  if (d_cost) sc.cost = d_cost;
  const int rc = solve_replicated(B, S, K, D, N, derivative, d_positions, d_end_derivatives, d_times, true, sc, st);
  if (rc != MINSNAP_OK) return rc;
  a.B = B * S; a.K = K; a.D = D; a.N = N;
  a.d_coeffs = sc.coeffs; a.d_times = d_times; a.d_scratch = sc.extrema;
  a.d_soft = d_soft; a.d_terms = d_terms; a.d_max_value = nullptr;
  a.d_objective = d_objective; a.d_cost = sc.cost; a.d_status = sc.status; a.time_penalty = time_penalty;
  CU(minsnap::launch_soft_constraint_cost(a, st));
  return MINSNAP_OK;
}

}  // namespace

int minsnap_soft_constraint_cost(long B, int K, int D, int N, const double* d_coeffs, const double* d_times,
                                 int n_constraints, const int32_t* h_derivatives, const double* h_limits, double weight,
                                 double maximum_cost, int extrema_flags, double* d_cost, double* d_terms,
                                 double* d_max_value, minsnap_stream_t stream) {
  if (B < 0 || K < 1 || D < 1 || D > 32 || !minsnap::supported_n(N)) return MINSNAP_ERR_ARG;
  minsnap::SoftConstraintArgs a;
  int rc = soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, &a);
  if (rc != MINSNAP_OK) return rc;
  if (B == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || !d_cost) return MINSNAP_ERR_ARG;
  cudaStream_t st = as_stream(stream);
  void* scratch = nullptr;
  retain_pool_memory();
  CU(cudaMallocAsync(&scratch, minsnap::soft_constraint_scratch_bytes(B, K, n_constraints), st));
  a.B = B; a.K = K; a.D = D; a.N = N;
  a.d_coeffs = d_coeffs; a.d_times = d_times; a.d_scratch = scratch;
  a.d_soft = d_cost; a.d_terms = d_terms; a.d_max_value = d_max_value;
  const cudaError_t e = minsnap::launch_soft_constraint_cost(a, st);
  if (e != cudaSuccess) rc = cuda_fail(e, "launch_soft_constraint_cost");
  cudaFreeAsync(scratch, st);
  return rc;
}

int minsnap_time_objective_soft(long B, int S, int K, int D, int N, int derivative, const double* d_positions,
                                const double* d_end_derivatives, const double* d_times, double time_penalty,
                                int n_constraints, const int32_t* h_derivatives, const double* h_limits, double weight,
                                double maximum_cost, int extrema_flags, double* d_objective, double* d_cost,
                                double* d_soft, double* d_terms, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || S < 1) return MINSNAP_ERR_ARG;
  minsnap::SoftConstraintArgs a;
  int rc = soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, &a);
  if (rc != MINSNAP_OK) return rc;
  if (B == 0) return MINSNAP_OK;
  if (!d_positions || !d_times || !d_objective) return MINSNAP_ERR_ARG;
  if (!minsnap::standard_supported(K, D, N, derivative)) return MINSNAP_ERR_UNSUPPORTED;
  cudaStream_t st = as_stream(stream);
  const size_t n = (size_t)B * S;
  const bool with_end = d_end_derivatives != nullptr;
  void* ws = nullptr;
  retain_pool_memory();
  CU(cudaMallocAsync(&ws, SoftScratch::bytes(n, K, D, N, with_end, n_constraints), st));
  const SoftScratch s(ws, n, K, D, N, with_end);
  rc = soft_objective_device(B, S, K, D, N, derivative, d_positions, d_end_derivatives, d_times, time_penalty, a,
                             d_objective, d_cost, d_soft, d_terms, s, st);
  cudaFreeAsync(ws, st);
  return rc;
}

// The descent of minsnap_optimize_segment_times on the objective with the soft terms, never leaving the device.
// Per iteration: solve at the incumbent, time gradient, 2K re-solved allocations per trajectory and their soft cost,
// the soft term's central difference added to the gradient, step ladder, the objective pipeline over the ladder,
// select.  Workspace (one stream-ordered allocation), with R = max(2K, n_steps) and n_c constraints:
//   8 B (R (K+1) D + R 2 (h-1) D [end derivatives given] + R K D N + R K + 3 R + K + 1) + 4 B R
//   + 32 B R K n_c bytes (+ alignment),
// 4.47 GB at B = 65,536, K = 10, n_steps = 16, D = 3, N = 10, two constraints, no end derivatives.
int minsnap_optimize_segment_times_soft(long B, int K, int D, int N, int derivative, const double* d_positions,
                                        const double* d_end_derivatives, double* d_times, int iterations,
                                        double time_penalty, int n_steps, double max_relative_step, double min_time,
                                        double gradient_increment, int n_constraints, const int32_t* h_derivatives,
                                        const double* h_limits, double weight, double maximum_cost, int extrema_flags,
                                        double* d_history, double* d_max_value, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || iterations < 0 || n_steps < 1 || !(max_relative_step > 0.0) ||
      !(min_time > 0.0) || !(gradient_increment > 0.0))
    return MINSNAP_ERR_ARG;
  minsnap::SoftConstraintArgs a;
  int rc = soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, &a);
  if (rc != MINSNAP_OK) return rc;
  if (B == 0) return MINSNAP_OK;
  if (!d_positions || !d_times) return MINSNAP_ERR_ARG;
  if (!minsnap::standard_supported(K, D, N, derivative)) return MINSNAP_ERR_UNSUPPORTED;
  cudaStream_t st = as_stream(stream);
  const size_t nb = (size_t)B, R = std::max<size_t>(2 * (size_t)K, (size_t)n_steps), n = nb * R;
  const bool with_end = d_end_derivatives != nullptr;
  const size_t head = align_up(SoftScratch::bytes(n, K, D, N, with_end, n_constraints), 256);
  char* ws = nullptr;
  retain_pool_memory();
  CU(cudaMallocAsync(reinterpret_cast<void**>(&ws), head + sizeof(double) * (n * K + 2 * n + nb * K + nb), st));
  const SoftScratch s(ws, n, K, D, N, with_end);
  double* cand = reinterpret_cast<double*>(ws + head);   // [B][R][K]: the 2K differences, then the ladder
  double* soft = cand + n * K;                          // [B][2K] soft cost of the differences
  double* obj = soft + n;                               // [B][n_steps] objective of the ladder
  double* grad = obj + n;
  double* incumbent = grad + nb * K;
  a.K = K; a.D = D; a.N = N;
  // the incumbent objective at the initial times: the candidate pipeline with one allocation per trajectory
  rc = soft_objective_device(B, 1, K, D, N, derivative, d_positions, d_end_derivatives, d_times, time_penalty, a,
                             incumbent, nullptr, nullptr, nullptr, s, st);
  if (rc == MINSNAP_OK && d_history)
    if (cudaMemcpyAsync(d_history, incumbent, sizeof(double) * nb, cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = MINSNAP_ERR_CUDA;
  for (int it = 0; it < iterations && rc == MINSNAP_OK; ++it) {
    rc = minsnap_solve_standard(B, K, D, N, derivative, d_positions, d_end_derivatives, d_times, 0.0, 0.0, 0.0, nullptr,
                                s.coeffs, nullptr, nullptr, nullptr, st);
    // d computeCost / dT = 0.5 dJ_d/dT (w_d = 0.5, w_t = 0), as minsnap_optimize_segment_times
    if (rc == MINSNAP_OK)
      rc = minsnap_time_gradient(B, K, D, N, derivative, s.coeffs, d_times, gradient_increment, 0.5, 0.0, grad, nullptr, st);
    cudaError_t e = cudaSuccess;
    if (rc == MINSNAP_OK) e = minsnap::launch_soft_gradient_candidates(B, K, d_times, gradient_increment, cand, st);
    if (rc == MINSNAP_OK && e == cudaSuccess)
      rc = solve_replicated(B, 2 * K, K, D, N, derivative, d_positions, d_end_derivatives, cand, false, s, st);
    if (rc == MINSNAP_OK && e == cudaSuccess) {
      minsnap::SoftConstraintArgs g = a;
      g.B = B * 2 * K; g.d_coeffs = s.coeffs; g.d_times = cand; g.d_scratch = s.extrema;
      g.d_soft = soft; g.d_terms = nullptr; g.d_max_value = nullptr;
      e = minsnap::launch_soft_constraint_cost(g, st);
    }
    if (rc == MINSNAP_OK && e == cudaSuccess) e = minsnap::launch_soft_gradient_add(B, K, soft, gradient_increment, grad, st);
    // the ladder adds the penalty's gradient 2 time_penalty sum(T)
    if (rc == MINSNAP_OK && e == cudaSuccess)
      e = minsnap::launch_time_candidates(B, n_steps, K, d_times, grad, time_penalty, max_relative_step, min_time, cand, st);
    if (rc == MINSNAP_OK && e == cudaSuccess)
      rc = soft_objective_device(B, n_steps, K, D, N, derivative, d_positions, d_end_derivatives, cand, time_penalty, a,
                                 obj, nullptr, nullptr, nullptr, s, st);
    // the first minimum among the finite objectives, accepted when strictly below the incumbent (no free values)
    if (rc == MINSNAP_OK && e == cudaSuccess)
      e = minsnap::launch_free_select(B, n_steps, 0, K, obj, nullptr, cand, nullptr, nullptr, d_times, incumbent, nullptr,
                                      d_history ? d_history + (size_t)(it + 1) * nb : nullptr, st);
    if (rc == MINSNAP_OK && e != cudaSuccess) rc = cuda_fail(e, "soft time descent glue");
  }
  // the maxima at the returned times, from the solve minsnap_solve_standard gives for this batch
  if (rc == MINSNAP_OK && d_max_value) {
    rc = minsnap_solve_standard(B, K, D, N, derivative, d_positions, d_end_derivatives, d_times, 0.0, 0.0, 0.0, nullptr,
                                s.coeffs, nullptr, nullptr, nullptr, st);
    if (rc == MINSNAP_OK) {
      minsnap::SoftConstraintArgs m = a;
      m.B = B; m.d_coeffs = s.coeffs; m.d_times = d_times; m.d_scratch = s.extrema;
      m.d_soft = nullptr; m.d_terms = nullptr; m.d_max_value = d_max_value;
      const cudaError_t e = minsnap::launch_soft_constraint_cost(m, st);
      if (e != cudaSuccess) rc = cuda_fail(e, "launch_soft_constraint_cost");
    }
  }
  cudaFreeAsync(ws, st);
  return rc;
}

// SURVEY 8(f)3: collision cost and its gradient against a dense distance grid (ref NL.i:1523-1709)
static int collision_args_check(long B, int K, int D, int N, const int32_t* h_dims, const double* h_origin,
                                double resolution, const double* h_min_bound, const double* h_max_bound, double dt,
                                double map_resolution, double epsilon) {
  if (B < 0 || K < 1 || !h_dims || !h_origin || !h_min_bound || !h_max_bound || !(resolution > 0.0) || !(dt > 0.0) ||
      !(map_resolution > 0.0) || !(epsilon > 0.0) || h_dims[0] < 1 || h_dims[1] < 1 || h_dims[2] < 1)
    return MINSNAP_ERR_ARG;
  if (D != 3 || N != 10) return MINSNAP_ERR_UNSUPPORTED;
  return MINSNAP_OK;
}

static int collision_call(long B, int K, int D, int N, const double* d_coeffs, const double* d_times,
                          const double* d_sdf, const int32_t* h_dims, const double* h_origin, double resolution,
                          double oob_value, const double* h_min_bound, const double* h_max_bound,
                          int use_continuous_distance, double dt, double map_resolution, double epsilon,
                          double robot_radius, double coll_pot_multiplier, bool want_gradient,
                          const int32_t* d_col_of_row, int n_fixed, int n_free, double* d_cost, double* d_grad_free,
                          int32_t* d_is_collision, int32_t* d_charged, minsnap_stream_t stream) {
  const int rc = collision_args_check(B, K, D, N, h_dims, h_origin, resolution, h_min_bound, h_max_bound, dt,
                                      map_resolution, epsilon);
  if (rc != MINSNAP_OK) return rc;
  if (want_gradient) {
    if (n_free < 0 || n_fixed < 0) return MINSNAP_ERR_ARG;
    if (!d_col_of_row && n_free != (K - 1) * (N / 2 - 1)) return MINSNAP_ERR_ARG;   // the standard mask's count
  }
  if (B == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || !d_sdf || !d_cost) return MINSNAP_ERR_ARG;
  if (want_gradient && n_free > 0 && !d_grad_free) return MINSNAP_ERR_ARG;
  minsnap::CollisionArgs a;
  a.B = B; a.K = K; a.N = N; a.d_coeffs = d_coeffs; a.d_times = d_times; a.d_sdf = d_sdf;
  a.nx = h_dims[0]; a.ny = h_dims[1]; a.nz = h_dims[2];
  for (int k = 0; k < 3; ++k) {
    a.origin[k] = h_origin[k];
    a.min_bound[k] = h_min_bound[k];
    a.max_bound[k] = h_max_bound[k];
  }
  a.resolution = resolution; a.oob_value = oob_value; a.use_continuous_distance = use_continuous_distance;
  a.dt = dt; a.map_resolution = map_resolution; a.epsilon = epsilon; a.robot_radius = robot_radius;
  a.coll_pot_multiplier = coll_pot_multiplier;
  a.d_cost = d_cost; a.d_is_collision = d_is_collision; a.d_charged = d_charged;
  a.d_grad_free = (want_gradient && n_free > 0) ? d_grad_free : nullptr;
  a.d_col_of_row = d_col_of_row; a.n_fixed = n_fixed; a.n_free = n_free;
  if (a.d_grad_free)   // the kernel adds its segments' contributions into the free columns
    CU(cudaMemsetAsync(d_grad_free, 0, sizeof(double) * (size_t)B * n_free * 3, as_stream(stream)));
  CU(minsnap::launch_collision_cost(a, as_stream(stream)));
  return MINSNAP_OK;
}

int minsnap_collision_cost(long B, int K, int D, int N, const double* d_coeffs, const double* d_times,
                           const double* d_sdf, const int32_t* h_dims, const double* h_origin, double resolution,
                           double oob_value, const double* h_min_bound, const double* h_max_bound,
                           int use_continuous_distance, double dt, double map_resolution, double epsilon,
                           double robot_radius, double coll_pot_multiplier, double* d_cost, int32_t* d_is_collision,
                           int32_t* d_charged, minsnap_stream_t stream) {
  return collision_call(B, K, D, N, d_coeffs, d_times, d_sdf, h_dims, h_origin, resolution, oob_value, h_min_bound,
                        h_max_bound, use_continuous_distance, dt, map_resolution, epsilon, robot_radius,
                        coll_pot_multiplier, false, nullptr, 0, 0, d_cost, nullptr, d_is_collision, d_charged, stream);
}

int minsnap_collision_gradient(long B, int K, int D, int N, const double* d_coeffs, const double* d_times,
                               const double* d_sdf, const int32_t* h_dims, const double* h_origin, double resolution,
                               double oob_value, const double* h_min_bound, const double* h_max_bound,
                               int use_continuous_distance, double dt, double map_resolution, double epsilon,
                               double robot_radius, double coll_pot_multiplier, const int32_t* d_col_of_row, int n_fixed,
                               int n_free, double* d_cost, double* d_grad_free, int32_t* d_is_collision,
                               int32_t* d_charged, minsnap_stream_t stream) {
  return collision_call(B, K, D, N, d_coeffs, d_times, d_sdf, h_dims, h_origin, resolution, oob_value, h_min_bound,
                        h_max_bound, use_continuous_distance, dt, map_resolution, epsilon, robot_radius,
                        coll_pot_multiplier, true, d_col_of_row, n_fixed, n_free, d_cost, d_grad_free, d_is_collision,
                        d_charged, stream);
}

// ---------------------------------------------------------------------------------------
// The free derivatives (and segment times) against J = w_d J_d + w_c J_c + w_t sum(T)
// (ref getCostAndGradientDerivative NL.i:1452-1521, getCostAndGradientCollision NL.i:1523-1709,
//  getCostAndGradientTime NL.i:2155-2243)
// ---------------------------------------------------------------------------------------
namespace {

// The distance grid and the walk's parameters of minsnap_collision_cost, carried as one value.
struct CollisionMap {
  const double* sdf;
  const int32_t* dims;
  const double* origin;
  double resolution, oob_value;
  const double* min_bound;
  const double* max_bound;
  int use_continuous_distance;
  double dt, map_resolution, epsilon, robot_radius, coll_pot_multiplier;

  int check(long B, int K, int D, int N) const {
    return collision_args_check(B, K, D, N, dims, origin, resolution, min_bound, max_bound, dt, map_resolution,
                                epsilon);
  }
  int cost(long B, int K, const double* coeffs, const double* times, double* out, int32_t* hit,
           cudaStream_t st) const {
    return minsnap_collision_cost(B, K, 3, 10, coeffs, times, sdf, dims, origin, resolution, oob_value, min_bound,
                                  max_bound, use_continuous_distance, dt, map_resolution, epsilon, robot_radius,
                                  coll_pot_multiplier, out, hit, nullptr, st);
  }
  int gradient(long B, int K, const double* coeffs, const double* times, const int32_t* col_of_row, int n_fixed,
               int n_free, double* out, double* grad, cudaStream_t st) const {
    return minsnap_collision_gradient(B, K, 3, 10, coeffs, times, sdf, dims, origin, resolution, oob_value, min_bound,
                                      max_bound, use_continuous_distance, dt, map_resolution, epsilon, robot_radius,
                                      coll_pot_multiplier, col_of_row, n_fixed, n_free, out, grad, nullptr, nullptr,
                                      st);
  }
};

minsnap::GeneralSolveArgs recovery_args(long B, int K, int D, int N, int derivative, int n_fixed, int n_free,
                                        const int32_t* d_col_of_row, const double* d_fixed_values,
                                        const double* d_free_values, const double* d_times) {
  minsnap::GeneralSolveArgs a;
  a.B = B; a.K = K; a.D = D; a.N = N; a.derivative = derivative; a.n_fixed = n_fixed; a.n_free = n_free;
  a.d_col_of_row = d_col_of_row; a.d_fixed_values = d_fixed_values; a.d_free_in = d_free_values;
  a.d_times = d_times; a.d_coeffs = nullptr; a.d_free_out = nullptr; a.d_cost = nullptr; a.d_status = nullptr;
  return a;
}

// The soft limits of the *_soft entries below: the constraints (shapes and pointers are set per launch), their weight
// w_sc in J, the scratch of the per-segment maxima (soft_constraint_scratch_bytes for the largest batch) and [n] for
// the soft cost of the candidates.
struct SoftTerm {
  minsnap::SoftConstraintArgs a;
  double w_sc;
  void* extrema;
  double* soft;
};

// The soft cost of n recovered trajectories, with their maxima (d_max_value, optional) and the scratch left for
// launch_soft_constraint_gradient.
cudaError_t launch_soft_term(const SoftTerm& t, long n, int K, int D, int N, const double* coeffs, const double* times,
                             double* d_soft, double* d_max_value, cudaStream_t st) {
  minsnap::SoftConstraintArgs a = t.a;
  a.B = n; a.K = K; a.D = D; a.N = N;
  a.d_coeffs = coeffs; a.d_times = times; a.d_scratch = t.extrema;
  a.d_soft = d_soft; a.d_terms = nullptr; a.d_max_value = d_max_value;
  return minsnap::launch_soft_constraint_cost(a, st);
}

// minsnap_free_objective on the device, the index map already built: recovery of the B*S candidates (fixed values
// shared by the S candidates of a trajectory), the collision walk, the combine kernel; with a soft term, its soft cost
// on the recovered coefficients, added last with weight w_sc.  Scratch: coeffs [B*S][K][D][N], cost and jc [B*S].
int free_objective_device(long B, int S, int K, int D, int N, int derivative, int n_fixed, int n_free,
                          const int32_t* d_col_of_row, const double* d_fixed_values, const double* d_free_values,
                          const double* d_times, double w_d, double w_c, double w_t, const CollisionMap& map,
                          double* d_objective, double* d_Jd, double* d_jc, int32_t* d_is_collision, double* coeffs,
                          double* cost, cudaStream_t st, const SoftTerm* soft = nullptr) {
  const long n = B * S;
  minsnap::GeneralSolveArgs a =
      recovery_args(n, K, D, N, derivative, n_fixed, n_free, d_col_of_row, d_fixed_values, d_free_values, d_times);
  a.fixed_div = S;
  a.d_coeffs = coeffs;
  a.d_cost = cost;
  CU(minsnap::launch_coeffs_from_constraints(a, st));
  const int rc = map.cost(n, K, coeffs, d_times, d_jc, d_is_collision, st);
  if (rc != MINSNAP_OK) return rc;
  CU(minsnap::launch_free_combine(n, K, cost, d_jc, d_times, w_d, w_c, w_t, d_objective, d_Jd, st));
  if (soft) {
    CU(launch_soft_term(*soft, n, K, D, N, coeffs, d_times, soft->soft, nullptr, st));
    CU(minsnap::launch_free_soft_add(n, soft->soft, soft->w_sc, d_objective, st));
  }
  return MINSNAP_OK;
}

}  // namespace

int minsnap_derivative_gradient(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                                const double* d_fixed_values, const double* d_free_values, const double* d_times,
                                double* d_coeffs, double* d_cost_Jd, double* d_grad_free, double* d_diag_free,
                                void* d_workspace, size_t workspace_bytes, minsnap_stream_t stream) {
  if (!shape_ok(B, K, D, N, derivative) || !h_fixed_mask) return MINSNAP_ERR_ARG;
  if (!d_workspace || workspace_bytes < SolveWorkspace::bytes(N, K)) return MINSNAP_ERR_WORKSPACE;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (B == 0) return MINSNAP_OK;
  if (!d_times || !d_cost_Jd || (n_fixed > 0 && !d_fixed_values) || (n_free > 0 && (!d_free_values || !d_grad_free)))
    return MINSNAP_ERR_ARG;
  cudaStream_t st = as_stream(stream);
  SolveWorkspace ws(d_workspace, N, K);
  CU(minsnap::launch_reorder_host_mask(N, K, h_fixed_mask, ws.mask, ws.col_of_row, ws.counts, st));
  minsnap::GeneralSolveArgs a =
      recovery_args(B, K, D, N, derivative, n_fixed, n_free, ws.col_of_row, d_fixed_values, d_free_values, d_times);
  a.d_coeffs = d_coeffs; a.d_cost = d_cost_Jd; a.d_grad_free = d_grad_free; a.d_diag_free = d_diag_free;
  CU(minsnap::launch_derivative_gradient(a, st));
  return MINSNAP_OK;
}

namespace {

// The limit on the mask launch_reorder_host_mask packs into kernel parameters.
bool mask_fits(int N, int K) { return (long)(K + 1) * (N / 2) <= 32L * minsnap::MaskBits::kWords; }

// The soft arguments of the *_soft free-derivative entries on top of soft_args: w_sc >= 0 and finite.
int free_soft_args(int N, int n_constraints, const int32_t* h_derivatives, const double* h_limits, double weight,
                   double maximum_cost, int extrema_flags, double w_sc, SoftTerm* t) {
  const int rc = soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, &t->a);
  if (rc != MINSNAP_OK) return rc;
  if (!(w_sc >= 0.0 && std::isfinite(w_sc))) return MINSNAP_ERR_ARG;
  t->w_sc = w_sc;
  return MINSNAP_OK;
}

int free_objective_call(long B, int S, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                        const double* d_fixed_values, const double* d_free_values, const double* d_times, double w_d,
                        double w_c, double w_t, const CollisionMap& map, SoftTerm* soft, double* d_objective,
                        double* d_Jd, double* d_Jc, int32_t* d_is_collision, double* d_soft, cudaStream_t st) {
  if (!shape_ok(B, K, D, N, derivative) || S < 1 || !h_fixed_mask) return MINSNAP_ERR_ARG;
  int rc = map.check(B, K, D, N);
  if (rc != MINSNAP_OK) return rc;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (soft && (!mask_fits(N, K) || minsnap::general_fits(N, K, D, n_fixed, n_free) != cudaSuccess))
    return MINSNAP_ERR_UNSUPPORTED;
  if (B == 0) return MINSNAP_OK;
  if (!d_times || !map.sdf || !d_objective || (n_fixed > 0 && !d_fixed_values) || (n_free > 0 && !d_free_values))
    return MINSNAP_ERR_ARG;
  const size_t n = (size_t)B * S;
  const size_t ws_head = align_up(SolveWorkspace::bytes(N, K), 256);
  const size_t n_doubles = n * ((size_t)K * D * N + 2 + (soft ? 1 : 0));
  const size_t extrema = soft ? minsnap::soft_constraint_scratch_bytes((long)n, K, soft->a.n_constraints) : 0;
  char* ws = nullptr;
  retain_pool_memory();
  CU(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_head + sizeof(double) * n_doubles + extrema, st));
  SolveWorkspace sw(ws, N, K);
  double* coeffs = reinterpret_cast<double*>(ws + ws_head);
  double* cost = coeffs + n * K * D * N;
  double* jc = cost + n;
  if (soft) {
    soft->soft = d_soft ? d_soft : jc + n;
    soft->extrema = jc + 2 * n;
  }
  const cudaError_t e = minsnap::launch_reorder_host_mask(N, K, h_fixed_mask, sw.mask, sw.col_of_row, sw.counts, st);
  if (e != cudaSuccess) rc = cuda_fail(e, "launch_reorder_host_mask");
  if (rc == MINSNAP_OK)
    rc = free_objective_device(B, S, K, D, N, derivative, n_fixed, n_free, sw.col_of_row, d_fixed_values,
                               d_free_values, d_times, w_d, w_c, w_t, map, d_objective, d_Jd, jc, d_is_collision,
                               coeffs, cost, st, soft);
  if (rc == MINSNAP_OK && d_Jc && cudaMemcpyAsync(d_Jc, jc, sizeof(double) * n, cudaMemcpyDeviceToDevice, st) != cudaSuccess)
    rc = MINSNAP_ERR_CUDA;
  cudaFreeAsync(ws, st);
  return rc;
}

// The descent of minsnap_optimize_free_constraints; with a soft term (minsnap_optimize_free_constraints_soft) its
// gradient joins the step and the time gradient, and its cost the objective.
int free_descent(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask, const double* d_fixed_values,
                 double* d_free_values, double* d_times, int optimize_times, double w_d, double w_c, double w_t,
                 const CollisionMap& map, SoftTerm* soft, int iterations, int n_steps, double max_relative_step,
                 double min_time, double gradient_increment, double* d_history, int32_t* d_is_collision,
                 double* d_max_value, cudaStream_t st) {
  if (!shape_ok(B, K, D, N, derivative) || !h_fixed_mask || iterations < 0 || n_steps < 1 || !(w_d > 0.0) ||
      !(max_relative_step > 0.0) || !(min_time > 0.0) || !(gradient_increment > 0.0))
    return MINSNAP_ERR_ARG;
  int rc = map.check(B, K, D, N);
  if (rc != MINSNAP_OK) return rc;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (soft && (!mask_fits(N, K) || minsnap::general_fits(N, K, D, n_fixed, n_free) != cudaSuccess))
    return MINSNAP_ERR_UNSUPPORTED;
  if (B == 0) return MINSNAP_OK;
  if (!d_times || !map.sdf || (n_fixed > 0 && !d_fixed_values) || (n_free > 0 && !d_free_values)) return MINSNAP_ERR_ARG;
  const size_t nb = (size_t)B, S = (size_t)n_steps, nfd = (size_t)n_free * D, nc = (size_t)K * D * N;
  const size_t ws_head = align_up(SolveWorkspace::bytes(N, K), 256);
  const size_t n_doubles = nb * (nc + 2 * nfd + n_free + K + 3) + nb * S * (nfd + K + nc + 3);
  const size_t n_ints = nb * (S + 1);
  // soft term: g_sc [B][n_free][D], the candidates' soft cost [B S], per-segment maxima of B S trajectories
  const size_t soft_doubles = soft ? nb * nfd + nb * S : 0;
  const size_t soft_head = align_up(sizeof(double) * n_doubles + sizeof(int32_t) * n_ints, 256);
  char* ws = nullptr;
  retain_pool_memory();
  if (soft)
    CU(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_head + soft_head + sizeof(double) * soft_doubles +
                       minsnap::soft_constraint_scratch_bytes((long)(nb * S), K, soft->a.n_constraints), st));
  else
    CU(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_head + sizeof(double) * n_doubles + sizeof(int32_t) * n_ints, st));
  SolveWorkspace sw(ws, N, K);
  double* coeffs = reinterpret_cast<double*>(ws + ws_head);   // the incumbent's
  double* grad_d = coeffs + nb * nc;
  double* grad_c = grad_d + nb * nfd;
  double* diag = grad_c + nb * nfd;
  double* grad_t = diag + nb * n_free;
  double* jd = grad_t + nb * K;
  double* jc = jd + nb;
  double* incumbent = jc + nb;
  double* cand_free = incumbent + nb;
  double* cand_times = cand_free + nb * S * nfd;
  double* cand_coeffs = cand_times + nb * S * K;
  double* cand_cost = cand_coeffs + nb * S * nc;
  double* cand_jc = cand_cost + nb * S;
  double* cand_obj = cand_jc + nb * S;
  int32_t* cand_hit = reinterpret_cast<int32_t*>(cand_obj + nb * S);
  int32_t* hit = d_is_collision ? d_is_collision : cand_hit + nb * S;
  double* grad_sc = nullptr;
  if (soft) {
    grad_sc = reinterpret_cast<double*>(ws + ws_head + soft_head);
    soft->soft = grad_sc + nb * nfd;
    soft->extrema = soft->soft + nb * S;
  }
  cudaError_t e = minsnap::launch_reorder_host_mask(N, K, h_fixed_mask, sw.mask, sw.col_of_row, sw.counts, st);
  if (e != cudaSuccess) rc = cuda_fail(e, "launch_reorder_host_mask");
  // the incumbent objective at the initial state: the candidate pipeline with one candidate per trajectory
  if (rc == MINSNAP_OK)
    rc = free_objective_device(B, 1, K, D, N, derivative, n_fixed, n_free, sw.col_of_row, d_fixed_values, d_free_values,
                               d_times, w_d, w_c, w_t, map, incumbent, nullptr, cand_jc, hit, cand_coeffs, cand_cost, st,
                               soft);
  if (rc == MINSNAP_OK && d_history)
    if (cudaMemcpyAsync(d_history, incumbent, sizeof(double) * nb, cudaMemcpyDeviceToDevice, st) != cudaSuccess) rc = MINSNAP_ERR_CUDA;
  for (int it = 0; it < iterations && rc == MINSNAP_OK; ++it) {
    minsnap::GeneralSolveArgs a =
        recovery_args(B, K, D, N, derivative, n_fixed, n_free, sw.col_of_row, d_fixed_values, d_free_values, d_times);
    a.d_coeffs = coeffs; a.d_cost = jd; a.d_grad_free = grad_d; a.d_diag_free = diag;
    e = minsnap::launch_derivative_gradient(a, st);
    if (e == cudaSuccess) rc = map.gradient(B, K, coeffs, d_times, sw.col_of_row, n_fixed, n_free, jc, grad_c, st);
    if (e == cudaSuccess && rc == MINSNAP_OK && optimize_times)
      rc = minsnap_time_gradient(B, K, D, N, derivative, coeffs, d_times, gradient_increment, w_d, w_t, grad_t, nullptr, st);
    // the soft term at the incumbent: its maxima, then g_sc, and w_sc dsoft/dT added to the time gradient
    if (e == cudaSuccess && rc == MINSNAP_OK && soft) {
      e = launch_soft_term(*soft, B, K, D, N, coeffs, d_times, nullptr, nullptr, st);
      if (e == cudaSuccess) {
        minsnap::SoftGradientArgs g;
        g.soft = soft->a;
        g.soft.B = B; g.soft.K = K; g.soft.D = D; g.soft.N = N;
        g.soft.d_coeffs = coeffs; g.soft.d_times = d_times; g.soft.d_scratch = soft->extrema;
        g.d_col_of_row = sw.col_of_row; g.n_fixed = n_fixed; g.n_free = n_free;
        g.d_grad_free = grad_sc;
        g.d_grad_times = optimize_times ? grad_t : nullptr;
        g.add_times = true;
        g.times_weight = soft->w_sc;
        e = minsnap::launch_soft_constraint_gradient(g, st);
      }
    }
    if (e == cudaSuccess && rc == MINSNAP_OK && optimize_times)
      e = minsnap::launch_time_candidates(B, n_steps, K, d_times, grad_t, 0.0, max_relative_step, min_time, cand_times, st);
    if (e == cudaSuccess && rc == MINSNAP_OK)
      e = minsnap::launch_free_candidates(B, n_steps, n_free, D, K, d_free_values, grad_d, grad_c, diag, w_d, w_c, d_times,
                                          cand_free, optimize_times ? nullptr : cand_times, st, grad_sc,
                                          soft ? soft->w_sc : 0.0);
    if (e == cudaSuccess && rc == MINSNAP_OK)
      rc = free_objective_device(B, n_steps, K, D, N, derivative, n_fixed, n_free, sw.col_of_row, d_fixed_values,
                                 cand_free, cand_times, w_d, w_c, w_t, map, cand_obj, nullptr, cand_jc, cand_hit,
                                 cand_coeffs, cand_cost, st, soft);
    if (e == cudaSuccess && rc == MINSNAP_OK)
      e = minsnap::launch_free_select(B, n_steps, (int)nfd, K, cand_obj, cand_free, cand_times, cand_hit, d_free_values,
                                      d_times, incumbent, hit, d_history ? d_history + (size_t)(it + 1) * nb : nullptr, st);
    if (rc == MINSNAP_OK && e != cudaSuccess) rc = cuda_fail(e, "free-constraint descent");
  }
  // the maxima at the returned state, from its recovered coefficients
  if (rc == MINSNAP_OK && soft && d_max_value) {
    minsnap::GeneralSolveArgs a =
        recovery_args(B, K, D, N, derivative, n_fixed, n_free, sw.col_of_row, d_fixed_values, d_free_values, d_times);
    a.d_coeffs = coeffs;
    e = minsnap::launch_coeffs_from_constraints(a, st);
    if (e == cudaSuccess) e = launch_soft_term(*soft, B, K, D, N, coeffs, d_times, nullptr, d_max_value, st);
    if (e != cudaSuccess) rc = cuda_fail(e, "soft-limit maxima");
  }
  cudaFreeAsync(ws, st);
  return rc;
}

}  // namespace

int minsnap_free_objective(long B, int S, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                           const double* d_fixed_values, const double* d_free_values, const double* d_times, double w_d,
                           double w_c, double w_t, const double* d_sdf, const int32_t* h_dims, const double* h_origin,
                           double resolution, double oob_value, const double* h_min_bound, const double* h_max_bound,
                           int use_continuous_distance, double dt, double map_resolution, double epsilon,
                           double robot_radius, double coll_pot_multiplier, double* d_objective, double* d_Jd,
                           double* d_Jc, int32_t* d_is_collision, minsnap_stream_t stream) {
  const CollisionMap map{d_sdf, h_dims, h_origin, resolution, oob_value, h_min_bound, h_max_bound,
                         use_continuous_distance, dt, map_resolution, epsilon, robot_radius, coll_pot_multiplier};
  return free_objective_call(B, S, K, D, N, derivative, h_fixed_mask, d_fixed_values, d_free_values, d_times, w_d, w_c,
                             w_t, map, nullptr, d_objective, d_Jd, d_Jc, d_is_collision, nullptr, as_stream(stream));
}

// A batched descent on the free derivatives (and optionally the segment times) that never leaves the device: every
// iteration is launches on `stream` only (recovery with the gradient of J_d, collision gradient, [time gradient,
// time ladder,] candidate ladder, recovery + walk + combine of the candidates, select); the workspace is one
// stream-ordered allocation and the mask reaches the device by value, so the call can be captured into a CUDA graph.
int minsnap_optimize_free_constraints(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                                      const double* d_fixed_values, double* d_free_values, double* d_times,
                                      int optimize_times, double w_d, double w_c, double w_t, const double* d_sdf,
                                      const int32_t* h_dims, const double* h_origin, double resolution,
                                      double oob_value, const double* h_min_bound, const double* h_max_bound,
                                      int use_continuous_distance, double dt, double map_resolution, double epsilon,
                                      double robot_radius, double coll_pot_multiplier, int iterations, int n_steps,
                                      double max_relative_step, double min_time, double gradient_increment,
                                      double* d_history, int32_t* d_is_collision, minsnap_stream_t stream) {
  const CollisionMap map{d_sdf, h_dims, h_origin, resolution, oob_value, h_min_bound, h_max_bound,
                         use_continuous_distance, dt, map_resolution, epsilon, robot_radius, coll_pot_multiplier};
  return free_descent(B, K, D, N, derivative, h_fixed_mask, d_fixed_values, d_free_values, d_times, optimize_times, w_d,
                      w_c, w_t, map, nullptr, iterations, n_steps, max_relative_step, min_time, gradient_increment,
                      d_history, d_is_collision, nullptr, as_stream(stream));
}

// ---------------------------------------------------------------------------------------
// The soft limits of minsnap_soft_constraint_cost in the free-derivative problem: their analytic gradient, the
// objective J + w_sc soft and the descent on it
// ---------------------------------------------------------------------------------------
int minsnap_soft_constraint_gradient(long B, int K, int D, int N, const uint8_t* h_fixed_mask, const double* d_coeffs,
                                     const double* d_times, int n_constraints, const int32_t* h_derivatives,
                                     const double* h_limits, double weight, double maximum_cost, int extrema_flags,
                                     double* d_cost, double* d_grad_free, double* d_grad_times, double* d_max_value,
                                     double* d_max_time, int32_t* d_max_segment, minsnap_stream_t stream) {
  if (B < 0 || K < 1 || D < 1 || D > 32 || !minsnap::supported_n(N) || !h_fixed_mask) return MINSNAP_ERR_ARG;
  SoftTerm t;
  int rc = free_soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, 0.0, &t);
  if (rc != MINSNAP_OK) return rc;
  if (!mask_fits(N, K)) return MINSNAP_ERR_UNSUPPORTED;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (B == 0) return MINSNAP_OK;
  if (!d_coeffs || !d_times || (n_free > 0 && !d_grad_free)) return MINSNAP_ERR_ARG;
  cudaStream_t st = as_stream(stream);
  const size_t ws_head = align_up(SolveWorkspace::bytes(N, K), 256);
  char* ws = nullptr;
  retain_pool_memory();
  CU(cudaMallocAsync(reinterpret_cast<void**>(&ws), ws_head + minsnap::soft_constraint_scratch_bytes(B, K, n_constraints),
                     st));
  SolveWorkspace sw(ws, N, K);
  t.extrema = ws + ws_head;
  cudaError_t e = minsnap::launch_reorder_host_mask(N, K, h_fixed_mask, sw.mask, sw.col_of_row, sw.counts, st);
  if (e == cudaSuccess) e = launch_soft_term(t, B, K, D, N, d_coeffs, d_times, d_cost, d_max_value, st);
  if (e == cudaSuccess) {
    minsnap::SoftGradientArgs g;
    g.soft = t.a;
    g.soft.B = B; g.soft.K = K; g.soft.D = D; g.soft.N = N;
    g.soft.d_coeffs = d_coeffs; g.soft.d_times = d_times; g.soft.d_scratch = t.extrema;
    g.d_col_of_row = sw.col_of_row; g.n_fixed = n_fixed; g.n_free = n_free;
    g.d_grad_free = d_grad_free; g.d_grad_times = d_grad_times;
    g.d_max_time = d_max_time; g.d_max_segment = d_max_segment;
    e = minsnap::launch_soft_constraint_gradient(g, st);
  }
  if (e != cudaSuccess) rc = cuda_fail(e, "soft-limit gradient");
  cudaFreeAsync(ws, st);
  return rc;
}

int minsnap_free_objective_soft(long B, int S, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                                const double* d_fixed_values, const double* d_free_values, const double* d_times,
                                double w_d, double w_c, double w_t, const double* d_sdf, const int32_t* h_dims,
                                const double* h_origin, double resolution, double oob_value, const double* h_min_bound,
                                const double* h_max_bound, int use_continuous_distance, double dt, double map_resolution,
                                double epsilon, double robot_radius, double coll_pot_multiplier, int n_constraints,
                                const int32_t* h_derivatives, const double* h_limits, double weight,
                                double maximum_cost, int extrema_flags, double w_sc, double* d_objective, double* d_Jd,
                                double* d_Jc, int32_t* d_is_collision, double* d_soft, minsnap_stream_t stream) {
  SoftTerm t;
  const int rc = free_soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, w_sc, &t);
  if (rc != MINSNAP_OK) return rc;
  const CollisionMap map{d_sdf, h_dims, h_origin, resolution, oob_value, h_min_bound, h_max_bound,
                         use_continuous_distance, dt, map_resolution, epsilon, robot_radius, coll_pot_multiplier};
  return free_objective_call(B, S, K, D, N, derivative, h_fixed_mask, d_fixed_values, d_free_values, d_times, w_d, w_c,
                             w_t, map, &t, d_objective, d_Jd, d_Jc, d_is_collision, d_soft, as_stream(stream));
}

int minsnap_optimize_free_constraints_soft(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                                           const double* d_fixed_values, double* d_free_values, double* d_times,
                                           int optimize_times, double w_d, double w_c, double w_t, const double* d_sdf,
                                           const int32_t* h_dims, const double* h_origin, double resolution,
                                           double oob_value, const double* h_min_bound, const double* h_max_bound,
                                           int use_continuous_distance, double dt, double map_resolution,
                                           double epsilon, double robot_radius, double coll_pot_multiplier,
                                           int n_constraints, const int32_t* h_derivatives, const double* h_limits,
                                           double weight, double maximum_cost, int extrema_flags, double w_sc,
                                           int iterations, int n_steps, double max_relative_step, double min_time,
                                           double gradient_increment, double* d_history, int32_t* d_is_collision,
                                           double* d_max_value, minsnap_stream_t stream) {
  SoftTerm t;
  const int rc = free_soft_args(N, n_constraints, h_derivatives, h_limits, weight, maximum_cost, extrema_flags, w_sc, &t);
  if (rc != MINSNAP_OK) return rc;
  const CollisionMap map{d_sdf, h_dims, h_origin, resolution, oob_value, h_min_bound, h_max_bound,
                         use_continuous_distance, dt, map_resolution, epsilon, robot_radius, coll_pot_multiplier};
  return free_descent(B, K, D, N, derivative, h_fixed_mask, d_fixed_values, d_free_values, d_times, optimize_times, w_d,
                      w_c, w_t, map, &t, iterations, n_steps, max_relative_step, min_time, gradient_increment, d_history,
                      d_is_collision, d_max_value, as_stream(stream));
}


// ---------------------------------------------------------------------------------------
// Host-buffer entry points
// ---------------------------------------------------------------------------------------
int minsnap_host_alloc(void** h_ptr, size_t bytes) {
  if (!h_ptr) return MINSNAP_ERR_ARG;
  CU(cudaHostAlloc(h_ptr, bytes ? bytes : 16, cudaHostAllocDefault));
  return MINSNAP_OK;
}

int minsnap_host_free(void* h_ptr) {
  if (!h_ptr) return MINSNAP_OK;
  CU(cudaFreeHost(h_ptr));
  return MINSNAP_OK;
}

int minsnap_reorder_host(int N, int K, long n_masks, const uint8_t* h_mask, int32_t* h_col_of_row,
                         int32_t* h_counts) {
  if (!minsnap::supported_n(N) || K < 1 || n_masks < 0 || !h_mask || !h_col_of_row || !h_counts)
    return MINSNAP_ERR_ARG;
  if (n_masks == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nm = (size_t)n_masks;
  const int i_mask = hc.in(h_mask, nm * (K + 1) * (N / 2));
  const int o_col = hc.out(h_col_of_row, sizeof(int32_t) * nm * N * K);
  const int o_cnt = hc.out(h_counts, sizeof(int32_t) * nm * 2);
  return hc.run([&](cudaStream_t st) {
    return minsnap_reorder(N, K, n_masks, hc.dev<uint8_t>(i_mask), hc.dev<int32_t>(o_col), hc.dev<int32_t>(o_cnt), st);
  });
}

int minsnap_solve_host(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                       const double* h_fixed_values, const double* h_times, double* h_coeffs,
                       double* h_free_values, double* h_cost, int32_t* h_status, int32_t* h_col_of_row) {
  if (!shape_ok(B, K, D, N, derivative) || !h_fixed_mask || !h_times || !h_coeffs) return MINSNAP_ERR_ARG;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (n_fixed > 0 && !h_fixed_values) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_fixed = hc.in(h_fixed_values, sizeof(double) * nb * n_fixed * D);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_coeffs = hc.out(h_coeffs, sizeof(double) * nb * K * D * N);
  const int o_free = hc.out(h_free_values, sizeof(double) * nb * n_free * D);
  const int o_cost = hc.out(h_cost, sizeof(double) * nb);
  const int o_status = hc.out(h_status, sizeof(int32_t) * nb);
  const int o_col = hc.out(h_col_of_row, sizeof(int32_t) * (size_t)N * K);
  const int t_ws = hc.scratch(SolveWorkspace::bytes(N, K));
  return hc.run([&](cudaStream_t st) {
    return minsnap_solve(B, K, D, N, derivative, h_fixed_mask, hc.dev<double>(i_fixed), hc.dev<double>(i_times),
                         hc.dev<double>(o_coeffs), hc.dev<double>(o_free), hc.dev_if<double>(o_cost, h_cost),
                         hc.dev<int32_t>(o_status), hc.dev<int32_t>(o_col), hc.dev<char>(t_ws),
                         SolveWorkspace::bytes(N, K), st);
  });
}

int minsnap_coeffs_from_constraints_host(long B, int K, int D, int N, const uint8_t* h_fixed_mask,
                                         const double* h_fixed_values, const double* h_free_values,
                                         const double* h_times, double* h_coeffs) {
  if (!shape_ok(B, K, D, N, 0) || !h_fixed_mask || !h_times || !h_coeffs) return MINSNAP_ERR_ARG;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if ((n_fixed > 0 && !h_fixed_values) || (n_free > 0 && !h_free_values)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_fixed = hc.in(h_fixed_values, sizeof(double) * nb * n_fixed * D);
  const int i_free = hc.in(h_free_values, sizeof(double) * nb * n_free * D);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_coeffs = hc.out(h_coeffs, sizeof(double) * nb * K * D * N);
  const int t_ws = hc.scratch(SolveWorkspace::bytes(N, K));
  return hc.run([&](cudaStream_t st) {
    return minsnap_coeffs_from_constraints(B, K, D, N, h_fixed_mask, hc.dev<double>(i_fixed), hc.dev<double>(i_free),
                                           hc.dev<double>(i_times), hc.dev<double>(o_coeffs), hc.dev<char>(t_ws),
                                           SolveWorkspace::bytes(N, K), st);
  });
}

int minsnap_derivative_gradient_host(long B, int K, int D, int N, int derivative, const uint8_t* h_fixed_mask,
                                     const double* h_fixed_values, const double* h_free_values, const double* h_times,
                                     double* h_coeffs, double* h_cost_Jd, double* h_grad_free, double* h_diag_free) {
  if (!shape_ok(B, K, D, N, derivative) || !h_fixed_mask) return MINSNAP_ERR_ARG;
  int n_fixed, n_free;
  count_mask(h_fixed_mask, N, K, &n_fixed, &n_free);
  if (B == 0) return MINSNAP_OK;
  if (!h_times || !h_cost_Jd || (n_fixed > 0 && !h_fixed_values) || (n_free > 0 && (!h_free_values || !h_grad_free)))
    return MINSNAP_ERR_ARG;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_fixed = hc.in(h_fixed_values, sizeof(double) * nb * n_fixed * D);
  const int i_free = hc.in(h_free_values, sizeof(double) * nb * n_free * D);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_coeffs = hc.out(h_coeffs, h_coeffs ? sizeof(double) * nb * K * D * N : 0);
  const int o_cost = hc.out(h_cost_Jd, sizeof(double) * nb);
  const int o_grad = hc.out(h_grad_free, sizeof(double) * nb * n_free * D);
  const int o_diag = hc.out(h_diag_free, h_diag_free ? sizeof(double) * nb * n_free : 0);
  const int t_ws = hc.scratch(SolveWorkspace::bytes(N, K));
  return hc.run([&](cudaStream_t st) {
    return minsnap_derivative_gradient(B, K, D, N, derivative, h_fixed_mask, hc.dev<double>(i_fixed),
                                       hc.dev<double>(i_free), hc.dev<double>(i_times),
                                       hc.dev_if<double>(o_coeffs, h_coeffs), hc.dev<double>(o_cost),
                                       hc.dev<double>(o_grad), hc.dev_if<double>(o_diag, h_diag_free),
                                       hc.dev<char>(t_ws), SolveWorkspace::bytes(N, K), st);
  });
}

int minsnap_cost_host(long B, int K, int D, int N, int derivative, const double* h_coeffs, const double* h_times,
                      double* h_cost) {
  if (!shape_ok(B, K, D, N, derivative) || !h_coeffs || !h_times || !h_cost) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_cost = hc.out(h_cost, sizeof(double) * nb);
  return hc.run([&](cudaStream_t st) {
    return minsnap_cost(B, K, D, N, derivative, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), hc.dev<double>(o_cost), st);
  });
}

int minsnap_extrema_host(long B, int K, int D, int N, const double* h_coeffs, const double* h_times, int derivative,
                         int mode, uint32_t dim_mask, double* h_max_time, double* h_max_value,
                         int32_t* h_max_segment, double* h_min_time, double* h_min_value, int32_t* h_min_segment,
                         double* h_cand_times, double* h_cand_values, int32_t* h_root_count) {
  if (!extrema_args_ok(B, K, D, N, derivative, mode, &dim_mask)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!h_coeffs || !h_times) return MINSNAP_ERR_ARG;
  const size_t nb = (size_t)B;
  const size_t max_roots = (size_t)minsnap::extrema_max_roots(N, derivative, __builtin_popcount(dim_mask));
  const size_t cand_bytes = sizeof(double) * nb * K * (max_roots + 2);
  // the minimum is produced in trajectory mode only: in optimisation mode the caller's h_min_* stay untouched
  const bool with_min = (mode & ~MINSNAP_EXTREMA_KEEP_SMALL_COEFFICIENTS) == MINSNAP_EXTREMA_TRAJECTORY;
  HostCall hc;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_xt = hc.out(h_max_time, sizeof(double) * nb);
  const int o_xv = hc.out(h_max_value, sizeof(double) * nb);
  const int o_xs = hc.out(h_max_segment, sizeof(int32_t) * nb);
  const int o_nt = hc.out(with_min ? h_min_time : nullptr, sizeof(double) * nb);
  const int o_nv = hc.out(with_min ? h_min_value : nullptr, sizeof(double) * nb);
  const int o_ns = hc.out(with_min ? h_min_segment : nullptr, sizeof(int32_t) * nb);
  const int o_ct = hc.out(h_cand_times, h_cand_times ? cand_bytes : 0);
  const int o_cv = hc.out(h_cand_values, h_cand_values ? cand_bytes : 0);
  const int o_rc = hc.out(h_root_count, h_root_count ? sizeof(int32_t) * nb * K : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_extrema(B, K, D, N, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), derivative, mode, dim_mask,
                           hc.dev<double>(o_xt), hc.dev<double>(o_xv), hc.dev<int32_t>(o_xs), hc.dev<double>(o_nt),
                           hc.dev<double>(o_nv), hc.dev<int32_t>(o_ns), hc.dev_if<double>(o_ct, h_cand_times),
                           hc.dev_if<double>(o_cv, h_cand_values), hc.dev_if<int32_t>(o_rc, h_root_count), st);
  });
}

// Large batches: a chunked copy / solve / copy pipeline of three stages on the thread's persistent streams
// (HostPipeline above); small ones: one staged call.
int minsnap_solve_standard_host(long B, int K, int D, int N, int derivative, const double* h_positions,
                                const double* h_end_derivatives, const double* h_times, double v_max,
                                double a_max, double magic, double* h_times_out, double* h_coeffs,
                                double* h_free_values, double* h_cost, int32_t* h_status) {
  if (!shape_ok(B, K, D, N, derivative)) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  if (!h_positions || !h_coeffs) return MINSNAP_ERR_ARG;
  if (!h_times && !(v_max > 0.0 && a_max > 0.0)) return MINSNAP_ERR_ARG;
  {
    const size_t nb = (size_t)B;
    const int hh = N / 2;
    const size_t n_free_s = (size_t)(K > 1 ? (K - 1) * (hh - 1) : 0);
    const size_t total = sizeof(double) * nb * ((K + 1) * D + 2 * (hh - 1) * D + 2 * K + K * D * N + n_free_s * D + 1) + 4 * nb;
    if (total + 4096 <= kSmallCallBytes) {
      HostCall hc;
      const int i_pos = hc.in(h_positions, sizeof(double) * nb * (K + 1) * D);
      const int i_end = hc.in(h_end_derivatives, sizeof(double) * nb * 2 * (hh - 1) * D);
      const int i_tm = hc.in(h_times, sizeof(double) * nb * K);
      const int o_tm = hc.out(h_times ? nullptr : h_times_out, sizeof(double) * nb * K);
      const int o_coeffs = hc.out(h_coeffs, sizeof(double) * nb * K * D * N);
      const int o_free = hc.out(h_free_values, h_free_values ? sizeof(double) * nb * n_free_s * D : 0);
      const int o_cost = hc.out(h_cost, h_cost ? sizeof(double) * nb : 0);
      const int o_status = hc.out(h_status, h_status ? sizeof(int32_t) * nb : 0);
      const int rc = hc.run([&](cudaStream_t st) {
        return minsnap_solve_standard(B, K, D, N, derivative, hc.dev<double>(i_pos),
                                      hc.dev_if<double>(i_end, h_end_derivatives), hc.dev_if<double>(i_tm, h_times), v_max,
                                      a_max, magic, (!h_times && h_times_out) ? hc.dev<double>(o_tm) : nullptr,
                                      hc.dev<double>(o_coeffs), hc.dev_if<double>(o_free, h_free_values),
                                      hc.dev_if<double>(o_cost, h_cost), hc.dev_if<int32_t>(o_status, h_status), st);
      });
      if (rc == MINSNAP_OK && h_times && h_times_out) std::memcpy(h_times_out, h_times, sizeof(double) * nb * K);
      return rc;
    }
  }
#define TRY(x) do { cudaError_t e__ = (x); if (e__ != cudaSuccess) { rc = cuda_fail(e__, #x); goto done; } } while (0)
  const int h = N / 2;
  const int n_free = (K - 1) * (h - 1);
  // chunk = unit of the copy/solve/copy pipeline; measured on B200 + PCIe Gen5: 4096-8192 is best (D2H stays busy,
  // small pipeline fill)
  const long chunk = std::min<long>(B, 4096);
  // Stage layout: one device block per pipeline stage, carved into the per-chunk arrays.
  const size_t nc = (size_t)chunk;
  size_t off = 0;
  auto carve = [&off](size_t bytes) { const size_t at = off; off += align_up(bytes ? bytes : 16, 256); return at; };
  const size_t o_pos = carve(sizeof(double) * nc * (K + 1) * D);
  const size_t o_end = carve(h_end_derivatives ? sizeof(double) * nc * 2 * (h - 1) * D : 0);
  const size_t o_tm = carve(sizeof(double) * nc * K);
  const size_t o_co = carve(sizeof(double) * nc * K * D * N);
  const size_t o_fr = carve(h_free_values ? sizeof(double) * nc * (n_free > 0 ? n_free : 1) * D : 0);
  const size_t o_cs = carve(h_cost ? sizeof(double) * nc : 0);
  const size_t o_ss = carve(h_status ? sizeof(int32_t) * nc : 0);
  CU(g_pipeline.ensure(off));
  int rc = MINSNAP_OK;
  {
    int stage = 0;
    for (long b0 = 0; b0 < B; b0 += chunk, stage = (stage + 1) % HostPipeline::kDepth) {
      const long nb = std::min(chunk, B - b0);
      cudaStream_t st = g_pipeline.stream[stage];
      char* base = g_pipeline.block[stage];
      double* d_pos = reinterpret_cast<double*>(base + o_pos);
      double* d_end = reinterpret_cast<double*>(base + o_end);
      double* d_tm = reinterpret_cast<double*>(base + o_tm);
      double* d_co = reinterpret_cast<double*>(base + o_co);
      double* d_fr = reinterpret_cast<double*>(base + o_fr);
      double* d_cs = reinterpret_cast<double*>(base + o_cs);
      int32_t* d_ss = reinterpret_cast<int32_t*>(base + o_ss);
      TRY(cudaMemcpyAsync(d_pos, h_positions + (size_t)b0 * (K + 1) * D, sizeof(double) * nb * (K + 1) * D,
                          cudaMemcpyHostToDevice, st));
      if (h_end_derivatives)
        TRY(cudaMemcpyAsync(d_end, h_end_derivatives + (size_t)b0 * 2 * (h - 1) * D,
                            sizeof(double) * nb * 2 * (h - 1) * D, cudaMemcpyHostToDevice, st));
      if (h_times)
        TRY(cudaMemcpyAsync(d_tm, h_times + (size_t)b0 * K, sizeof(double) * nb * K, cudaMemcpyHostToDevice, st));
      rc = minsnap_solve_standard(nb, K, D, N, derivative, d_pos, h_end_derivatives ? d_end : nullptr,
                                  h_times ? d_tm : nullptr, v_max, a_max, magic,
                                  (!h_times && h_times_out) ? d_tm : nullptr, d_co, h_free_values ? d_fr : nullptr,
                                  h_cost ? d_cs : nullptr, h_status ? d_ss : nullptr, st);
      if (rc != MINSNAP_OK) goto done;
      TRY(cudaMemcpyAsync(h_coeffs + (size_t)b0 * K * D * N, d_co, sizeof(double) * nb * K * D * N,
                          cudaMemcpyDeviceToHost, st));
      if (h_times_out) {
        if (h_times) std::memcpy(h_times_out + (size_t)b0 * K, h_times + (size_t)b0 * K, sizeof(double) * nb * K);
        else TRY(cudaMemcpyAsync(h_times_out + (size_t)b0 * K, d_tm, sizeof(double) * nb * K,
                                 cudaMemcpyDeviceToHost, st));
      }
      if (h_free_values && n_free > 0)
        TRY(cudaMemcpyAsync(h_free_values + (size_t)b0 * n_free * D, d_fr, sizeof(double) * nb * n_free * D,
                            cudaMemcpyDeviceToHost, st));
      if (h_cost) TRY(cudaMemcpyAsync(h_cost + b0, d_cs, sizeof(double) * nb, cudaMemcpyDeviceToHost, st));
      if (h_status) TRY(cudaMemcpyAsync(h_status + b0, d_ss, sizeof(int32_t) * nb, cudaMemcpyDeviceToHost, st));
    }
  done:;
  }
  for (auto st : g_pipeline.stream) {
    cudaError_t es = cudaStreamSynchronize(st);
    if (rc == MINSNAP_OK && es != cudaSuccess) rc = cuda_fail(es, "cudaStreamSynchronize");
  }
  return rc;
}

#undef TRY

int minsnap_sample_at_host(long B, int K, int D, int N, const double* h_coeffs, const double* h_times, int M,
                           const double* h_t, long t_stride, int n_deriv, double* h_out, int32_t* h_segment) {
  if (B < 0 || K < 1 || D < 1 || !minsnap::supported_n(N) || M < 0 || n_deriv < 1 || !h_coeffs || !h_times ||
      !h_t || !h_out || (t_stride != 0 && t_stride < M))
    return MINSNAP_ERR_ARG;
  if (B == 0 || M == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const size_t n_t = t_stride == 0 ? (size_t)M : nb * (size_t)t_stride;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int i_t = hc.in(h_t, sizeof(double) * n_t);
  const int o_out = hc.out(h_out, sizeof(double) * nb * M * n_deriv * D);
  const int o_seg = hc.out(h_segment, h_segment ? sizeof(int32_t) * nb * M : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_sample_at(B, K, D, N, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), M, hc.dev<double>(i_t),
                             t_stride, n_deriv, hc.dev<double>(o_out), hc.dev_if<int32_t>(o_seg, h_segment), st);
  });
}

int minsnap_sample_uniform_host(long B, int K, int D, int N, const double* h_coeffs, const double* h_times, int M,
                                int n_deriv, double* h_out, double* h_t_out) {
  if (B < 0 || K < 1 || D < 1 || !minsnap::supported_n(N) || M < 0 || n_deriv < 1 || !h_coeffs || !h_times || !h_out)
    return MINSNAP_ERR_ARG;
  if (B == 0 || M == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_out = hc.out(h_out, sizeof(double) * nb * M * n_deriv * D);
  const int o_t = hc.out(h_t_out, h_t_out ? sizeof(double) * nb * M : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_sample_uniform(B, K, D, N, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), M, n_deriv,
                                  hc.dev<double>(o_out), hc.dev_if<double>(o_t, h_t_out), st);
  });
}

int minsnap_evaluate_range_host(int K, int D, int N, const double* h_coeffs, const double* h_times, double t_start,
                                double t_end, double dt, int derivative, int max_samples, double* h_out,
                                double* h_t_out, int32_t* h_count) {
  if (K < 1 || D < 1 || !minsnap::supported_n(N) || !(dt > 0.0) || derivative < 0 || max_samples < 0 || !h_coeffs ||
      !h_times || !h_out || !h_count)
    return MINSNAP_ERR_ARG;
  HostCall hc;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * (size_t)K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * (size_t)K);
  const int o_out = hc.out(nullptr, sizeof(double) * (size_t)max_samples * D);   // fetched below: only the emitted samples
  const int o_t = hc.out(nullptr, sizeof(double) * (size_t)max_samples);
  const int o_cnt = hc.out(h_count, sizeof(int32_t));
  int rc = hc.run([&](cudaStream_t st) {
    return minsnap_evaluate_range(1, K, D, N, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), t_start, t_end, dt,
                                  derivative, max_samples, hc.dev<double>(o_out), hc.dev<double>(o_t),
                                  hc.dev<int32_t>(o_cnt), st);
  });
  if (rc != MINSNAP_OK) return rc;
  const size_t n_emit = (size_t)std::max(0, std::min(*h_count, max_samples));
  if ((rc = hc.fetch(o_out, h_out, sizeof(double) * n_emit * D)) != MINSNAP_OK) return rc;
  if (h_t_out) rc = hc.fetch(o_t, h_t_out, sizeof(double) * n_emit);
  return rc;
}

int minsnap_segment_matrices_host(long n, int N, int derivative, const double* h_T, double* h_A, double* h_Ainv,
                                  double* h_Q, double* h_H) {
  if (n < 0 || !minsnap::supported_n(N) || derivative < 0 || derivative > N / 2 - 1 || !h_T) return MINSNAP_ERR_ARG;
  if (n == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t mat = sizeof(double) * (size_t)n * N * N;
  const int i_T = hc.in(h_T, sizeof(double) * (size_t)n);
  const int o_A = hc.out(h_A, h_A ? mat : 0), o_Ai = hc.out(h_Ainv, h_Ainv ? mat : 0);
  const int o_Q = hc.out(h_Q, h_Q ? mat : 0), o_H = hc.out(h_H, h_H ? mat : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_segment_matrices(n, N, derivative, hc.dev<double>(i_T), hc.dev_if<double>(o_A, h_A),
                                    hc.dev_if<double>(o_Ai, h_Ainv), hc.dev_if<double>(o_Q, h_Q),
                                    hc.dev_if<double>(o_H, h_H), st);
  });
}

int minsnap_estimate_segment_times_host(long B, int K, int D, const double* h_positions, double v_max,
                                        double a_max, double magic, double* h_times) {
  if (B < 0 || K < 1 || D < 1 || !h_positions || !h_times) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_pos = hc.in(h_positions, sizeof(double) * nb * (K + 1) * D);
  const int o_times = hc.out(h_times, sizeof(double) * nb * K);
  return hc.run([&](cudaStream_t st) {
    return minsnap_estimate_segment_times(B, K, D, hc.dev<double>(i_pos), v_max, a_max, magic, hc.dev<double>(o_times), st);
  });
}

int minsnap_cost_sweep_host(long B, int S, int K, int D, int N, int derivative, const double* h_positions,
                            const double* h_end_derivatives, const double* h_times, double* h_cost, int32_t* h_status) {
  if (!shape_ok(B, K, D, N, derivative) || S < 1 || !h_positions || !h_times || !h_cost) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_pos = hc.in(h_positions, sizeof(double) * nb * (K + 1) * D);
  const int i_end = hc.in(h_end_derivatives, sizeof(double) * nb * 2 * (N / 2 - 1) * D);
  const int i_tm = hc.in(h_times, sizeof(double) * nb * S * K);
  const int o_cost = hc.out(h_cost, sizeof(double) * nb * S);
  const int o_status = hc.out(h_status, h_status ? sizeof(int32_t) * nb * S : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_cost_sweep(B, S, K, D, N, derivative, hc.dev<double>(i_pos), hc.dev_if<double>(i_end, h_end_derivatives),
                              hc.dev<double>(i_tm), hc.dev<double>(o_cost), hc.dev_if<int32_t>(o_status, h_status), st);
  });
}

int minsnap_time_objective_host(long B, int S, int K, int D, int N, int derivative, const double* h_positions,
                                const double* h_end_derivatives, const double* h_times, double time_penalty,
                                double* h_objective, double* h_cost, int32_t* h_status) {
  if (!shape_ok(B, K, D, N, derivative) || S < 1 || !h_positions || !h_times || !h_objective) return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_pos = hc.in(h_positions, sizeof(double) * nb * (K + 1) * D);
  const int i_end = hc.in(h_end_derivatives, sizeof(double) * nb * 2 * (N / 2 - 1) * D);
  const int i_tm = hc.in(h_times, sizeof(double) * nb * S * K);
  const int o_obj = hc.out(h_objective, sizeof(double) * nb * S);
  const int o_cost = hc.out(h_cost, h_cost ? sizeof(double) * nb * S : 0);
  const int o_status = hc.out(h_status, h_status ? sizeof(int32_t) * nb * S : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_time_objective(B, S, K, D, N, derivative, hc.dev<double>(i_pos),
                                  hc.dev_if<double>(i_end, h_end_derivatives), hc.dev<double>(i_tm), time_penalty,
                                  hc.dev<double>(o_obj), hc.dev_if<double>(o_cost, h_cost),
                                  hc.dev_if<int32_t>(o_status, h_status), st);
  });
}

int minsnap_time_gradient_host(long B, int K, int D, int N, int derivative, const double* h_coeffs, const double* h_times,
                               double increment, double w_d, double w_t, double* h_gradient, double* h_segment_cost) {
  if (!shape_ok(B, K, D, N, derivative) || !(increment > 0.0) || !h_coeffs || !h_times || (!h_gradient && !h_segment_cost))
    return MINSNAP_ERR_ARG;
  if (B == 0) return MINSNAP_OK;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int o_grad = hc.out(h_gradient, h_gradient ? sizeof(double) * nb * K : 0);
  const int o_seg = hc.out(h_segment_cost, h_segment_cost ? sizeof(double) * nb * K : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_time_gradient(B, K, D, N, derivative, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), increment, w_d,
                                 w_t, hc.dev_if<double>(o_grad, h_gradient), hc.dev_if<double>(o_seg, h_segment_cost), st);
  });
}

int minsnap_collision_cost_host(long B, int K, int D, int N, const double* h_coeffs, const double* h_times,
                                const double* h_sdf, const int32_t* h_dims, const double* h_origin, double resolution,
                                double oob_value, const double* h_min_bound, const double* h_max_bound,
                                int use_continuous_distance, double dt, double map_resolution, double epsilon,
                                double robot_radius, double coll_pot_multiplier, double* h_cost, int32_t* h_is_collision,
                                int32_t* h_charged) {
  if (B < 0 || K < 1 || !h_dims || h_dims[0] < 1 || h_dims[1] < 1 || h_dims[2] < 1) return MINSNAP_ERR_ARG;
  if (D != 3 || N != 10) return MINSNAP_ERR_UNSUPPORTED;
  if (B == 0) return MINSNAP_OK;
  if (!h_coeffs || !h_times || !h_sdf || !h_cost) return MINSNAP_ERR_ARG;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int i_sdf = hc.in(h_sdf, sizeof(double) * (size_t)h_dims[0] * h_dims[1] * h_dims[2]);
  const int o_cost = hc.out(h_cost, sizeof(double) * nb);
  const int o_hit = hc.out(h_is_collision, h_is_collision ? sizeof(int32_t) * nb : 0);
  const int o_chg = hc.out(h_charged, h_charged ? sizeof(int32_t) * nb : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_collision_cost(B, K, D, N, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), hc.dev<double>(i_sdf), h_dims,
                                  h_origin, resolution, oob_value, h_min_bound, h_max_bound, use_continuous_distance, dt,
                                  map_resolution, epsilon, robot_radius, coll_pot_multiplier, hc.dev<double>(o_cost),
                                  hc.dev_if<int32_t>(o_hit, h_is_collision), hc.dev_if<int32_t>(o_chg, h_charged), st);
  });
}

int minsnap_collision_gradient_host(long B, int K, int D, int N, const double* h_coeffs, const double* h_times,
                                    const double* h_sdf, const int32_t* h_dims, const double* h_origin, double resolution,
                                    double oob_value, const double* h_min_bound, const double* h_max_bound,
                                    int use_continuous_distance, double dt, double map_resolution, double epsilon,
                                    double robot_radius, double coll_pot_multiplier, const int32_t* h_col_of_row,
                                    int n_fixed, int n_free, double* h_cost, double* h_grad_free, int32_t* h_is_collision,
                                    int32_t* h_charged) {
  if (B < 0 || K < 1 || n_free < 0 || !h_dims || h_dims[0] < 1 || h_dims[1] < 1 || h_dims[2] < 1) return MINSNAP_ERR_ARG;
  if (D != 3 || N != 10) return MINSNAP_ERR_UNSUPPORTED;
  if (B == 0) return MINSNAP_OK;
  if (!h_coeffs || !h_times || !h_sdf || !h_cost || (n_free > 0 && !h_grad_free)) return MINSNAP_ERR_ARG;
  HostCall hc;
  const size_t nb = (size_t)B;
  const int i_coeffs = hc.in(h_coeffs, sizeof(double) * nb * K * D * N);
  const int i_times = hc.in(h_times, sizeof(double) * nb * K);
  const int i_sdf = hc.in(h_sdf, sizeof(double) * (size_t)h_dims[0] * h_dims[1] * h_dims[2]);
  const int i_col = hc.in(h_col_of_row, h_col_of_row ? sizeof(int32_t) * (size_t)N * K : 0);
  const int o_cost = hc.out(h_cost, sizeof(double) * nb);
  const int o_grad = hc.out(h_grad_free, sizeof(double) * nb * n_free * 3);
  const int o_hit = hc.out(h_is_collision, h_is_collision ? sizeof(int32_t) * nb : 0);
  const int o_chg = hc.out(h_charged, h_charged ? sizeof(int32_t) * nb : 0);
  return hc.run([&](cudaStream_t st) {
    return minsnap_collision_gradient(B, K, D, N, hc.dev<double>(i_coeffs), hc.dev<double>(i_times), hc.dev<double>(i_sdf),
                                      h_dims, h_origin, resolution, oob_value, h_min_bound, h_max_bound,
                                      use_continuous_distance, dt, map_resolution, epsilon, robot_radius,
                                      coll_pot_multiplier, hc.dev_if<int32_t>(i_col, h_col_of_row), n_fixed, n_free,
                                      hc.dev<double>(o_cost), hc.dev_if<double>(o_grad, n_free > 0 ? h_grad_free : nullptr),
                                      hc.dev_if<int32_t>(o_hit, h_is_collision), hc.dev_if<int32_t>(o_chg, h_charged), st);
  });
}

int minsnap_fp64_peak(int repeats, double* tflops) {
  if (!tflops || repeats < 1) return MINSNAP_ERR_ARG;
  CU(minsnap::run_fp64_peak(repeats, tflops));
  return MINSNAP_OK;
}

}  // extern "C"
