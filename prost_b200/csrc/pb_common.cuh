// pb_common.cuh -- context, error plumbing and device buffers shared by all translation units.
#pragma once

#include <cuda_runtime.h>

#include <chrono>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <memory>
#include <sstream>
#include <stdexcept>
#include <string>
#include <vector>

#include "prost_b200.h"

namespace pb {

// Host-side error type; converted to pb_status + pb_last_error() at the C boundary.
// The message prefixes follow the strings the reference throws (exception.hpp:29-41).
struct Error : public std::runtime_error {
  int status;
  Error(int st, const std::string& msg) : std::runtime_error(msg), status(st) {}
};

[[noreturn]] inline void fail(int status, const std::string& msg) { throw Error(status, msg); }

#define PB_CUDA(expr)                                                                   \
  do {                                                                                  \
    cudaError_t pb_err__ = (expr);                                                      \
    if (pb_err__ != cudaSuccess) {                                                      \
      std::ostringstream pb_ss__;                                                       \
      pb_ss__ << "CUDA error: " << cudaGetErrorString(pb_err__) << " (" << #expr << " at " \
              << __FILE__ << ":" << __LINE__ << ")";                                    \
      ::pb::fail(pb_err__ == cudaErrorMemoryAllocation ? PB_ERR_OOM : PB_ERR_CUDA,      \
                 pb_ss__.str());                                                        \
    }                                                                                   \
  } while (0)

#define PB_CHECK_LAUNCH() PB_CUDA(cudaGetLastError())

constexpr int kNumSMs = 148;          // B200: 2 dies x 74 SMs
constexpr int kBlock = 256;           // threads per CTA for the streaming kernels

struct Context {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool owns_stream = false;
  int num_sms = kNumSMs;
  unsigned long long launches = 0;    // kernels launched through this context
  // Optional device flag observed by every operator-apply kernel: while *skip_flag != 0 the
  // kernels return without touching memory.  Lets a device-resident loop (the CGLS projection of
  // BackendADMM, pb_admm.cu) stop early without a host round trip per inner iteration.
  const int* skip_flag = nullptr;
  // two pinned staging buffers for copies to / from pageable host memory (pb_hostio.cu), allocated on
  // first use and released by pb_context_destroy
  void* stage[2] = {nullptr, nullptr};
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};

  void bind() const { PB_CUDA(cudaSetDevice(device)); }
};

// ---- host <-> device copies (pb_hostio.cu) ----------------------------------------------------------
// Blocking copy of n floats from device memory into host memory.  Pinned / registered destinations are
// written by one DMA; pageable ones through the context's pinned staging ring with a multi-threaded
// copy-out, which is several times faster than cudaMemcpy into cold pageable memory (the final
// x, z, y, w read of Solver::Solve, solver.cu:152-167, is 400 MB for a 4096^2 image).
void download_to_host(Context* ctx, float* h, const float* d, size_t n);
// Blocking copy of n floats from host memory into device memory (same split; the source is only read).
void upload_from_host(Context* ctx, float* d, const float* h, size_t n);
// Touches every page of a pageable host range (content preserved) so that a later copy into it does not
// pay the first-touch page faults; no-op for pinned memory.  Safe to run on a helper thread.
void prefault_host_range(void* p, size_t bytes);
void release_host_staging(Context* ctx);

// PB_TRACE=1: wall-clock of the host-side phases (Problem::Initialize, Backend::Initialize, solution
// read-back ...) on stderr; the device is synchronised at both ends of a scope so that asynchronous work
// is attributed to the phase that enqueued it.  Off by default (no synchronisation, no output).
inline bool trace_enabled() {
  static const bool on = [] { const char* e = getenv("PB_TRACE"); return e && atoi(e) != 0; }();
  return on;
}
struct TraceScope {
  const char* name;
  std::chrono::steady_clock::time_point t0;
  explicit TraceScope(const char* n) : name(n) {
    if (trace_enabled()) { cudaDeviceSynchronize(); t0 = std::chrono::steady_clock::now(); }
  }
  ~TraceScope() {
    if (!trace_enabled()) return;
    cudaDeviceSynchronize();
    const double ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
    std::fprintf(stderr, "[pb trace] %-44s %9.3f ms\n", name, ms);
  }
};
#define PB_TRACE_CAT2(a, b) a##b
#define PB_TRACE_CAT(a, b) PB_TRACE_CAT2(a, b)
#define PB_TRACE_SCOPE(name) ::pb::TraceScope PB_TRACE_CAT(pb_trace_scope_, __LINE__)(name)

// ---- device memory (pb_hostio.cu) -----------------------------------------------------------------------
// cudaMalloc / cudaFree with a per-process cache of released blocks (exact-size reuse): a solver that is
// created, solved and destroyed repeatedly -- the reference's usage, one prost::Solver per solve -- asks for
// the same few buffer sizes every time, and cudaMalloc right after cudaFree of gigabytes costs up to 100 ms
// (measured: 3-97 ms for the first allocation of a solve), more than 500 fused PDHG iterations at 4096^2.
// A block enters the cache only after the device is idle (cudaDeviceSynchronize, like the implicit
// synchronisation of cudaFree), so it can be handed to any stream afterwards.  PB_POOL_MB caps the cached
// bytes per process (default 32768, 0 disables); pb_release_cached_memory() returns everything to the driver.
void* device_alloc(size_t bytes);                  // throws Error(PB_ERR_OOM / PB_ERR_CUDA)
void device_free(void* p, size_t bytes, int device);
void device_cache_release();
// pinned host blocks with exact-size reuse (pb_hostio.cu)
void* host_pool_alloc(size_t bytes);
void host_pool_free(void* p);

// RAII device allocation (replaces thrust::device_vector members of the reference).
template <typename T>
class DeviceBuffer {
 public:
  DeviceBuffer() = default;
  explicit DeviceBuffer(size_t n) { resize(n); }
  DeviceBuffer(const DeviceBuffer&) = delete;
  DeviceBuffer& operator=(const DeviceBuffer&) = delete;
  DeviceBuffer(DeviceBuffer&& o) noexcept : ptr_(o.ptr_), n_(o.n_), dev_(o.dev_) { o.ptr_ = nullptr; o.n_ = 0; }
  DeviceBuffer& operator=(DeviceBuffer&& o) noexcept {
    if (this != &o) { release(); ptr_ = o.ptr_; n_ = o.n_; dev_ = o.dev_; o.ptr_ = nullptr; o.n_ = 0; }
    return *this;
  }
  ~DeviceBuffer() { release(); }

  void resize(size_t n) {
    release();
    if (n == 0) return;
    ptr_ = static_cast<T*>(device_alloc(n * sizeof(T)));
    cudaGetDevice(&dev_);
    n_ = n;
  }
  void release() {
    if (ptr_) device_free(ptr_, n_ * sizeof(T), dev_);
    ptr_ = nullptr;
    n_ = 0;
  }
  void zero(cudaStream_t s) { if (n_) PB_CUDA(cudaMemsetAsync(ptr_, 0, n_ * sizeof(T), s)); }
  void upload(const T* h, size_t n, cudaStream_t s) {
    if (n > n_) fail(PB_ERR_INVALID, "DeviceBuffer::upload: size mismatch");
    if (n) PB_CUDA(cudaMemcpyAsync(ptr_, h, n * sizeof(T), cudaMemcpyHostToDevice, s));
  }
  void download(T* h, size_t n, cudaStream_t s) const {
    if (n > n_) fail(PB_ERR_INVALID, "DeviceBuffer::download: size mismatch");
    if (n) PB_CUDA(cudaMemcpyAsync(h, ptr_, n * sizeof(T), cudaMemcpyDeviceToHost, s));
  }
  void assign(const std::vector<T>& h, cudaStream_t s) {
    resize(h.size());
    upload(h.data(), h.size(), s);
    PB_CUDA(cudaStreamSynchronize(s));   // h may be a temporary
  }
  T* data() { return ptr_; }
  const T* data() const { return ptr_; }
  size_t size() const { return n_; }
  void swap(DeviceBuffer& o) { std::swap(ptr_, o.ptr_); std::swap(n_, o.n_); std::swap(dev_, o.dev_); }

 private:
  T* ptr_ = nullptr;
  size_t n_ = 0;
  int dev_ = 0;
};

// grid size for a 1-thread-per-item streaming kernel
inline unsigned grid_for(size_t items, int block = kBlock) {
  size_t g = (items + block - 1) / block;
  if (g == 0) g = 1;
  if (g > 0x7fffffffull) fail(PB_ERR_INVALID, "problem too large for a 1-D grid");
  return static_cast<unsigned>(g);
}

// 31-bit division by a runtime constant via multiply-high (Granlund-Montgomery): with
// s = ceil(log2 d) and m = ceil(2^(31+s) / d) (fits 32 bits), n / d == umulhi(n, m) >> (s-1)
// exactly for every n < 2^31.  Used to decode (x, y, l) from linear indices without the
// ~20-instruction hardware udiv sequence per element.
struct FastDiv {
  uint32_t d = 1, mul = 0, shift = 0;
  FastDiv() = default;
  explicit FastDiv(uint64_t div64) {
    if (div64 == 0 || div64 >= (1ull << 31)) fail(PB_ERR_INVALID, "FastDiv: divisor out of range");
    d = static_cast<uint32_t>(div64);
    if (d == 1) return;
    uint32_t s = 0;
    while ((1ull << s) < d) ++s;
    mul = static_cast<uint32_t>(((1ull << (31 + s)) + d - 1) / d);
    shift = s - 1;
  }
  __host__ __device__ __forceinline__ uint32_t div(uint32_t n) const {
    if (d == 1) return n;
#ifdef __CUDA_ARCH__
    return __umulhi(n, mul) >> shift;
#else
    return static_cast<uint32_t>((static_cast<uint64_t>(n) * mul) >> 32) >> shift;
#endif
  }
  __host__ __device__ __forceinline__ void divmod(uint32_t n, uint32_t& q, uint32_t& r) const {
    q = div(n);
    r = n - q * d;
  }
};

}  // namespace pb
