// topolow_b200/csrc/common.cuh - shared device/host helpers.
#pragma once

#include <cuda_runtime.h>

#include <cfloat>
#include <chrono>
#include <cstdlib>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <stdexcept>
#include <string>

#define TL_HD __host__ __device__ __forceinline__
#define TL_D __device__ __forceinline__

namespace tl {

struct CudaError : std::runtime_error {
  using std::runtime_error::runtime_error;
};

inline void cuda_check(cudaError_t e, const char* what, const char* file, int line) {
  if (e != cudaSuccess) {
    char buf[512];
    std::snprintf(buf, sizeof buf, "CUDA error: %s (%s) at %s:%d", cudaGetErrorString(e), what, file, line);
    throw CudaError(buf);
  }
}
#define TL_CUDA(x) ::tl::cuda_check((x), #x, __FILE__, __LINE__)

// Owning handles: everything a host routine allocates is released on every exit path.
template <class T>
struct DeviceBuf {
  T* p = nullptr;
  DeviceBuf() {}
  explicit DeviceBuf(size_t count) { TL_CUDA(cudaMalloc(&p, (count ? count : 1) * sizeof(T))); }
  DeviceBuf(const DeviceBuf&) = delete;
  DeviceBuf& operator=(const DeviceBuf&) = delete;
  DeviceBuf(DeviceBuf&& o) noexcept : p(o.p) { o.p = nullptr; }
  ~DeviceBuf() { if (p) cudaFree(p); }
  T* release() { T* r = p; p = nullptr; return r; }
  operator T*() const { return p; }
};
// Stream-ordered scratch from the device's default memory pool (kept by the pool between calls: the
// first fit pays for the allocation, the following ones reuse it).
template <class T>
struct AsyncBuf {
  T* p = nullptr;
  cudaStream_t s = nullptr;
  AsyncBuf(size_t count, cudaStream_t stream) : s(stream) {
    TL_CUDA(cudaMallocAsync((void**)&p, (count ? count : 1) * sizeof(T), stream));
  }
  AsyncBuf(const AsyncBuf&) = delete;
  AsyncBuf& operator=(const AsyncBuf&) = delete;
  ~AsyncBuf() { if (p) cudaFreeAsync(p, s); }
  T* release() { T* r = p; p = nullptr; return r; }
  operator T*() const { return p; }
};
// Long-lived device buffers of plans and edge stores come from the same pool (a CV grid creates and
// destroys hundreds of plans per call; cudaMalloc / cudaFree would serialise them on the driver).
template <class T>
inline void pool_alloc(T*& p, size_t bytes) {
  TL_CUDA(cudaMallocAsync((void**)&p, bytes ? bytes : 1, cudaStreamPerThread));
}
inline void pool_ready() { TL_CUDA(cudaStreamSynchronize(cudaStreamPerThread)); }   // allocations usable on any stream
inline void pool_free(void* p) { if (p) cudaFreeAsync(p, cudaStreamPerThread); }
// Makes `device` current for the lifetime of the object (destructors free on the device that owns the memory).
struct DeviceScope {
  int prev = -1;
  explicit DeviceScope(int device) { if (cudaGetDevice(&prev) != cudaSuccess) prev = -1; if (prev != device) cudaSetDevice(device); else prev = -1; }
  DeviceScope(const DeviceScope&) = delete;
  ~DeviceScope() { if (prev >= 0) cudaSetDevice(prev); }
};
inline void keep_pool_memory(int device) {
  cudaMemPool_t pool;
  if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
    unsigned long long keep = ~0ull;
    cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
  }
}
template <class T>
struct PinnedBuf {
  T* p = nullptr;
  PinnedBuf() {}
  explicit PinnedBuf(size_t count, unsigned flags = cudaHostAllocDefault) {
    TL_CUDA(cudaHostAlloc((void**)&p, (count ? count : 1) * sizeof(T), flags));
  }
  PinnedBuf(const PinnedBuf&) = delete;
  PinnedBuf& operator=(const PinnedBuf&) = delete;
  PinnedBuf(PinnedBuf&& o) noexcept : p(o.p) { o.p = nullptr; }
  ~PinnedBuf() { if (p) cudaFreeHost(p); }
  operator T*() const { return p; }
};
struct StreamGuard {
  cudaStream_t s = nullptr;
  StreamGuard() { TL_CUDA(cudaStreamCreate(&s)); }
  StreamGuard(const StreamGuard&) = delete;
  ~StreamGuard() { if (s) cudaStreamDestroy(s); }
  operator cudaStream_t() const { return s; }
};
struct EventGuard {
  cudaEvent_t e = nullptr;
  explicit EventGuard(unsigned flags = cudaEventDefault) { TL_CUDA(cudaEventCreateWithFlags(&e, flags)); }
  EventGuard(const EventGuard&) = delete;
  ~EventGuard() { if (e) cudaEventDestroy(e); }
  operator cudaEvent_t() const { return e; }
};

// Phase timer for TOPOLOW_DEBUG=1 runs: prints host wall-clock milliseconds per labelled phase (and
// synchronises the stream at every mark, so it is off unless asked for).
struct PhaseTimer {
  bool on;
  cudaStream_t s;
  std::chrono::steady_clock::time_point t;
  explicit PhaseTimer(cudaStream_t stream) : on(std::getenv("TOPOLOW_DEBUG") != nullptr), s(stream), t(std::chrono::steady_clock::now()) {}
  void mark(const char* what) {
    if (!on) return;
    cudaStreamSynchronize(s);
    const auto now = std::chrono::steady_clock::now();
    std::fprintf(stderr, "[topolow] %-28s %8.2f ms\n", what, std::chrono::duration<double, std::milli>(now - t).count());
    t = now;
  }
};

// ---------------------------------------------------------------------------
// Convergence controller.  One instance per fit lives in device memory and is
// advanced by one thread; the host reads it back between launches.
// Follows src/optimization.cpp:168-181 (state), :289 (cooling), :294-357
// (three-way classification), :368-374 (restore).
// ---------------------------------------------------------------------------
struct FitParams {
  int n_iter;
  double k0, cooling_rate, c_repulsion, relative_epsilon;
  int convergence_window, convergence_check_freq;
};

struct FitState {
  double k;              // current spring constant
  double best_mae;       // DBL_MAX until the first check
  double best_k;
  double last_error;     // MAE of the latest check
  int best_iter;
  int worsening_count;
  int converge_count;
  int converged;         // plateau or worsening exit taken
  int stop;              // loop must not run further iterations (converged or failed)
  int iter;              // iterations completed so far
  int snapshot;          // set by controller_check when best_* was updated by this check
  int status;            // 0 ok, 2 non-finite, kStatusStopped
  int fail_iter;
  int pad;
  unsigned long long pair_updates;
};

// FitState::status of a fit that the caller stopped through the batch's abort word (TileDev::abort) before it
// converged or ran all its iterations (the value of TOPOLOW_ERR_INTERRUPTED).
constexpr int kStatusStopped = 5;

TL_HD void state_init(FitState& s, const FitParams& p) {
  s.k = p.k0;
  s.best_mae = DBL_MAX;
  s.best_k = p.k0;
  s.last_error = 0.0;
  s.best_iter = 0;
  s.worsening_count = 0;
  s.converge_count = 0;
  s.converged = 0;
  s.stop = 0;
  s.iter = 0;
  s.snapshot = 0;
  s.status = 0;
  s.fail_iter = 0;
  s.pad = 0;
  s.pair_updates = 0ULL;
}

TL_HD bool is_check_iter(int iter /*0-based, just completed*/, const FitParams& p) {
  int freq = p.convergence_check_freq < 1 ? 10 : p.convergence_check_freq;
  return ((iter + 1) % freq == 0) || (iter == p.n_iter - 1);
}

// `iter` is the 0-based iteration that just finished; s.k already cooled.
// Sets s.snapshot when the caller must copy positions -> best positions.
TL_HD void controller_check(FitState& s, const FitParams& p, int iter, double total, long long count) {
  const double current_error = (count > 0) ? total / (double)count : 0.0;
  s.last_error = current_error;
  s.snapshot = 0;
  const double improvement_threshold = s.best_mae * (1.0 - p.relative_epsilon);
  const double worsening_threshold = s.best_mae * (1.0 + p.relative_epsilon);
  if (current_error < improvement_threshold) {
    s.best_mae = current_error; s.best_k = s.k; s.best_iter = iter + 1; s.snapshot = 1;
    s.worsening_count = 0; s.converge_count = 0;
  } else if (current_error <= worsening_threshold) {
    if (current_error < s.best_mae) {
      s.best_mae = current_error; s.best_k = s.k; s.best_iter = iter + 1; s.snapshot = 1;
    }
    s.worsening_count = 0;
    s.converge_count++;
    if (s.converge_count >= p.convergence_window) { s.converged = 1; s.stop = 1; }
  } else {
    s.converge_count = 0;
    s.worsening_count++;
    if (s.worsening_count >= p.convergence_window) { s.converged = 1; s.stop = 1; }
  }
}

// ---------------------------------------------------------------------------
// Small stateless integer mixing used by the schedule (host == device).
// ---------------------------------------------------------------------------
TL_HD uint64_t mix64(uint64_t x) {
  x ^= x >> 30; x *= 0xbf58476d1ce4e5b9ULL;
  x ^= x >> 27; x *= 0x94d049bb133111ebULL;
  x ^= x >> 31;
  return x;
}

}  // namespace tl
