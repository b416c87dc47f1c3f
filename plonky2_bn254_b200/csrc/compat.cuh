// Build-mode glue.
//
// Product build (nvcc, sm_100a): every kernel is a real CUDA kernel; there is NO CPU fallback.
// Test-only "hostsim" build (g++ -DPB254_HOSTSIM, output tests/hostsim/libpb254_hostsim.so):
// the same source compiled for the CPU so that host orchestration (transcript, proof assembly,
// kernel argument plumbing) and the per-thread kernel bodies can be checked against the oracle
// in the GPU-less container. The product package never loads the hostsim library.
#pragma once
#include <cstdint>
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <stdexcept>
#include <string>
#include <atomic>
#include <mutex>
#include <algorithm>

typedef uint64_t u64;
typedef uint32_t u32;
typedef int64_t i64;
typedef unsigned __int128 u128;

struct Pb254Error : std::runtime_error {
  int code;
  Pb254Error(int c, const std::string& m) : std::runtime_error(m), code(c) {}
};

#ifdef PB254_HOSTSIM
// ------------------------------------------------------------------------------------------
#define PB_HD inline
#define PB_D inline
#define PB_INLINE inline
#define PB_HOSTSIM 1
typedef void* pbStream;
static inline void pb_check_last(const char*) {}
static inline void* pb_dev_alloc(size_t bytes) {
  void* p = malloc(bytes ? bytes : 1);
  if (!p) throw Pb254Error(5, "hostsim: out of memory");
  return p;
}
static inline void pb_dev_free(void* p) { free(p); }
static inline void pb_h2d(void* d, const void* h, size_t n, pbStream) { memcpy(d, h, n); }
static inline void pb_d2h(void* h, const void* d, size_t n, pbStream) { memcpy(h, d, n); }
static inline void pb_d2d(void* d, const void* s, size_t n, pbStream) { memmove(d, s, n); }
static inline void pb_memset(void* d, int v, size_t n, pbStream) { memset(d, v, n); }
// `height` rows of `width` bytes, row r at d + r * dpitch / s_ + r * spitch (device to device)
static inline void pb_copy2d(void* d, size_t dpitch, const void* s_, size_t spitch, size_t width, size_t height, pbStream) {
  for (size_t r = 0; r < height; r++) memmove((char*)d + r * dpitch, (const char*)s_ + r * spitch, width);
}
static inline void pb_sync(pbStream) {}
static inline void pb_set_device(int) {}
struct PbDeviceGuard {
  explicit PbDeviceGuard(int) {}
};

extern std::atomic<unsigned long long> g_pb_launches;
template <class F>
static inline void pb_launch(const char*, F f, size_t n, pbStream, int = 256) {
#pragma omp parallel for schedule(static)
  for (size_t gid = 0; gid < n; gid++) f(gid);
}
template <int THREADS, int MIN_CTAS, class F>
static inline void pb_launch_lb(const char* name, F f, size_t n, pbStream s) {
  pb_launch(name, f, n, s);
}
#else
// ------------------------------------------------------------------------------------------
#include <cuda_runtime.h>
#define PB_HD __host__ __device__ __forceinline__
#define PB_D __device__ __forceinline__
#define PB_INLINE __forceinline__
#define PB_HOSTSIM 0
typedef cudaStream_t pbStream;

#define PB_CUDA(call)                                                                              \
  do {                                                                                             \
    cudaError_t e_ = (call);                                                                       \
    if (e_ != cudaSuccess)                                                                         \
      throw Pb254Error(e_ == cudaErrorMemoryAllocation ? 5 : 4,                                    \
                       std::string(#call) + ": " + cudaGetErrorString(e_));                        \
  } while (0)

static inline void pb_check_last(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) throw Pb254Error(4, std::string(what) + ": " + cudaGetErrorString(e));
}
static inline void* pb_dev_alloc(size_t bytes) {
  void* p = nullptr;
  PB_CUDA(cudaMalloc(&p, bytes ? bytes : 1));
  return p;
}
static inline void pb_dev_free(void* p) { cudaFree(p); }
static inline void pb_h2d(void* d, const void* h, size_t n, pbStream s) {
  PB_CUDA(cudaMemcpyAsync(d, h, n, cudaMemcpyHostToDevice, s));
}
static inline void pb_d2h(void* h, const void* d, size_t n, pbStream s) {
  PB_CUDA(cudaMemcpyAsync(h, d, n, cudaMemcpyDeviceToHost, s));
}
static inline void pb_d2d(void* d, const void* s_, size_t n, pbStream s) {
  PB_CUDA(cudaMemcpyAsync(d, s_, n, cudaMemcpyDeviceToDevice, s));
}
static inline void pb_memset(void* d, int v, size_t n, pbStream s) { PB_CUDA(cudaMemsetAsync(d, v, n, s)); }
// `height` rows of `width` bytes, row r at d + r * dpitch / s_ + r * spitch (device to device)
static inline void pb_copy2d(void* d, size_t dpitch, const void* s_, size_t spitch, size_t width, size_t height,
                             pbStream s) {
  if (width && height) PB_CUDA(cudaMemcpy2DAsync(d, dpitch, s_, spitch, width, height, cudaMemcpyDeviceToDevice, s));
}
static inline void pb_sync(pbStream s) { PB_CUDA(cudaStreamSynchronize(s)); }
static inline void pb_set_device(int d) { PB_CUDA(cudaSetDevice(d)); }
// An entry point works on its context's device and leaves the CALLER's current device as it found it (the host
// language - torch, a Rust CUDA binding - keeps its own notion of the current device).
struct PbDeviceGuard {
  int prev = -1;
  explicit PbDeviceGuard(int d) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != d) PB_CUDA(cudaSetDevice(d));
  }
  ~PbDeviceGuard() {
    if (prev >= 0) (void)cudaSetDevice(prev);
  }
  PbDeviceGuard(const PbDeviceGuard&) = delete;
  PbDeviceGuard& operator=(const PbDeviceGuard&) = delete;
};
// free memory of device d (bytes)
static inline size_t pb_free_bytes(int d) {
  PbDeviceGuard device_guard(d);
  size_t free_b = 0, total_b = 0;
  PB_CUDA(cudaMemGetInfo(&free_b, &total_b));
  return free_b;
}

// launch counter (reported by bench.py as gpu_launches)
extern std::atomic<unsigned long long> g_pb_launches;

template <class F>
__global__ void pb_kernel(F f, size_t n) {
  size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid < n) f(gid);
}
// Same with a register budget: at least MIN_CTAS resident CTAs of THREADS threads per SM.
template <class F, int THREADS, int MIN_CTAS>
__global__ void __launch_bounds__(THREADS, MIN_CTAS) pb_kernel_lb(F f, size_t n) {
  size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (gid < n) f(gid);
}
template <int THREADS, int MIN_CTAS, class F>
static inline void pb_launch_lb(const char* name, F f, size_t n, pbStream s) {
  if (n == 0) return;
  size_t grid = (n + THREADS - 1) / THREADS;
  pb_kernel_lb<F, THREADS, MIN_CTAS><<<(unsigned)grid, THREADS, 0, s>>>(f, n);
  g_pb_launches++;
  pb_check_last(name);
}
// One thread per work item; functor passed by value. `name` only documents the call site.
template <class F>
static inline void pb_launch(const char* name, F f, size_t n, pbStream s, int block = 256) {
  if (n == 0) return;
  size_t grid = (n + block - 1) / block;
  pb_kernel<F><<<(unsigned)grid, block, 0, s>>>(f, n);
  g_pb_launches++;
  pb_check_last(name);
}
#endif
