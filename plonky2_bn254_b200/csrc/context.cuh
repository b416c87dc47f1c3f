// Per-GPU prover context: stream, twiddle/shift tables and a bump-allocated device workspace that
// is grown on demand and reused across proofs of the same shape (no cudaMalloc on the hot path).
#pragma once
#include "ntt_tables.cuh"
#include <vector>
#include <string>
#include <time.h>

struct Arena {
  char* base = nullptr;
  size_t cap = 0, off = 0, high = 0;
  // The caller sizes the arena from the proof shape before the first kernel is launched; not fitting is reported
  // as PB254_E_OOM like a failed cudaMalloc of the reservation itself.
  void* alloc(size_t bytes) {
    size_t a = (off + 255) & ~(size_t)255;
    if (a + bytes > cap) throw Pb254Error(5 /* PB254_E_OOM */, "device workspace exhausted");
    off = a + bytes;
    if (off > high) high = off;
    return base + a;
  }
  template <class T>
  T* alloc_n(size_t n) { return (T*)alloc(n * sizeof(T)); }
  void reset() { off = 0; }
  void reserve(size_t bytes) {
    if (bytes <= cap) return;
    if (base) pb_dev_free(base);
    base = nullptr;
    cap = 0;
    base = (char*)pb_dev_alloc(bytes);
    cap = bytes;
  }
  void destroy() {
    if (base) pb_dev_free(base);
    base = nullptr;
    cap = off = 0;
  }
};

// Per-stage device timing: CUDA events on the context's stream, resolved after the stream is
// synchronised. bench.py reads these for the roofline figures.
struct StageTimes {
  struct Rec {
    std::string name;
    double ms;
#if !PB_HOSTSIM
    cudaEvent_t a, b;
#else
    double t0;
#endif
  };
  std::vector<Rec> recs;
  bool enabled = true;
  StageTimes() = default;
  ~StageTimes() { clear(); }  // the events belong to this object: no copies
  StageTimes(const StageTimes&) = delete;
  StageTimes& operator=(const StageTimes&) = delete;
#if PB_HOSTSIM
  static double now() {
    struct timespec ts;
    clock_gettime(CLOCK_MONOTONIC, &ts);
    return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
  }
#endif
  void clear() {
#if !PB_HOSTSIM
    for (auto& r : recs) {
      cudaEventDestroy(r.a);
      cudaEventDestroy(r.b);
    }
#endif
    recs.clear();
  }
  int begin(const char* name, pbStream s) {
    if (!enabled) return -1;
    Rec r;
    r.name = name;
    r.ms = 0;
#if !PB_HOSTSIM
    PB_CUDA(cudaEventCreate(&r.a));
    PB_CUDA(cudaEventCreate(&r.b));
    PB_CUDA(cudaEventRecord(r.a, s));
#else
    (void)s;
    r.t0 = now();
#endif
    recs.push_back(r);
    return (int)recs.size() - 1;
  }
  void end(int id, pbStream s) {
    if (id < 0) return;
#if !PB_HOSTSIM
    PB_CUDA(cudaEventRecord(recs[id].b, s));
#else
    (void)s;
    recs[id].ms = now() - recs[id].t0;
#endif
  }
  void end_nothrow(int id, pbStream s) noexcept {
    if (id < 0) return;
#if !PB_HOSTSIM
    (void)cudaEventRecord(recs[id].b, s);  // an error here is sticky and is reported by the next pb_sync
#else
    (void)s;
    recs[id].ms = now() - recs[id].t0;
#endif
  }
  // call after the stream has been synchronised
  void resolve() {
#if !PB_HOSTSIM
    for (auto& r : recs) {
      float ms = 0;
      if (cudaEventElapsedTime(&ms, r.a, r.b) == cudaSuccess) r.ms = ms;
    }
#endif
  }
};

struct pb254_ctx {
  int device = 0;
  pbStream stream = 0;
  bool own_stream = false;
  ntt::TableSet tables;
  Arena arena;
  StageTimes times;
  void* g2_pow2 = nullptr;  // hash_to_g2's fixed-base table 2^j G2 (h2g2::TableK), built by the first call
};
