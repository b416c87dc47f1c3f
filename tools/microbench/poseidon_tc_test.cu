// GPU check + timing of the tensor-core Poseidon (csrc/poseidon_tc.cuh) against the dp2a form (csrc/poseidon.cuh)
// and the canonical host permutation.
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -lineinfo -o bin/poseidon_tc_test poseidon_tc_test.cu
//   ./bin/poseidon_tc_test [log2(states) | tiles of 128 states] [permutations per state]
#include "../../plonky2_bn254_b200/csrc/poseidon_tc.cuh"
#include <vector>
std::atomic<unsigned long long> g_pb_launches{0};

__global__ void __launch_bounds__(128, 6) k_ref(const u64* in, u64* out, size_t n, int reps) {
  __shared__ __align__(16) u64 rc2[poseidon::RC2_WORDS];
  for (int i = threadIdx.x; i < poseidon::RC2_WORDS; i += blockDim.x) rc2[i] = poseidon::RC2_DEV[i];
  __syncthreads();
  const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= n) return;
  u64 s[12];
  for (int i = 0; i < 12; i++) s[i] = in[i * n + j];
  for (int r = 0; r < reps; r++) poseidon::lazy::permute(s, rc2);
  for (int i = 0; i < 12; i++) out[i * n + j] = s[i];
}

__global__ void __launch_bounds__(128, poseidon::tc::CTAS_PER_SM) k_tc(const u64* in, u64* out, size_t n, int reps) {
  extern __shared__ unsigned char dyn[];
  __shared__ u64 bar;
  __shared__ u32 slot[2];
  poseidon::tc::Ctx c;
  poseidon::tc::setup(c, dyn, &bar, slot);
  const size_t j = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = j < n;
  u64 s[12];
  for (int i = 0; i < 12; i++) s[i] = live ? in[i * n + j] : 0;
  for (int r = 0; r < reps; r++) poseidon::tc::permute(s, c);
  if (live)
    for (int i = 0; i < 12; i++) out[i * n + j] = s[i];
  poseidon::tc::teardown(c);
}

#define CK(x)                                                                    \
  do {                                                                           \
    cudaError_t e = (x);                                                         \
    if (e != cudaSuccess) {                                                      \
      printf("%s: %s\n", #x, cudaGetErrorString(e));                             \
      return 1;                                                                  \
    }                                                                            \
  } while (0)

int main(int argc, char** argv) {
  // first argument: log2(states), or (>= 64) the number of 128-state tiles
  const int lg = argc > 1 ? atoi(argv[1]) : 20, reps = argc > 2 ? atoi(argv[2]) : 8;
  const size_t n = lg >= 64 ? (size_t)lg * 128 : (size_t)1 << lg;
  std::vector<u64> h(12 * n);
  u64 x = 0x9E3779B97F4A7C15ULL;
  for (auto& v : h) {
    x ^= x << 13; x ^= x >> 7; x ^= x << 17;
    v = x % gl::P;
  }
  // edge values in the first states
  for (int i = 0; i < 12; i++) { h[i * n + 0] = 0; h[i * n + 1] = gl::P - 1; h[i * n + 2] = 0xFFFFFFFFULL; h[i * n + 3] = 0xFFFFFFFF00000000ULL; }
  u64 *din, *d1, *d2;
  CK(cudaMalloc(&din, 96 * n)); CK(cudaMalloc(&d1, 96 * n)); CK(cudaMalloc(&d2, 96 * n));
  CK(cudaMemcpy(din, h.data(), 96 * n, cudaMemcpyHostToDevice));
  CK(cudaMemset(d2, 0xEE, 96 * n));
  CK(cudaFuncSetAttribute(k_tc, cudaFuncAttributeMaxDynamicSharedMemorySize, poseidon::tc::SMEM_BYTES));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  const unsigned grid = (unsigned)((n + 127) / 128);
  float ms_ref = 0, ms_tc = 0;
  for (int it = 0; it < 3; it++) {
    cudaEventRecord(e0);
    k_ref<<<grid, 128>>>(din, d1, n, reps);
    cudaEventRecord(e1);
    CK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms_ref, e0, e1);
  }
  printf("dp2a : %.3f ms, %.3f Gperm/s\n", ms_ref, n * (double)reps / ms_ref * 1e-6);
  fflush(stdout);
  for (int it = 0; it < 3; it++) {
    cudaEventRecord(e0);
    k_tc<<<grid, 128, poseidon::tc::SMEM_BYTES>>>(din, d2, n, reps);
    cudaEventRecord(e1);
    CK(cudaEventSynchronize(e1));
    cudaEventElapsedTime(&ms_tc, e0, e1);
  }
  CK(cudaGetLastError());
  printf("tcgen05 (ctas %d): %.3f ms, %.3f Gperm/s\n", poseidon::tc::CTAS_PER_SM, ms_tc, n * (double)reps / ms_tc * 1e-6);
  std::vector<u64> r1(12 * n), r2(12 * n);
  CK(cudaMemcpy(r1.data(), d1, 96 * n, cudaMemcpyDeviceToHost));
  CK(cudaMemcpy(r2.data(), d2, 96 * n, cudaMemcpyDeviceToHost));
  size_t bad = 0, first = (size_t)-1;
  for (size_t i = 0; i < 12 * n; i++)
    if (r1[i] != r2[i]) { if (!bad) first = i; bad++; }
  // host check of a few states
  size_t hostbad = 0;
  for (size_t j = 0; j < 64 && j < n; j++) {
    u64 s[12];
    for (int i = 0; i < 12; i++) s[i] = h[i * n + j];
    for (int r = 0; r < reps; r++) poseidon::permute_generic(s);
    for (int i = 0; i < 12; i++) hostbad += s[i] != r1[i * n + j];
  }
  printf("mismatches tc vs dp2a: %zu of %zu (first at %zu: lane %zu state %zu), dp2a vs host: %zu\n", bad, 12 * n, first,
         first == (size_t)-1 ? 0 : first / n, first == (size_t)-1 ? 0 : first % n, hostbad);
  if (bad) {
    for (int i = 0; i < 12; i++) printf("  lane %2d  want %016llx  got %016llx\n", i, (unsigned long long)r1[i * n + (first % n)], (unsigned long long)r2[i * n + (first % n)]);
  }
  printf(bad || hostbad ? "FAIL\n" : "OK\n");
  return bad || hostbad ? 2 : 0;
}
