// Poseidon-Goldilocks with the linear layer on the 5th-generation tensor cores (tcgen05, sm_100a).
// Same function as poseidon::lazy::permute (plonky2 0.2.2 hash/poseidon.rs::Poseidon::poseidon, reached from
// src/starks/common/prover.rs:31-38 through PolynomialBatch::from_values / MerkleTree::new), bit-identical
// results; used by the leaf-hash kernel, where > 99 % of a proof's permutations are.
//
// Why. The dp2a form of the MDS layer (poseidon.cuh) costs 288 IDP.2A + ~215 recombination instructions per
// layer and thread and keeps the FMA-heavy pipe 85 % busy; 30 layers are 62 % of the 24.5 k instructions of a
// permutation. The layer IS a matrix product with 6-bit entries, so one CTA of 128 threads (one sponge state per
// thread) hands it to the tensor core as a u8 x u8 -> s32 product:
//
//   A [128 states x 128 k]   row t = the 96 bytes of thread t's state (k = 8 i + q: byte q of lane i, i.e. the
//                            little-endian u64 lanes as they are - no piece extraction) followed by 32 bytes that
//                            depend on the layer (below); shared memory, K-major, 128-byte swizzle
//   B [ 96 n      x 128 k]   one of two constant 12 KB tiles (tools/gen_poseidon_constants.py), n = 8 r + q'
//   D [128 states x  96 n]   s32 in tensor memory: D[t][8 r + q'] = the byte-weight q' sum of output lane r, < 2^20
//
// A permutation is 19 products: 4 full rounds, 11 FUSED layers of two partial rounds each, 4 full rounds.
//   full round L     B = poseidon_constants_tcb.inc: B[n][8 i + q] = MDS[r][i] (q == q'), B[n][96 + L] = byte q' of
//                    the NEXT round's constant of lane r; A[96 + L] = 1 (a one-hot of the round: the constant
//                    addition rides along), the rest of k = 96 .. 127 zero
//   partial rounds   B = poseidon_constants_tcf.inc. With s' = the state after round r's S-box (r = 4, 6, .., 24) and
//   r, r + 1         u0 = row 0 of MDS s' + RC[r + 1][0], which the thread computes itself (12 dp2a products of 16-bit
//                    pieces, as in poseidon.cuh), the two rounds are
//                      v = (M P M) s' + sbox(u0) M e0 + M P RC[r + 1] + RC[r + 2]      (P zeroes lane 0)
//                    M P M has 13-bit entries, taken as lo + 256 hi over two byte weights; the one product that
//                    would land at weight 8 (hi byte7 2^64) is reduced with 2^64 = 2^32 - 1 (mod p) through a
//                    complement byte 255 - byte7 of each lane. A[96 .. 103] = sbox(u0), A[104 + j] = 1 (fused layer
//                    j), A[115 + i] = 255 - byte 7 of lane i, A[127] = 0.
// So both kinds of layer have the same 96 output columns and the same fold; a fused layer costs the thread two
// S-boxes and one 12-term row product, and saves the whole CTA round trip and the 12-lane fold of a partial round.
//
// tcgen05.mma.kind::i8 products (M 128, K 32 per instruction: four K steps, each as an N = 64 and an N = 32 half, see
// CTAS_PER_SM below) per layer, issued by one thread, completion through an mbarrier;
// every thread then reads its own row of D with tcgen05.ld (TMEM lane = state = thread), folds the eight byte-weight
// sums of each lane into a lazy u64 representative (4 shift-adds + the 15-instruction piece recombination of the
// dp2a form) and goes on with the S-boxes. Per layer and thread: 8 shared-memory stores, 1 barrier, 3 TMEM loads
// and ~230 ALU instructions instead of ~500, and the FMA pipe is left to the S-box multiplications.
// Five CTAs per SM (5 x (64 + 32) TMEM columns, 5 x 41 KB shared memory) hide the MMA round trip of one CTA behind
// the S-boxes and recombinations of the others.
#pragma once
#include "poseidon.cuh"

#if !PB_HOSTSIM
namespace poseidon {
namespace tc {

static constexpr int CTA = 128;                 // threads = states = TMEM lanes per CTA
static constexpr int A_BYTES = 128 * 128;       // state tile
static constexpr int B_BYTES = 96 * 128;        // one B tile (MDS + round constants, or the fused partial rounds)
// Tensor memory: 512 columns per SM, allocations are powers of two >= 32. The 96 accumulator columns are taken as
// 64 + 32 (two allocations, the product is issued as an N = 64 and an N = 32 half), so FIVE CTAs fit on an SM instead
// of four; the shared-memory request keeps a sixth from becoming resident (it would spin in tcgen05.alloc):
// A + two B tiles + alignment slack = 41 KB, 5 x 42 KB with the per-CTA reservation fit in 228 KB, 6 do not.
static constexpr int CTAS_PER_SM = 5;
static constexpr int SMEM_BYTES = 41 * 1024;
static_assert(A_BYTES + 2 * B_BYTES + 1024 <= SMEM_BYTES && SMEM_BYTES <= 48 * 1024, "shared-memory plan");
// instruction descriptor (kind::i8): D = s32 (2 << 4), A = B = u8 (0), both K-major, N (>> 3 at bit 17),
// M = 128 (>> 4 at bit 24)
__host__ __device__ constexpr u32 idesc(u32 n) { return (2u << 4) | ((n >> 3) << 17) | ((128u >> 4) << 24); }

static __device__ const uint4 B_IMAGE[B_BYTES / 16] = {
#include "poseidon_constants_tcb.inc"
};
static __device__ const uint4 BF_IMAGE[B_BYTES / 16] = {
#include "poseidon_constants_tcf.inc"
};

__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }

// shared-memory matrix descriptor: K-major, 128-byte swizzle, 8-row groups 1024 bytes apart, version 1 (sm_100)
__device__ __forceinline__ u64 smem_desc(u32 addr) {
  return (u64)((addr & 0x3FFFFu) >> 4) | ((u64)(1024u >> 4) << 32) | (1ull << 46) | (2ull << 61);
}

struct Ctx {
  unsigned char* row;  // this thread's row of the A tile
  u32 r7;              // row & 7: the swizzle of this row
  u32 bar;             // mbarrier (shared address)
  u32 tmem0, tmem1;    // the two TMEM allocations (64 and 32 columns: lanes 0-7 and 8-11 of the state)
  u64 adesc, bdesc, bfdesc;  // A tile, full-round B tile, fused-partial-round B tile
  u32 parity;
};

// Called by all 128 threads. dyn: dynamic shared memory (SMEM_BYTES); bar / slot: 8 + 2 x 4 bytes of static shared memory.
__device__ __forceinline__ void setup(Ctx& c, unsigned char* dyn, u64* bar, u32* slot) {
  const u32 t = threadIdx.x;
  unsigned char* base = dyn + ((1024u - (smem_u32(dyn) & 1023u)) & 1023u);
  unsigned char* a = base;
  unsigned char* b = base + A_BYTES;
  unsigned char* bf = b + B_BYTES;
  for (int i = t; i < B_BYTES / 16; i += CTA) {
    reinterpret_cast<uint4*>(b)[i] = B_IMAGE[i];
    reinterpret_cast<uint4*>(bf)[i] = BF_IMAGE[i];
  }
  c.row = a + t * 128;
  c.r7 = t & 7;
  c.bar = smem_u32(bar);
  if (t == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(c.bar));
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (t < 32) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 64;" ::"r"(smem_u32(slot)) : "memory");
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 32;" ::"r"(smem_u32(slot + 1)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  c.tmem0 = reinterpret_cast<volatile u32*>(slot)[0];
  c.tmem1 = reinterpret_cast<volatile u32*>(slot)[1];
  c.adesc = smem_desc(smem_u32(a));
  c.bdesc = smem_desc(smem_u32(b));
  c.bfdesc = smem_desc(smem_u32(bf));
  c.parity = 0;
}

__device__ __forceinline__ void teardown(const Ctx& c) {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x < 32) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 64;" ::"r"(c.tmem0) : "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 32;" ::"r"(c.tmem1) : "memory");
  }
}

template <u32 N>
__device__ __forceinline__ void mma_i8(u32 d_tmem, u64 adesc, u64 bdesc, u32 accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(adesc), "l"(bdesc), "n"(idesc(N)), "r"(accumulate)
      : "memory");
}

#define PB_TMEM_LD32(v, addr)                                                                                       \
  asm volatile(                                                                                                     \
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, "   \
      "%15, %16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"                \
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]), "=r"(v[8]), \
        "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]), "=r"(v[16]),      \
        "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]), "=r"(v[24]),     \
        "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])                   \
      : "r"(addr)                                                                                                   \
      : "memory")

// acc0 + acc1 2^16 + acc2 2^32 + acc3 2^48 (acc < 2^31) -> some u64 congruent to it; ALU pipe only (poseidon.cuh)
__device__ __forceinline__ u64 recombine4(u32 acc0, u32 acc1, u32 acc2, u32 acc3) {
  const u32 t1 = __byte_perm(acc1, 0, 0x1044), u1 = __byte_perm(acc1, 0, 0x4432);
  const u32 t3 = __byte_perm(acc3, 0, 0x1044), u3 = __byte_perm(acc3, 0, 0x4432);
  u32 lo, hi;
  asm("{\n\t"
      ".reg .u32 w2, c;\n\t"
      "add.cc.u32   %0, %2, %3;\n\t"
      "addc.u32     %1, %4, %5;\n\t"
      "add.cc.u32   %1, %1, %6;\n\t"
      "addc.u32     w2, %7, 0;\n\t"
      "add.cc.u32   %1, %1, w2;\n\t"
      "addc.u32     c, 0, 0;\n\t"
      "sub.cc.u32   %0, %0, w2;\n\t"
      "subc.u32     %1, %1, 0;\n\t"
      "sub.u32      c, 0, c;\n\t"
      "add.cc.u32   %0, %0, c;\n\t"
      "addc.u32     %1, %1, 0;\n\t"
      "}"
      : "=&r"(lo), "=&r"(hi)
      : "r"(acc0), "r"(t1), "r"(u1), "r"(acc2), "r"(t3), "r"(u3));
  return ((u64)hi << 32) | lo;
}

// The eight byte-weight sums a_q < 2^20 of one lane -> a lazy u64 representative of sum a_q 2^(8 q).
__device__ __forceinline__ u64 fold8(const u32* q) {
  return recombine4(q[0] + (q[1] << 8), q[2] + (q[3] << 8), q[4] + (q[5] << 8), q[6] + (q[7] << 8));
}

// Measured and dropped (tools/microbench/poseidon_tc_test.cu, 2^20 states x 16 permutations, on the one-round-per-
// product form: 1.246 Gperm/s; the dp2a form 1.09, this form 1.443): one 128-column allocation and one N = 96 product
// per K step with four CTAs per SM (1.20); one
// persistent CTA of 4 or 5 groups of 128 threads on named barriers owning all 512 columns (1.20 / 1.16, top stall
// `barrier`); one TMEM wait for all 96 columns (1.22); the fold in plain 128-bit integer code (ptxas moves a third
// of it to the FMA pipe but emits 23 instead of 19 instructions: 1.13); the wrap correction of the multiplication on
// the FMA pipe (1.23); twelve S-boxes unrolled (1.25, not worth the code); the S-box of a partial round interleaved
// with the folds of the other eleven lanes (1.24); a fold that ptxas keeps on the FMA pipe (four IMAD and three
// IMAD.WIDE with the running value as 64-bit addend, 15 instructions with 8 on the ALU pipe instead of 19 with 17: 1.257
// against 1.264 on 8140 tiles) - i.e. neither the ALU pipe nor the instruction count binds: with five warps per
// scheduler the kernel is bound by the latency of its serial phases (S-box chain, barrier, product round trip, TMEM
// load). ncu (profiles/): 18.1 k thread-instructions per permutation against 24.5 k, issue slots 64 % busy, ALU pipe
// 71 %, FMA pipe 24 %, tensor pipe 20 %; 128-row tiles beyond a whole number of waves cost little (8192 tiles on 740
// CTA slots: +1.6 % time for +0.6 % work, the lone CTAs of the last wave run faster). That is why the partial rounds
// are now fused in pairs: 30 -> 19 of those round trips per permutation.

// byte p (0 .. 31) of k = 96 .. 127 set to 1, as word w of the two 16-byte chunks; p outside 0 .. 31: nothing set
__device__ __forceinline__ u32 onehot(int p, int w) { return (p >> 2) == w ? 1u << ((p & 3) * 8) : 0u; }

// 255 - byte 7 of lanes i0, i1, i2, i3 (as bytes 0 .. 3)
__device__ __forceinline__ u32 complement4(const u64 s[12], int i0, int i1, int i2, int i3) {
  const u32 a = __byte_perm((u32)(s[i0] >> 32), (u32)(s[i1] >> 32), 0x0073);
  const u32 b = __byte_perm((u32)(s[i2] >> 32), (u32)(s[i3] >> 32), 0x0073);
  return ~__byte_perm(a, b, 0x5410);
}

// s <- the product of the A row (the state, then x6 / x7 as k = 96 .. 127) with the B tile `bdesc`, all 128 threads
// of the CTA together
__device__ __forceinline__ void product(u64 s[12], Ctx& c, u64 bdesc, uint4 x6, uint4 x7) {
#pragma unroll
  for (int ch = 0; ch < 6; ch++)
    *reinterpret_cast<uint4*>(c.row + ((ch ^ c.r7) << 4)) =
        make_uint4((u32)s[2 * ch], (u32)(s[2 * ch] >> 32), (u32)s[2 * ch + 1], (u32)(s[2 * ch + 1] >> 32));
  *reinterpret_cast<uint4*>(c.row + ((6 ^ c.r7) << 4)) = x6;
  *reinterpret_cast<uint4*>(c.row + ((7 ^ c.r7) << 4)) = x7;
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // generic-proxy stores -> visible to the tensor core
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (threadIdx.x == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
#pragma unroll
    for (int k = 0; k < 4; k++) {  // 32 bytes of K per step; B rows 0-63 (lanes 0-7) and 64-95 (lanes 8-11)
      mma_i8<64>(c.tmem0, c.adesc + 2 * k, bdesc + 2 * k, k > 0);
      mma_i8<32>(c.tmem1, c.adesc + 2 * k, bdesc + (64 * 128 >> 4) + 2 * k, k > 0);
    }
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(c.bar) : "memory");
  }
  {
    u32 ok;
    do {
      asm volatile(
          "{\n\t"
          ".reg .pred p;\n\t"
          "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
          "selp.u32 %0, 1, 0, p;\n\t"
          "}"
          : "=r"(ok)
          : "r"(c.bar), "r"(c.parity)
          : "memory");
    } while (!ok);
    c.parity ^= 1;
  }
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  {
    const u32 lane_off = ((threadIdx.x >> 5) * 32u) << 16;  // a warp reads the 32 TMEM lanes of its own states
    const u32 t0 = c.tmem0 + lane_off, t1 = c.tmem0 + lane_off + 32, t2 = c.tmem1 + lane_off;
#define PB_TC_FOLD(a, base)                                                                                   \
  _Pragma("unroll") for (int r = 0; r < 4; r++) {                                                             \
    const u32* q = a + 8 * r;                                                                                 \
    s[base + r] = fold8(q);                                                                                   \
  }
    // the next 32 columns are in flight while the previous 32 are folded
    u32 a[32], b[32];
    PB_TMEM_LD32(a, t0);
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    PB_TMEM_LD32(b, t1);
    PB_TC_FOLD(a, 0)
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    PB_TMEM_LD32(a, t2);
    PB_TC_FOLD(b, 4)
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    PB_TC_FOLD(a, 8)
#undef PB_TC_FOLD
  }
}

// Inputs canonical, outputs canonical; every thread of the CTA must call it (threads without work pass zeros).
__device__ __forceinline__ void permute(u64 s[12], Ctx& c) {
#pragma unroll
  for (int i = 0; i < 12; i++) {
    const u64 k = RC_DEV[i];
    u64 t = s[i] + k;
    if (t < k) t += gl::EPS;
    s[i] = t;
  }
  // layers 0-3 and 15-18: full rounds 0-3 and 26-29; layer 4 + j: partial rounds 4 + 2 j and 5 + 2 j
  constexpr int N_FUSED = N_PARTIAL / 2, N_LAYERS = 2 * HALF_FULL + N_FUSED;
#pragma unroll 1
  for (int L = 0; L < N_LAYERS; L++) {
    uint4 x6, x7;
    u64 bdesc;
    if (L < HALF_FULL || L >= HALF_FULL + N_FUSED) {
#pragma unroll 1
      for (int j = 0; j < 2; j++) {  // six lanes per iteration, then the two halves swap places
        u64 t[6];
#pragma unroll
        for (int i = 0; i < 6; i++) t[i] = lazy::sbox(s[i]);
#pragma unroll
        for (int i = 0; i < 6; i++) {
          s[i] = s[i + 6];
          s[i + 6] = t[i];
        }
      }
      // round R adds the constants of round R + 1 through k = 96 + R; the last round has none (all zero)
      const int R = L < HALF_FULL ? L : L + N_FUSED;
      const int p = R < N_ROUNDS - 1 ? R : -1;
      x6 = make_uint4(onehot(p, 0), onehot(p, 1), onehot(p, 2), onehot(p, 3));
      x7 = make_uint4(onehot(p, 4), onehot(p, 5), onehot(p, 6), onehot(p, 7));
      bdesc = c.bdesc;
    } else {
      const int j = L - HALF_FULL, r = HALF_FULL + 2 * j;
      s[0] = lazy::sbox(s[0]);
      // u0 = row 0 of MDS s + RC[r + 1][0]: the constant's 16-bit pieces seed the dp2a accumulators (poseidon.cuh)
      u32 X[6][4];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        const u32 a0 = (u32)s[2 * k], a1 = (u32)(s[2 * k] >> 32), b0 = (u32)s[2 * k + 1], b1 = (u32)(s[2 * k + 1] >> 32);
        X[k][0] = __byte_perm(a0, b0, 0x5410);
        X[k][1] = __byte_perm(a0, b0, 0x7632);
        X[k][2] = __byte_perm(a1, b1, 0x5410);
        X[k][3] = __byte_perm(a1, b1, 0x7632);
      }
      const uint4 k0 = *reinterpret_cast<const uint4*>(RC2_DEV + (r + 1) * 24);
      u32 acc[4] = {k0.x, k0.y, k0.z, k0.w};
      lazy::dp_row<0, 0>(acc, X);
      const u64 t = lazy::sbox(recombine4(acc[0], acc[1], acc[2], acc[3]));
      const int p = 8 + j;  // k = 104 + j
      x6 = make_uint4((u32)t, (u32)(t >> 32), onehot(p, 2), onehot(p, 3));
      x7 = make_uint4(onehot(p, 4) | (~(u32)(s[0] >> 32) & 0xFF000000u), complement4(s, 1, 2, 3, 4),
                      complement4(s, 5, 6, 7, 8), complement4(s, 9, 10, 11, 11) & 0x00FFFFFFu);
      bdesc = c.bfdesc;
    }
    product(s, c, bdesc, x6, x7);
  }
#pragma unroll
  for (int i = 0; i < 12; i++) s[i] = s[i] >= gl::P ? s[i] - gl::P : s[i];
}

}  // namespace tc
}  // namespace poseidon
#endif
