// K14 `hash_to_g2`: the native HashToG2 witness (src/utils/hash_to_g2.rs:76-148, cofactor clearing :195-208) batched
// on the device, one message per work item. The contract is the Python restatement in workloads.py, word for word.
//   1. hash     one thread per message: the plonky2 Challenger over the message with the per-thread Poseidon
//               permutation, 32 challenges, two 512-bit integers of their low 32 bits, reduced mod p (hash_to_fq2)
//   2. map      one thread per u: Shallue-van de Woestijne with Z = 1, branch for branch as
//               workloads._map_with_tv4 (square roots a^((p+1)/4) in Fq, the complex method of inputs.fq2_sqrt in Fq2)
//   3. offsets  one thread per message draws k_i from SplitMix64; one warp per message adds the table points
//               2^j G2 of the set bits of k_i (chains::warp_bit_sum), then the batched affine conversion
//   4. clearing the singleton chains (cofactor, x_i) from offset_i through chains::run; hash_i = sum_i - offset_i
// Errors record the lowest failing message in one slot per kind (BAD_*).
#pragma once
#include "chains.cuh"
#include "poseidon.cuh"

namespace h2g2 {

using bn::F2;
using bn::Fq;
using bn::Fq2;
typedef bn::Jac<F2> Jac;
typedef bn::Aff<F2> Aff;

static constexpr size_t MAX_N = chains::MAX_TERMS;
static constexpr size_t MAX_MSG_ELEMS = (size_t)1 << 24;  // n * msg_len: 128 MB of messages
enum { BAD_CANONICAL, BAD_EXCEPTIONAL, BAD_K, BAD_HASH_INF, N_BAD };

// canonical words of the constants of workloads.py (Fq2: c0 then c1)
#define H2G2_G2_B {0x3267e6dc24a138e5ull, 0xb5b4c5e559dbefa3ull, 0x81be18991be06ac3ull, 0x2b149d40ceb8aaaeull, \
                   0xe4a2bd0685c315d2ull, 0xa74fa084e52d1852ull, 0xcd2cafadeed8fdf4ull, 0x009713b03af0fed4ull}
#define H2G2_NEG_HALF {0x9e10460b6c3e7ea3ull, 0xcbc0b548b438e546ull, 0xdc2822db40c0ac2eull, 0x183227397098d014ull, 0, 0, 0, 0}
#define H2G2_TV4 {0xfcbe57377b5ca1ecull, 0x2e6da55f90a3e510ull, 0xb801fa95b21af64eull, 0x29fd332ab7260112ull, \
                  0xb1e9154d01565034ull, 0x5e76f77b1267a846ull, 0xf8408aee24ba0b86ull, 0x303d1eff1426764bull}
#define H2G2_TV6 {0x21010b008d4eaf99ull, 0xb4e6a9c08b986767ull, 0x8632fe0eb2ac5a41ull, 0x17365bbe63b1d207ull, \
                  0x388732a995d03755ull, 0xfe164d7f4694786bull, 0xd689d7aa4209cad8ull, 0x0f57ffe5fc79e19cull}
#define H2G2_G2_GEN {0x46debd5cd992f6edull, 0x674322d4f75edaddull, 0x426a00665e5c4479ull, 0x1800deef121f1e76ull, \
                     0x97e485b7aef312c2ull, 0xf1aa493335a9e712ull, 0x7260bfb731fb5d25ull, 0x198e9393920d483aull, \
                     0x4ce6cc0166fa7daaull, 0xe3d1e7690c43d37bull, 0x4aab71808dcb408full, 0x12c85ea5db8c6debull, \
                     0x55acdadcd122975bull, 0xbc4b313370b38ef3ull, 0xec9e99ad690c3395ull, 0x090689d0585ff075ull}
#define H2G2_COFACTOR {0x345f2299c0f9fa8dull, 0x06ceecda572a2489ull, 0xb85045b68181585eull, 0x30644e72e131a029ull}
#define H2G2_R {0x43e1f593f0000001ull, 0x2833e84879b97091ull, 0xb85045b68181585dull, 0x30644e72e131a029ull}
// exponents (p - 1) / 2 (Legendre symbol) and (p + 1) / 4 (square root, p = 3 mod 4), 32-bit limbs
#define H2G2_LEGENDRE_EXP {0x6c3e7ea3u, 0x9e10460bu, 0xb438e546u, 0xcbc0b548u, 0x40c0ac2eu, 0xdc2822dbu, 0x7098d014u, 0x18322739u}
#define H2G2_SQRT_EXP {0xb61f3f52u, 0x4f082305u, 0x5a1c72a3u, 0x65e05aa4u, 0xa0605617u, 0x6e14116du, 0xb84c680au, 0x0c19139cu}

PB_HD Fq2 fq2_const(const u64 (&w)[8]) { return Fq2{bn::to_mont(bn::from_words(w)), bn::to_mont(bn::from_words(w + 4))}; }
PB_HD bool fq2_eq(const Fq2& a, const Fq2& b) { return bn::eq(a.c0, b.c0) && bn::eq(a.c1, b.c1); }
PB_HD Fq2 fq2_neg(const Fq2& a) { return Fq2{bn::neg(a.c0), bn::neg(a.c1)}; }
PB_HD Fq fq_norm(const Fq2& a) { return bn::add(bn::sqr(a.c0), bn::sqr(a.c1)); }
// g(x) = x^3 + b'
PB_HD Fq2 curve_g(const Fq2& x) {
  const u64 b[8] = H2G2_G2_B;
  return F2::add(F2::mul(F2::sqr(x), x), fq2_const(b));
}
// a is a square in Fq2 iff its norm is a square in Fq; 0 is not (workloads._fq2_is_qr)
PB_HD bool fq2_is_qr(const Fq2& a) {
  const u32 e[8] = H2G2_LEGENDRE_EXP;
  return bn::eq(bn::pow(fq_norm(a), e), bn::one());
}
// inputs.fq_sqrt: r = a^((p+1)/4), a root iff r^2 = a
PB_HD bool fq_sqrt(const Fq& a, Fq& r) {
  const u32 e[8] = H2G2_SQRT_EXP;
  r = bn::pow(a, e);
  return bn::eq(bn::sqr(r), a);
}
// inputs.fq2_sqrt, branch for branch. The a1 = 0 branch is there for parity only: no u of the map reaches it.
PB_HD bool fq2_sqrt(const Fq2& a, Fq2& r) {
  Fq t;
  if (bn::is_zero(a.c1)) {
    if (fq_sqrt(a.c0, t)) {
      r = Fq2{t, bn::zero()};
      return true;
    }
    if (!fq_sqrt(bn::neg(a.c0), t)) return false;
    r = Fq2{bn::zero(), t};
    return true;
  }
  Fq n;
  if (!fq_sqrt(fq_norm(a), n)) return false;
  const u64 nh[8] = H2G2_NEG_HALF;
  const Fq half = bn::neg(bn::to_mont(bn::from_words(nh)));
  for (int k = 0; k < 2; k++) {
    const Fq cand = bn::mul(k == 0 ? bn::add(a.c0, n) : bn::sub(a.c0, n), half);
    Fq x0;
    if (fq_sqrt(cand, x0) && !bn::is_zero(x0)) {
      const Fq2 x{x0, bn::mul(a.c1, bn::inv(bn::dbl(x0)))};
      if (fq2_eq(F2::sqr(x), a)) {
        r = x;
        return true;
      }
    }
  }
  return false;
}
// src/fields/sgn.rs:20-27 on canonical values
PB_HD bool fq2_sgn(const Fq2& a) {
  const Fq c0 = bn::from_mont(a.c0);
  return (c0.l[0] & 1) || (bn::is_zero(c0) && (bn::from_mont(a.c1).l[0] & 1));
}

// workloads._map_with_tv4(u, _TV4); false for an exceptional u (tv1 tv2 = 0, where Python raises)
PB_HD bool map_to_curve(const Fq2& u, Aff& out) {
  const u64 b[8] = H2G2_G2_B, nh[8] = H2G2_NEG_HALF, w4[8] = H2G2_TV4, w6[8] = H2G2_TV6;
  const Fq2 one = F2::one(), gz = F2::add(fq2_const(b), one), neg_half = fq2_const(nh);
  Fq2 tv1 = F2::mul(F2::sqr(u), gz);
  const Fq2 tv2 = F2::add(one, tv1);
  tv1 = F2::sub(one, tv1);
  const Fq2 d = F2::mul(tv1, tv2);
  if (F2::is_zero(d)) return false;
  const Fq2 tv3 = F2::inv(d);
  const Fq2 tv5 = F2::mul(F2::mul(F2::mul(u, tv1), tv3), fq2_const(w4));
  Fq2 x = F2::sub(neg_half, tv5);  // x1
  if (!fq2_is_qr(curve_g(x))) {
    x = F2::add(neg_half, tv5);  // x2
    if (!fq2_is_qr(curve_g(x))) {
      const Fq2 t = F2::mul(F2::sqr(tv2), tv3);
      x = F2::add(one, F2::mul(fq2_const(w6), F2::sqr(t)));  // x3
    }
  }
  Fq2 y;
  fq2_sqrt(curve_g(x), y);  // g(x) is a square for the chosen x; the chains check every point against the curve
  if (fq2_sgn(u) != fq2_sgn(y)) y = fq2_neg(y);
  out.x = x;
  out.y = y;
  return true;
}

// 1. hash_to_fq2 (workloads.hash_to_fq2): u[i] in Montgomery form
struct HashK {
  const u64* msgs;  // [n][len]
  size_t len;
  Fq2* u;
  unsigned* bad;
  PB_HD void operator()(size_t i) const {
    const u64* m = msgs + i * len;
    u64 s[12];
#pragma unroll
    for (int k = 0; k < 12; k++) s[k] = 0;
    bool canonical = true;
    for (size_t pos = 0; pos < len; pos += 8) {  // observed elements overwrite the rate lanes; 8 of them duplex
      const size_t take = len - pos < 8 ? len - pos : 8;
#pragma unroll
      for (int k = 0; k < 8; k++) {  // constant lane indices keep the state in registers
        if ((size_t)k >= take) continue;
        const u64 v = m[pos + k];
        canonical &= v < gl::P;
        s[k] = v < gl::P ? v : 0;  // the permutation needs canonical lanes
      }
      if (take == 8) poseidon::permute(s);
    }
    if (!canonical) tg::set_lowest(bad + BAD_CANONICAL, (unsigned)i);
    // a pending partial input or an empty output buffer (len = 0) forces a permutation; a full last input leaves
    // its 8 outputs. Challenges pop from the end of the rate lanes, 8 per permutation.
    if (len % 8 || len == 0) poseidon::permute(s);
    u32 limbs[32];  // challenge k (in pop order) is limb k % 16 of value k / 16
#pragma unroll
    for (int b = 0; b < 4; b++) {
      if (b) poseidon::permute(s);
#pragma unroll
      for (int t = 0; t < 8; t++) limbs[8 * b + t] = (u32)s[7 - t];
    }
    // v = lo + 2^256 hi: Montgomery form lo R + hi R^2 = to_mont(lo) + to_mont(to_mont(hi)). bn::mul(a, b) leaves
    // (a b + m p) / 2^256 < p + a b / 2^256 < 2p for any a < 2^256 and b < p, and its one conditional subtraction
    // makes that canonical, so lo, hi >= p need no reduction first.
    Fq2 out;
#pragma unroll
    for (int h = 0; h < 2; h++) {
      Fq lo, hi;
#pragma unroll
      for (int k = 0; k < 8; k++) {
        lo.l[k] = limbs[16 * h + k];
        hi.l[k] = limbs[16 * h + 8 + k];
      }
      (h ? out.c1 : out.c0) = bn::add(bn::to_mont(lo), bn::to_mont(bn::to_mont(hi)));
    }
    u[i] = out;
  }
};

// the map_to_g2 entry point's u: canonical words -> Montgomery form
struct LoadUK {
  const u64* w;  // [n][8]
  Fq2* u;
  unsigned* bad;
  PB_HD void operator()(size_t i) const {
    Fq2 v;
    if (!tg::FieldIO<F2>::load(w + i * 8, v)) {
      tg::set_lowest(bad + BAD_CANONICAL, (unsigned)i);
      v = F2::zero();
    }
    u[i] = v;
  }
};

// 2. the SvdW map
struct MapK {
  const Fq2* u;
  Aff* pts;
  unsigned* bad;
  PB_HD void operator()(size_t i) const {
    Aff p;
    if (!map_to_curve(u[i], p)) {
      tg::set_lowest(bad + BAD_EXCEPTIONAL, (unsigned)i);
      p.x = p.y = F2::one();
    }
    pts[i] = p;
  }
};

// canonical words of affine points: out + i * stride = x.c0, x.c1, y.c0, y.c1
struct PutK {
  const Aff* pts;
  u64* out;
  size_t stride;
  PB_HD void operator()(size_t i) const {
    chains::put_coord(out + i * stride, pts[i].x);
    chains::put_coord(out + i * stride + 8, pts[i].y);
  }
};
// the scalar of chain row i: the G2 cofactor (hash_to_g2.rs:68-74)
struct CofactorK {
  u64* terms;  // [n][20]
  PB_HD void operator()(size_t i) const {
    const u64 c[4] = H2G2_COFACTOR;
    for (int k = 0; k < 4; k++) terms[i * 20 + k] = c[k];
  }
};

// 3a. k_i = the bits256() of SplitMix64(seed) draws 4i+1 .. 4i+4, masked to 254 bits. The state after j draws is
// seed + j * gamma, so every message draws on its own. k_i = 0 mod r (k_i = 0 or r below 2^254) is an error.
PB_HD u64 splitmix64_draw(u64 seed, u64 j) {
  u64 z = seed + j * 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}
struct DrawK {
  u64 seed;
  u64* k;  // [n][4]
  unsigned* bad;
  PB_HD void operator()(size_t i) const {
    const u64 r[4] = H2G2_R;
    u64 w[4];
    bool zero = true, eq_r = true;
    for (int t = 0; t < 4; t++) {
      w[t] = splitmix64_draw(seed, 4 * (u64)i + 1 + t);
      if (t == 3) w[t] &= ((u64)1 << 62) - 1;
      zero &= w[t] == 0;
      eq_r &= w[t] == r[t];
      k[i * 4 + t] = w[t];
    }
    if (zero || eq_r) tg::set_lowest(bad + BAD_K, (unsigned)i);
  }
};

// the fixed-base table T_j = 2^j G2, j < 256, in Jacobian coordinates (one thread: the doubling chain)
static constexpr int TABLE_POINTS = 256;
struct TableK {
  Jac* T;
  PB_HD void operator()(size_t) const {
    const u64 g[16] = H2G2_G2_GEN;
    Jac p;
    tg::FieldIO<F2>::load(g, p.X);
    tg::FieldIO<F2>::load(g + 8, p.Y);
    p.Z = F2::one();
    for (int j = 0; j < TABLE_POINTS; j++) {
      T[j] = p;
      p = bn::jac_double<F2>(p);
    }
  }
};

#if PB_HOSTSIM
// 3b, one work item per thread
struct FixedBaseK {
  const Jac* T;
  const u64* k;
  Jac* out;
  PB_HD void operator()(size_t i) const {
    Jac acc = chains::infinity<F2>();
    for (int j = 0; j < TABLE_POINTS; j++)
      if (tg::scalar_bit(k + i * 4, j)) acc = bn::jac_add_complete<F2>(acc, T[j]);
    out[i] = acc;
  }
};
#else
// 3b. one warp per message: k_i G2 (k_i != 0 mod r, so never at infinity)
static constexpr int FB_WARPS = 4;
__global__ void __launch_bounds__(32 * FB_WARPS) k_fixed_base_sum(const Jac* __restrict__ T, const u64* __restrict__ k,
                                                                  size_t n, Jac* __restrict__ out) {
  __shared__ Jac part[FB_WARPS][32];
  const size_t i = (size_t)blockIdx.x * FB_WARPS + (threadIdx.x >> 5);
  if (i >= n) return;  // whole warps
  Jac* p = part[threadIdx.x >> 5];
  chains::warp_bit_sum<F2>(p, k + i * 4, T, 1);
  if ((threadIdx.x & 31) == 0) out[i] = p[0];
}
#endif

inline void fixed_base(const Jac* T, const u64* k, size_t n, Jac* out, pbStream s) {
#if PB_HOSTSIM
  pb_launch("h2g2 fixed base", FixedBaseK{T, k, out}, n, s);
#else
  if (!n) return;
  k_fixed_base_sum<<<(unsigned)((n + FB_WARPS - 1) / FB_WARPS), 32 * FB_WARPS, 0, s>>>(T, k, n, out);
  g_pb_launches++;
  pb_check_last("h2g2 fixed base");
#endif
}

// 5. hash_i = sum_i - offset_i (hash_to_g2.rs:204-208), before the affine pass; at infinity when cofactor x_i is
struct SubOffsetK {
  const u64* sums;     // [n][16] cofactor x_i + offset_i
  const u64* offsets;  // [n][16]
  Jac* out;
  unsigned* bad;
  PB_HD void operator()(size_t i) const {
    Jac a, b;
    tg::FieldIO<F2>::load(sums + i * 16, a.X);
    tg::FieldIO<F2>::load(sums + i * 16 + 8, a.Y);
    tg::FieldIO<F2>::load(offsets + i * 16, b.X);
    tg::FieldIO<F2>::load(offsets + i * 16 + 8, b.Y);
    b.Y = fq2_neg(b.Y);
    a.Z = b.Z = F2::one();
    Jac h = bn::jac_add_complete<F2>(a, b);
    if (F2::is_zero(h.Z)) {
      tg::set_lowest(bad + BAD_HASH_INF, (unsigned)i);
      h.Z = F2::one();  // keeps the affine pass defined; the call fails
    }
    out[i] = h;
  }
};

}  // namespace h2g2
