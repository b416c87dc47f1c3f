// Curve input handling shared by the trace generator (tracegen.cu) and the scalar-multiplication chains
// (chains.cuh): the device error word, canonical loads and curve checks of G1 / G2 points, and the batched
// Jacobian -> affine conversion.
#pragma once
#include "tracegen.h"
#include "bn254.cuh"

namespace tg {

PB_HD void set_err(int* err, int code) {
#ifdef __CUDA_ARCH__
  atomicMax(err, code);
#else
  int cur = __atomic_load_n(err, __ATOMIC_RELAXED);
  while (cur < code && !__atomic_compare_exchange_n(err, &cur, code, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
#endif
}
// *slot = min(*slot, v): the lowest failing index of a batch (slots start at 0xffffffff)
PB_HD void set_lowest(unsigned* slot, unsigned v) {
#ifdef __CUDA_ARCH__
  atomicMin(slot, v);
#else
  unsigned cur = __atomic_load_n(slot, __ATOMIC_RELAXED);
  while (v < cur && !__atomic_compare_exchange_n(slot, &cur, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {
  }
#endif
}

PB_HD bool words_lt_p(const u64* w4) {
  bn::Fq t = bn::from_words(w4);
  return !bn::geq_p(t.l);
}
PB_HD bool scalar_bit(const u64* s, int j) { return (s[j >> 6] >> (j & 63)) & 1; }

template <class F>
struct FieldIO;
template <>
struct FieldIO<bn::F1> {
  static constexpr int WORDS = 4, NDEN = 1;
  static PB_HD bool load(const u64* w, bn::Fq& out) {
    if (!words_lt_p(w)) return false;
    out = bn::to_mont(bn::from_words(w));
    return true;
  }
  // y^2 = x^3 + 3
  static PB_HD bool on_curve(const bn::Aff<bn::F1>& p) {
    return bn::eq(bn::sqr(p.y), bn::add(bn::mul(bn::sqr(p.x), p.x), bn::small(3)));
  }
};
template <>
struct FieldIO<bn::F2> {
  static constexpr int WORDS = 8, NDEN = 3;
  static PB_HD bool load(const u64* w, bn::Fq2& out) {
    if (!words_lt_p(w) || !words_lt_p(w + 4)) return false;
    out.c0 = bn::to_mont(bn::from_words(w));
    out.c1 = bn::to_mont(bn::from_words(w + 4));
    return true;
  }
  // y^2 = x^3 + 3 / (9 + u), checked as (9 + u) (y^2 - x^3) = 3
  static PB_HD bool on_curve(const bn::Aff<bn::F2>& p) {
    const bn::Fq2 d = bn::F2::sub(bn::F2::sqr(p.y), bn::F2::mul(bn::F2::sqr(p.x), p.x));
    const bn::Fq nine = bn::small(9);
    const bn::Fq c0 = bn::sub(bn::mul(nine, d.c0), d.c1), c1 = bn::add(d.c0, bn::mul(nine, d.c1));
    return bn::eq(c0, bn::small(3)) && bn::is_zero(c1);
  }
};

#if !PB_HOSTSIM
// dst[dst_off + i] = affine(src[i]); one thread per AFF_CH consecutive points sharing one Fermat inversion
// (Montgomery's trick): 3 multiplications per point for the inverse instead of ~380
static constexpr int AFF_CH = 16;
template <class F>
__global__ void __launch_bounds__(128) k_to_affine(const bn::Jac<F>* __restrict__ src, bn::Aff<F>* __restrict__ dst,
                                                   size_t count, size_t dst_off, int* err) {
  typedef typename F::T T;
  const size_t base = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) * AFF_CH;
  if (base >= count) return;
  const int cnt = (int)(count - base < (size_t)AFF_CH ? count - base : (size_t)AFF_CH);
  T pref[AFF_CH];
  T acc = F::one();
  for (int i = 0; i < cnt; i++) {
    T z = src[base + i].Z;
    if (F::is_zero(z)) {  // only after an error was flagged upstream
      set_err(err, ERR_INFINITY);
      z = F::one();
    }
    pref[i] = acc;
    acc = F::mul(acc, z);
  }
  T inv = F::inv(acc);
  for (int i = cnt - 1; i >= 0; i--) {
    const bn::Jac<F> p = src[base + i];
    const T z = F::is_zero(p.Z) ? F::one() : p.Z;
    const T zi = F::mul(inv, pref[i]);
    inv = F::mul(inv, z);
    const T zi2 = F::sqr(zi);
    bn::Aff<F> a;
    a.x = F::mul(p.X, zi2);
    a.y = F::mul(p.Y, F::mul(zi, zi2));
    dst[dst_off + base + i] = a;
  }
}
#endif

}  // namespace tg
