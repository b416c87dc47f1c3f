// BN254 base-field arithmetic for trace generation (K1): Fq in Montgomery form on 8 x 32-bit limbs
// (32x32+64 -> 64 multiply-adds map to IMAD.WIDE), Fq2 = Fq[u]/(u^2+1), and Jacobian point
// arithmetic generic over the coordinate field. Replaces the ark-bn254 / ark-ff calls of
// src/starks/curves/g1/add.rs:54-56,66,80, g2/add.rs:61-63,73,84 and fields/mul.rs:28-30.
// Only canonical affine coordinates ever reach the trace, so any correct arithmetic is bit-exact.
#pragma once
#include "compat.cuh"

namespace bn {

struct Fq {
  u32 l[8];
};

#define BN_P_LIMBS {0xd87cfd47u, 0x3c208c16u, 0x6871ca8du, 0x97816a91u, 0x8181585du, 0xb85045b6u, 0xe131a029u, 0x30644e72u}
#define BN_ONE_LIMBS {0xc58f0d9du, 0xd35d438du, 0xf5c70b3du, 0x0a78eb28u, 0x7879462cu, 0x666ea36fu, 0x9a07df2fu, 0x0e0a77c1u}
#define BN_R2_LIMBS {0x538afa89u, 0xf32cfc5bu, 0xd44501fbu, 0xb5e71911u, 0x0a417ff6u, 0x47ab1effu, 0xcab8351fu, 0x06d89f71u}
static constexpr u32 N0INV = 0xe4866389u;  // -p^-1 mod 2^32

PB_HD Fq zero() {
  Fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = 0;
  return r;
}
PB_HD Fq one() {  // R mod p
  const u32 c[8] = BN_ONE_LIMBS;
  Fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = c[i];
  return r;
}
PB_HD bool is_zero(const Fq& a) {
  u32 o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.l[i];
  return o == 0;
}
PB_HD bool eq(const Fq& a, const Fq& b) {
  u32 o = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) o |= a.l[i] ^ b.l[i];
  return o == 0;
}
// a >= p ?
PB_HD bool geq_p(const u32 a[8]) {
  const u32 P[8] = BN_P_LIMBS;
#pragma unroll
  for (int i = 7; i >= 0; i--) {
    if (a[i] > P[i]) return true;
    if (a[i] < P[i]) return false;
  }
  return true;
}
PB_HD void sub_p(u32 a[8]) {
  const u32 P[8] = BN_P_LIMBS;
  u64 borrow = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u64 d = (u64)a[i] - P[i] - borrow;
    a[i] = (u32)d;
    borrow = (d >> 32) & 1;
  }
}
PB_HD Fq add(const Fq& a, const Fq& b) {
  Fq r;
  u64 c = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    c += (u64)a.l[i] + b.l[i];
    r.l[i] = (u32)c;
    c >>= 32;
  }
  // p < 2^254 so a + b < 2^255: no carry out
  if (geq_p(r.l)) sub_p(r.l);
  return r;
}
PB_HD Fq sub(const Fq& a, const Fq& b) {
  const u32 P[8] = BN_P_LIMBS;
  Fq r;
  u64 borrow = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u64 d = (u64)a.l[i] - b.l[i] - borrow;
    r.l[i] = (u32)d;
    borrow = (d >> 32) & 1;
  }
  if (borrow) {
    u64 c = 0;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      c += (u64)r.l[i] + P[i];
      r.l[i] = (u32)c;
      c >>= 32;
    }
  }
  return r;
}
PB_HD Fq neg(const Fq& a) { return sub(zero(), a); }
PB_HD Fq dbl(const Fq& a) { return add(a, a); }

// Montgomery product a * b * 2^-256 mod p (CIOS, 32-bit limbs)
PB_HD Fq mul(const Fq& a, const Fq& b) {
  const u32 P[8] = BN_P_LIMBS;
  u32 t[10];
#pragma unroll
  for (int i = 0; i < 10; i++) t[i] = 0;
#pragma unroll
  for (int i = 0; i < 8; i++) {
    u64 c = 0;
#pragma unroll
    for (int j = 0; j < 8; j++) {
      c += (u64)a.l[j] * b.l[i] + t[j];
      t[j] = (u32)c;
      c >>= 32;
    }
    c += t[8];
    t[8] = (u32)c;
    t[9] = (u32)(c >> 32);
    u32 m = t[0] * N0INV;
    c = (u64)m * P[0] + t[0];
    c >>= 32;
#pragma unroll
    for (int j = 1; j < 8; j++) {
      c += (u64)m * P[j] + t[j];
      t[j - 1] = (u32)c;
      c >>= 32;
    }
    c += t[8];
    t[7] = (u32)c;
    t[8] = t[9] + (u32)(c >> 32);
  }
  Fq r;
#pragma unroll
  for (int i = 0; i < 8; i++) r.l[i] = t[i];
  if (t[8] || geq_p(r.l)) sub_p(r.l);
  return r;
}
PB_HD Fq sqr(const Fq& a) { return mul(a, a); }

PB_HD Fq to_mont(const Fq& raw) {
  const u32 c[8] = BN_R2_LIMBS;
  Fq r2;
#pragma unroll
  for (int i = 0; i < 8; i++) r2.l[i] = c[i];
  return mul(raw, r2);
}
PB_HD Fq from_mont(const Fq& m) {
  Fq o = zero();
  o.l[0] = 1;
  return mul(m, o);
}
PB_HD Fq small(u32 k) {  // k in Montgomery form
  Fq r = zero();
  r.l[0] = k;
  return to_mont(r);
}
// a^(p-2) by square-and-multiply (a != 0)
PB_HD Fq inv(const Fq& a) {
  const u32 P[8] = BN_P_LIMBS;
  Fq r = one();
#pragma unroll 1
  for (int i = 253; i >= 0; i--) {
    r = sqr(r);
    u32 w = P[i >> 5];
    if (i < 32) w = P[0] - 2;  // exponent p - 2 differs from p only in the lowest limb
    if ((w >> (i & 31)) & 1) r = mul(r, a);
  }
  return r;
}
// a^e for an exponent given as 8 little-endian 32-bit limbs, square-and-multiply from bit 255. The limb of each step
// is picked by unrolled selects, so that a constant exponent stays in registers (no local-memory indexing).
PB_HD Fq pow(const Fq& a, const u32 (&e)[8]) {
  Fq r = one();
#pragma unroll 1
  for (int i = 255; i >= 0; i--) {
    r = sqr(r);
    u32 w = e[0];
#pragma unroll
    for (int k = 1; k < 8; k++) w = (i >> 5) == k ? e[k] : w;
    if ((w >> (i & 31)) & 1) r = mul(r, a);
  }
  return r;
}
PB_HD Fq from_words(const u64 w[4]) {
  Fq r;
#pragma unroll
  for (int i = 0; i < 4; i++) {
    r.l[2 * i] = (u32)w[i];
    r.l[2 * i + 1] = (u32)(w[i] >> 32);
  }
  return r;
}
PB_HD void to_limbs16(const Fq& raw, int out[16]) {
#pragma unroll
  for (int i = 0; i < 8; i++) {
    out[2 * i] = (int)(raw.l[i] & 0xffff);
    out[2 * i + 1] = (int)(raw.l[i] >> 16);
  }
}

// ---- Fq2 ---------------------------------------------------------------------------------
struct Fq2 {
  Fq c0, c1;
};

// Field policies used by the generic curve code
struct F1 {
  typedef Fq T;
  static PB_HD T add(const T& a, const T& b) { return bn::add(a, b); }
  static PB_HD T sub(const T& a, const T& b) { return bn::sub(a, b); }
  static PB_HD T mul(const T& a, const T& b) { return bn::mul(a, b); }
  static PB_HD T sqr(const T& a) { return bn::sqr(a); }
  static PB_HD T dbl(const T& a) { return bn::dbl(a); }
  static PB_HD bool is_zero(const T& a) { return bn::is_zero(a); }
  static PB_HD T zero() { return bn::zero(); }
  static PB_HD T one() { return bn::one(); }
  static PB_HD T inv(const T& a) { return bn::inv(a); }
};
struct F2 {
  typedef Fq2 T;
  static PB_HD T add(const T& a, const T& b) { return T{bn::add(a.c0, b.c0), bn::add(a.c1, b.c1)}; }
  static PB_HD T sub(const T& a, const T& b) { return T{bn::sub(a.c0, b.c0), bn::sub(a.c1, b.c1)}; }
  static PB_HD T mul(const T& a, const T& b) {
    // Karatsuba: 3 base multiplications
    Fq v0 = bn::mul(a.c0, b.c0), v1 = bn::mul(a.c1, b.c1);
    Fq s = bn::mul(bn::add(a.c0, a.c1), bn::add(b.c0, b.c1));
    return T{bn::sub(v0, v1), bn::sub(bn::sub(s, v0), v1)};
  }
  static PB_HD T sqr(const T& a) {
    // (c0 + c1)(c0 - c1), 2 c0 c1
    Fq t = bn::mul(bn::add(a.c0, a.c1), bn::sub(a.c0, a.c1));
    Fq m = bn::mul(a.c0, a.c1);
    return T{t, bn::dbl(m)};
  }
  static PB_HD T dbl(const T& a) { return T{bn::dbl(a.c0), bn::dbl(a.c1)}; }
  static PB_HD bool is_zero(const T& a) { return bn::is_zero(a.c0) && bn::is_zero(a.c1); }
  static PB_HD T zero() { return T{bn::zero(), bn::zero()}; }
  static PB_HD T one() { return T{bn::one(), bn::zero()}; }
  static PB_HD T inv(const T& a) {
    Fq n = bn::add(bn::sqr(a.c0), bn::sqr(a.c1));
    Fq ni = bn::inv(n);
    return T{bn::mul(a.c0, ni), bn::mul(bn::neg(a.c1), ni)};
  }
};

// ---- Jacobian points (a = 0 curves): (X, Y, Z) ~ (X/Z^2, Y/Z^3) --------------------------------
template <class F>
struct Jac {
  typename F::T X, Y, Z;
};
template <class F>
struct Aff {
  typename F::T x, y;
};

// dbl-2009-l
template <class F>
PB_HD Jac<F> jac_double(const Jac<F>& p) {
  typedef typename F::T T;
  T A = F::sqr(p.X), B = F::sqr(p.Y), C = F::sqr(B);
  T t = F::add(p.X, B);
  T D = F::dbl(F::sub(F::sub(F::sqr(t), A), C));
  T E = F::add(F::dbl(A), A);
  T Fv = F::sqr(E);
  Jac<F> r;
  r.X = F::sub(Fv, F::dbl(D));
  T C8 = F::dbl(F::dbl(F::dbl(C)));
  r.Y = F::sub(F::mul(E, F::sub(D, r.X)), C8);
  r.Z = F::dbl(F::mul(p.Y, p.Z));
  return r;
}

// mixed addition p (Jacobian, Z != 0) + q (affine). status: 0 ok, 1 = p == q (result is the
// doubling), 2 = p == -q (point at infinity; result undefined)
template <class F>
PB_HD Jac<F> jac_add_mixed(const Jac<F>& p, const Aff<F>& q, int& status) {
  typedef typename F::T T;
  T Z1Z1 = F::sqr(p.Z);
  T U2 = F::mul(q.x, Z1Z1);
  T S2 = F::mul(q.y, F::mul(p.Z, Z1Z1));
  T H = F::sub(U2, p.X);
  T rr = F::sub(S2, p.Y);
  if (F::is_zero(H)) {
    if (F::is_zero(rr)) {
      status = 1;
      return jac_double<F>(p);
    }
    status = 2;
    return p;
  }
  status = 0;
  T HH = F::sqr(H), HHH = F::mul(H, HH), V = F::mul(p.X, HH);
  Jac<F> r;
  r.X = F::sub(F::sub(F::sqr(rr), HHH), F::dbl(V));
  r.Y = F::sub(F::mul(rr, F::sub(V, r.X)), F::mul(p.Y, HHH));
  r.Z = F::mul(p.Z, H);
  return r;
}


// complete addition of two Jacobian points; Z = 0 encodes the point at infinity
template <class F>
PB_HD Jac<F> jac_add_complete(const Jac<F>& p, const Jac<F>& q) {
  typedef typename F::T T;
  if (F::is_zero(p.Z)) return q;
  if (F::is_zero(q.Z)) return p;
  T Z1Z1 = F::sqr(p.Z), Z2Z2 = F::sqr(q.Z);
  T U1 = F::mul(p.X, Z2Z2), U2 = F::mul(q.X, Z1Z1);
  T S1 = F::mul(p.Y, F::mul(q.Z, Z2Z2)), S2 = F::mul(q.Y, F::mul(p.Z, Z1Z1));
  T H = F::sub(U2, U1), rr = F::sub(S2, S1);
  if (F::is_zero(H)) {
    if (F::is_zero(rr)) return jac_double<F>(p);  // a point of order two doubles to Z = 0
    Jac<F> inf;
    inf.X = F::one();
    inf.Y = F::one();
    inf.Z = F::zero();
    return inf;
  }
  T HH = F::sqr(H), HHH = F::mul(H, HH), V = F::mul(U1, HH);
  Jac<F> r;
  r.X = F::sub(F::sub(F::sqr(rr), HHH), F::dbl(V));
  r.Y = F::sub(F::mul(rr, F::sub(V, r.X)), F::mul(S1, HHH));
  r.Z = F::mul(F::mul(p.Z, q.Z), H);
  return r;
}

}  // namespace bn
