// Host verifier for the proofs this library serializes. Mirrors, step for step,
//   verify()                      src/starks/common/verifier.rs:32-98
//   g1_generate_ctl_values        src/starks/curves/g1/scalar_mul_ctl.rs:57-80 (G2 / Fq analogues)
//   sum_ctl_values                src/starks/common/ctl_values.rs:28-47
//   verify_stark_proof_with_challenges, verify_fri_proof   starky 0.4.0 / plonky2 0.2.2 (un-vendored)
// and evaluates the constraint system at zeta in the quadratic extension in the emission order of
//   eval_ext_circuit's native twin eval_packed_generic (SURVEY.md Appendix D).
// One walk (verify_walk) runs the checks in the reference's order. Its two heavy parts come from a Checks provider:
// the native CTL values (one scalar multiplication, or x^s, per instance: 0.2 - 2.3 s serially at the BASELINE sizes,
// profiles/r1_configs.md) and the Merkle openings of every query. HostChecks computes them here on the CPU
// (pb254_verify); verify_dev.cuh computes them on the context's GPU (pb254_verify_device). The per-instance native
// output and the Merkle path walk are PB_HD and shared by both, so both report the same error for every input.
// The transcript, the quotient identity at zeta and the FRI folds stay on the host.
#pragma once
#include "../../include/pb254.h"
#include "prover.cuh"
#include "chains.cuh"
#include <vector>

namespace verify {

using gl::E2;
typedef poseidon::Digest Digest;

struct VerifyError : Pb254Error {
  explicit VerifyError(const std::string& m) : Pb254Error(PB254_E_VERIFY, "verify: " + m) {}
};

// ---- extension-field helpers --------------------------------------------------------------------
static inline E2 X(u64 v) { return gl::e2(v, 0); }
static inline E2 operator+(E2 a, E2 b) { return gl::eadd(a, b); }
static inline E2 operator-(E2 a, E2 b) { return gl::esub(a, b); }
static inline E2 operator*(E2 a, E2 b) { return gl::emul(a, b); }
static inline bool operator==(E2 a, E2 b) { return a.a == b.a && a.b == b.b; }
static inline E2 dbl(E2 a) { return a + a; }

// Horner accumulation acc = acc * alpha + c per challenge (ConstraintConsumer)
struct Consumer {
  std::vector<u64> alphas;
  std::vector<E2> acc;
  E2 z_last, l_first, l_last;
  size_t count = 0;
  void constraint(E2 c) {
    for (size_t j = 0; j < alphas.size(); j++) acc[j] = gl::emul_base(acc[j], alphas[j]) + c;
    count++;
  }
  void transition(E2 c) { constraint(c * z_last); }
  void first_row(E2 c) { constraint(c * l_first); }
  void last_row(E2 c) { constraint(c * l_last); }
};

struct Rows {
  const E2 *local, *next, *aux, *aux_next;
};

static const u64 P16[16] = {64839, 55420, 35862, 15392, 51853, 26737, 27281, 38785,
                            22621, 33153, 17846, 47184, 41001, 57649, 20082, 12388};

// pol_mul_wide on extension elements
static inline void conv31(const E2* a, const E2* b, E2* out) {
  for (int k = 0; k < 31; k++) {
    E2 s = X(0);
    for (int i = (k > 15 ? k - 15 : 0); i <= (k < 15 ? k : 15); i++) s = s + a[i] * b[k - i];
    out[k] = s;
  }
}

// eval_modulus_zero (modular/modulus_zero.rs:163-198): 33 constraints under `filter`
static inline void eval_modulus_zero(Consumer& y, E2 filter, const E2* in31, const E2* aux80) {
  const E2 s = aux80[0];
  y.constraint(filter * (s * s - s));
  const E2 sign = dbl(s) - X(1);
  E2 q[17];
  for (int i = 0; i < 17; i++) q[i] = sign * aux80[1 + i];
  E2 ap_prev = X(0);
  for (int k = 0; k < 32; k++) {
    E2 c = X(0);
    for (int i = (k > 15 ? k - 15 : 0); i <= (k < 16 ? k : 16); i++) c = c + gl::emul_base(q[i], P16[k - i]);
    E2 ap = X(0);
    if (k < 31) ap = aux80[18 + k] - X((u64)1 << 29) + gl::emul_base(aux80[49 + k], (u64)1 << 16);
    c = c + ap_prev - gl::emul_base(ap, (u64)1 << 16);
    if (k < 31) c = c - in31[k];
    y.constraint(filter * c);
    ap_prev = ap;
  }
}

// eval_is_modulus_zero (modular/is_modulus_zero.rs:69-84): 49 constraints
static inline void eval_is_modulus_zero(Consumer& y, E2 filter, const E2* dx16, E2 is_zero, const E2* aux96) {
  E2 in[31];
  conv31(dx16, aux96, in);
  in[0] = in[0] + is_zero - X(1);
  eval_modulus_zero(y, filter, in, aux96 + 16);
  for (int i = 0; i < 16; i++) y.constraint(filter * is_zero * dx16[i]);
}

static inline void ext_conv(const E2* x0, const E2* x1, const E2* y0, const E2* y1, E2* c0, E2* c1) {
  E2 t[31];
  conv31(x0, y0, c0);
  conv31(x1, y1, t);
  for (int i = 0; i < 31; i++) c0[i] = c0[i] - t[i];
  conv31(x0, y1, c1);
  conv31(x1, y0, t);
  for (int i = 0; i < 31; i++) c1[i] = c1[i] + t[i];
}

static inline void eval_add_g1(Consumer& y, const tg::Layout& l, const E2* v, E2 filter) {
  const E2 *a = v + l.a, *b = v + l.b, *c = v + l.c, *A = v + l.aux;
  E2 dx[16], dy[16], in[31], in2[31];
  for (int i = 0; i < 16; i++) {
    dx[i] = b[i] - a[i];
    dy[i] = b[16 + i] - a[16 + i];
  }
  eval_is_modulus_zero(y, filter, dx, A[0], A + 1);
  const E2 is_x_eq = A[0], is_x_eq_filter = A[97];
  y.constraint(filter * is_x_eq - is_x_eq_filter);
  const E2* lam = A + 98;
  conv31(lam, dx, in);
  for (int i = 0; i < 16; i++) in[i] = in[i] - dy[i];
  eval_modulus_zero(y, filter - is_x_eq_filter, in, A + 114);
  conv31(a, a, in2);
  conv31(lam, a + 16, in);
  for (int i = 0; i < 31; i++) in[i] = dbl(in[i]) - (dbl(in2[i]) + in2[i]);
  eval_modulus_zero(y, is_x_eq_filter, in, A + 114);
  for (int i = 0; i < 16; i++) y.constraint(is_x_eq_filter * (a[16 + i] - b[16 + i]));
  conv31(lam, lam, in);
  for (int i = 0; i < 16; i++) in[i] = in[i] - (a[i] + b[i] + c[i]);
  eval_modulus_zero(y, filter, in, A + 194);
  E2 t0[16];
  for (int i = 0; i < 16; i++) t0[i] = c[i] - a[i];
  conv31(lam, t0, in);
  for (int i = 0; i < 16; i++) in[i] = in[i] + c[16 + i] + a[16 + i];
  eval_modulus_zero(y, filter, in, A + 274);
}

static inline void eval_add_g2(Consumer& y, const tg::Layout& l, const E2* v, E2 filter) {
  const E2 *a = v + l.a, *b = v + l.b, *c = v + l.c, *A = v + l.aux;  // x.c0 | x.c1 | y.c0 | y.c1
  const E2 is_x_eq = A[0], z0 = A[1], z1 = A[2];
  y.constraint(filter * (z0 * z1 - is_x_eq));
  E2 u0[16], u1[16], c0[31], c1[31], d0[31], d1[31];
  for (int i = 0; i < 16; i++) {
    u0[i] = b[i] - a[i];
    u1[i] = b[16 + i] - a[16 + i];
  }
  eval_is_modulus_zero(y, filter, u0, z0, A + 3);
  eval_is_modulus_zero(y, filter, u1, z1, A + 99);
  const E2 is_x_eq_filter = A[195];
  y.constraint(filter * is_x_eq - is_x_eq_filter);
  const E2 *l0 = A + 196, *l1 = A + 212;
  ext_conv(l0, l1, u0, u1, c0, c1);
  for (int i = 0; i < 16; i++) {
    c0[i] = c0[i] - (b[32 + i] - a[32 + i]);
    c1[i] = c1[i] - (b[48 + i] - a[48 + i]);
  }
  eval_modulus_zero(y, filter - is_x_eq_filter, c0, A + 228);
  eval_modulus_zero(y, filter - is_x_eq_filter, c1, A + 308);
  ext_conv(a, a + 16, a, a + 16, d0, d1);
  ext_conv(l0, l1, a + 32, a + 48, c0, c1);
  for (int i = 0; i < 31; i++) {
    c0[i] = dbl(c0[i]) - (dbl(d0[i]) + d0[i]);
    c1[i] = dbl(c1[i]) - (dbl(d1[i]) + d1[i]);
  }
  eval_modulus_zero(y, is_x_eq_filter, c0, A + 228);
  eval_modulus_zero(y, is_x_eq_filter, c1, A + 308);
  for (int i = 0; i < 32; i++) y.constraint(is_x_eq_filter * (a[32 + i] - b[32 + i]));
  ext_conv(l0, l1, l0, l1, c0, c1);
  for (int i = 0; i < 16; i++) {
    c0[i] = c0[i] - (a[i] + b[i] + c[i]);
    c1[i] = c1[i] - (a[16 + i] + b[16 + i] + c[16 + i]);
  }
  eval_modulus_zero(y, filter, c0, A + 388);
  eval_modulus_zero(y, filter, c1, A + 468);
  for (int i = 0; i < 16; i++) {
    u0[i] = c[i] - a[i];
    u1[i] = c[16 + i] - a[16 + i];
  }
  ext_conv(l0, l1, u0, u1, c0, c1);
  for (int i = 0; i < 16; i++) {
    c0[i] = c0[i] + c[32 + i] + a[32 + i];
    c1[i] = c1[i] + c[48 + i] + a[48 + i];
  }
  eval_modulus_zero(y, filter, c0, A + 548);
  eval_modulus_zero(y, filter, c1, A + 628);
}

static inline void eval_mul_fq(Consumer& y, const tg::Layout& l, const E2* v, E2 filter) {
  E2 in[31];
  conv31(v + l.a, v + l.b, in);
  for (int i = 0; i < 16; i++) in[i] = in[i] - v[l.c + i];
  eval_modulus_zero(y, filter, in, v + l.aux);
}

// all constraints of one (local, next) pair, in the reference's emission order
static inline void eval_all(Consumer& y, int kind, const Rows& R, const aux::Challenges& ch) {
  const tg::Layout l = tg::layout_for(kind);
  const E2 *lv = R.local, *nv = R.next;
  const int L = l.L;
  const E2 one = X(1);
  const E2 filter = lv[l.filter], is_first = lv[l.rf], is_last = lv[l.rf + 1];
  if (kind == 0)
    eval_add_g1(y, l, lv, filter);
  else if (kind == 1)
    eval_add_g2(y, l, lv, filter);
  else
    eval_mul_fq(y, l, lv, filter);
  y.constraint(is_first * (lv[l.flag_op] - one));
  for (int i = 0; i < L; i++) y.constraint(is_first * (lv[l.reg0 + i] - lv[l.b + i]));
  const E2 bit0 = lv[l.bits];
  for (int i = 0; i < L; i++) y.constraint(bit0 * is_first * (lv[l.reg1 + i] - lv[l.c + i]));
  for (int i = 0; i < L; i++) y.constraint((one - bit0) * is_first * (lv[l.reg1 + i] - lv[l.a + i]));
  if (kind == 2)
    for (int k = 0; k < 16; k++) y.constraint(is_first * (lv[l.a + k] - X(k == 0 ? 1 : 0)));
  const E2 fs = lv[l.flag_sq_nl], nbit0 = nv[l.bits];
  for (int i = 0; i < L; i++) y.constraint(fs * (nv[l.a + i] - lv[l.reg1 + i]));
  for (int i = 0; i < L; i++) y.constraint(fs * (nv[l.b + i] - lv[l.reg0 + i]));
  for (int i = 0; i < L; i++) y.constraint(nbit0 * fs * (nv[l.reg1 + i] - nv[l.c + i]));
  for (int i = 0; i < L; i++) y.constraint((one - nbit0) * fs * (nv[l.reg1 + i] - nv[l.a + i]));
  for (int i = 0; i < L; i++) y.constraint(fs * (nv[l.reg0 + i] - lv[l.reg0 + i]));
  y.constraint(fs * (nv[l.flag_op] - one));
  y.constraint(fs * nv[l.flag_sq_nl]);
  for (int k = 0; k < 256; k++) y.constraint(fs * (nv[l.bits + k] - lv[l.bits + ((k + 1) & 255)]));
  const E2 g = lv[l.flag_op];
  const E2 is_next_not_last = nv[l.filter] - nv[l.rf + 1];
  for (int i = 0; i < L; i++) y.constraint(g * (nv[l.a + i] - lv[l.reg0 + i]));
  for (int i = 0; i < L; i++) y.constraint(g * (nv[l.b + i] - lv[l.reg0 + i]));
  for (int i = 0; i < L; i++) y.constraint(g * (nv[l.reg1 + i] - lv[l.reg1 + i]));
  for (int i = 0; i < L; i++) y.constraint(g * (nv[l.reg0 + i] - nv[l.c + i]));
  y.constraint(g * nv[l.flag_op]);
  y.constraint(g * (nv[l.flag_sq_nl] - is_next_not_last));
  for (int k = 0; k < 256; k++) y.constraint(g * (nv[l.bits + k] - lv[l.bits + k]));
  {  // eval_round_flags (common/round_flags.rs:46-81)
    const E2 counter = lv[l.rf + 2], inv_c = lv[l.rf + 3], inv_cp = lv[l.rf + 4], next_counter = nv[l.rf + 2];
    const E2 not_filter = one - filter;
    y.constraint(not_filter * is_first);
    y.constraint(not_filter * is_last);
    y.constraint(filter * (counter * inv_c - (one - is_first)));
    y.constraint(filter * counter * is_first);
    const E2 cprime = counter - X((u64)(tg::PERIOD - 1));
    y.constraint(filter * (cprime * inv_cp - (one - is_last)));
    y.constraint(filter * cprime * is_last);
    y.constraint(filter * (one - is_last) * (next_counter - counter - one));
    y.constraint(filter * is_last * next_counter);
  }
  y.constraint((filter - is_last) * (nv[l.ts] - lv[l.ts]));
  y.constraint((filter - is_last) * (nv[l.filter] - filter));
  {
    const E2 rc = lv[l.range_counter], d = nv[l.range_counter] - rc;
    y.transition(d * d - d);
    y.last_row(rc - X(65535));
  }
  // logUp lookups (starky lookup.rs eval_packed_lookups_generic)
  const int ncols = l.rc_hi - l.rc_lo, nh = (ncols + 1) / 2;
  for (int j = 0; j < ch.nch; j++) {
    const E2 beta = X(ch.beta[j]);
    const E2 *h = R.aux + j * (nh + 1), *hn = R.aux_next + j * (nh + 1);
    E2 hs = X(0);
    for (int k = 0; k < nh; k++) {
      hs = hs + h[k];
      const E2 c0 = lv[l.rc_lo + 2 * k] + beta;
      if (2 * k + 1 < ncols) {
        const E2 c1 = lv[l.rc_lo + 2 * k + 1] + beta;
        y.constraint(c1 * c0 * h[k] - c1 - c0);
      } else {
        y.constraint(c0 * h[k] - one);
      }
    }
    const E2 z = h[nh], nz = hn[nh];
    y.first_row(z);
    const E2 table = lv[l.range_counter] + beta;
    const E2 yv = hs * table - lv[l.freq];
    y.constraint((nz - z) * table - yv);
  }
  // cross-table lookups (starky cross_table_lookup.rs eval_cross_table_lookup_checks)
  const E2 *zc = R.aux + (nh + 1) * ch.nch, *zcn = R.aux_next + (nh + 1) * ch.nch;
  for (int c = 0; c < 2; c++) {
    const E2 f = c == 0 ? is_first : is_last;
    for (int j = 0; j < ch.nch; j++) {
      const u64 beta = ch.beta[j];
      E2 comb = lv[l.ts];
      if (c == 0) {
        for (int k = 15; k >= 0; k--) {
          E2 limb = X(0);
          for (int b = 15; b >= 0; b--) limb = dbl(limb) + lv[l.bits + 16 * k + b];
          comb = gl::emul_base(comb, beta) + limb;
        }
        if (kind != 2)
          for (int k = L - 1; k >= 0; k--) comb = gl::emul_base(comb, beta) + lv[l.a + k];
        for (int k = L - 1; k >= 0; k--) comb = gl::emul_base(comb, beta) + lv[l.b + k];
      } else {
        for (int k = L - 1; k >= 0; k--) comb = gl::emul_base(comb, beta) + lv[l.reg1 + k];
      }
      comb = comb + X(ch.gamma[j]);
      const E2 lz = zc[c * ch.nch + j], nz = zcn[c * ch.nch + j];
      y.last_row(comb * lz - f);
      y.transition(comb * (lz - nz) - f);
    }
  }
}

// ---- native CTL tuples (g1_generate_ctl_values and analogues) --------------------------------------
// Per-instance outcome of the native computation (host and device): NATIVE_OK or the first failed check.
enum { NATIVE_OK, NATIVE_NOT_CANONICAL, NATIVE_ORDER_TWO, NATIVE_INTERMEDIATE_INF, NATIVE_RESULT_INF };
static inline Pb254Error native_error(int status) {
  switch (status) {
    case NATIVE_NOT_CANONICAL: return Pb254Error(PB254_E_NOT_CANONICAL, "input coordinate >= p");
    case NATIVE_ORDER_TWO: return Pb254Error(PB254_E_INFINITY, "native result: point of order two");
    case NATIVE_INTERMEDIATE_INF: return Pb254Error(PB254_E_INFINITY, "native result: intermediate point at infinity");
    default: return Pb254Error(PB254_E_INFINITY, "native result: s * x + offset is the point at infinity");
  }
}

// r = s * x + off by double-and-add from the top bit of s, as g1_generate_ctl_values computes it; x need not lie in
// the prime-order subgroup (hash_to_g2 rows). Returns NATIVE_OK or the NATIVE_* infinity that stopped the ladder.
template <class F>
PB_HD int native_scalar_mul(const u64* s, const bn::Aff<F>& x, const bn::Aff<F>& off, bn::Aff<F>& r) {
  bn::Jac<F> acc;
  bool started = false;
  int st = 0;
#pragma unroll 1
  for (int j = 255; j >= 0; j--) {
    if (started) {
      if (F::is_zero(acc.Y)) return NATIVE_ORDER_TWO;
      acc = bn::jac_double<F>(acc);
    }
    if ((s[j >> 6] >> (j & 63)) & 1) {
      if (!started) {
        acc.X = x.x;
        acc.Y = x.y;
        acc.Z = F::one();
        started = true;
      } else {
        acc = bn::jac_add_mixed<F>(acc, x, st);
        if (st == 2) return NATIVE_INTERMEDIATE_INF;
      }
    }
  }
  if (!started) {
    r = off;
    return NATIVE_OK;
  }
  acc = bn::jac_add_mixed<F>(acc, off, st);
  if (st == 2) return NATIVE_RESULT_INF;
  typename F::T zi = F::inv(acc.Z), zi2 = F::sqr(zi);
  r.x = F::mul(acc.X, zi2);
  r.y = F::mul(acc.Y, F::mul(zi, zi2));
  return NATIVE_OK;
}

// x^s, square-and-multiply from bit 255 (fq_exp)
PB_HD bn::Fq native_fq_exp(const u64* s, const bn::Fq& x) {
  bn::Fq acc = bn::one();
#pragma unroll 1
  for (int j = 255; j >= 0; j--) {
    acc = bn::sqr(acc);
    if ((s[j >> 6] >> (j & 63)) & 1) acc = bn::mul(acc, x);
  }
  return acc;
}

PB_HD bool words_canonical(const u64* w) {
  const u64 PW[4] = {0x3c208c16d87cfd47ULL, 0x97816a916871ca8dULL, 0xb85045b68181585dULL, 0x30644e72e131a029ULL};
#pragma unroll
  for (int i = 3; i >= 0; i--) {
    if (w[i] < PW[i]) return true;
    if (w[i] > PW[i]) return false;
  }
  return false;
}
static inline void push_limbs(std::vector<u64>& out, const u64* w) {
  for (int i = 0; i < 16; i++) out.push_back((w[i >> 2] >> (16 * (i & 3))) & 0xffff);
}
// the Montgomery form of the canonical words at w; false if they are >= p
PB_HD bool load_fq(const u64* w, bn::Fq& out) {
  if (!words_canonical(w)) return false;
  out = bn::to_mont(bn::from_words(w));
  return true;
}

// Canonical words of the native output of the input row w: x^s (4 words), s * x + offset in G1 (x, y: 8) or G2
// (x.c0, x.c1, y.c0, y.c1: 16). Returns NATIVE_OK or the first failed check, in the order of the reference walk.
template <int KIND>
PB_HD int native_output(const u64* w, u64* out) {
  if (KIND == 2) {
    bn::Fq x;
    if (!load_fq(w + 4, x)) return NATIVE_NOT_CANONICAL;
    chains::put_fq(out, native_fq_exp(w, x));
    return NATIVE_OK;
  } else if (KIND == 0) {
    bn::Aff<bn::F1> x, off, r;
    if (!(load_fq(w + 4, x.x) & load_fq(w + 8, x.y) & load_fq(w + 12, off.x) & load_fq(w + 16, off.y)))
      return NATIVE_NOT_CANONICAL;
    const int st = native_scalar_mul<bn::F1>(w, x, off, r);
    if (st) return st;
    chains::put_fq(out, r.x);
    chains::put_fq(out + 4, r.y);
    return NATIVE_OK;
  } else {
    bn::Aff<bn::F2> x, off, r;
    if (!(load_fq(w + 4, x.x.c0) & load_fq(w + 8, x.x.c1) & load_fq(w + 12, x.y.c0) & load_fq(w + 16, x.y.c1) &
          load_fq(w + 20, off.x.c0) & load_fq(w + 24, off.x.c1) & load_fq(w + 28, off.y.c0) & load_fq(w + 32, off.y.c1)))
      return NATIVE_NOT_CANONICAL;
    const int st = native_scalar_mul<bn::F2>(w, x, off, r);
    if (st) return st;
    chains::put_fq(out, r.x.c0);
    chains::put_fq(out + 4, r.x.c1);
    chains::put_fq(out + 8, r.y.c0);
    chains::put_fq(out + 12, r.y.c1);
    return NATIVE_OK;
  }
}
static inline int native_output(int kind, const u64* w, u64* out) {
  return kind == 0 ? native_output<0>(w, out) : kind == 1 ? native_output<1>(w, out) : native_output<2>(w, out);
}

// tuples[0][k] = looked values of CTL 0 (inputs) for instance k, tuples[1][k] = CTL 1 (outputs)
static inline void ctl_tuples(int kind, const u64* inputs, const u64* ts, size_t K, std::vector<std::vector<u64>> tuples[2]) {
  const tg::Layout l = tg::layout_for(kind);
  const int out_words = kind == 0 ? 8 : kind == 1 ? 16 : 4;
  tuples[0].assign(K, {});
  tuples[1].assign(K, {});
  // the lowest failing instance's error is reported, also when the hostsim build runs this loop with OpenMP
  size_t err_k = K;
  int err_status = NATIVE_OK;
#pragma omp parallel for schedule(dynamic, 4)
  for (long long kk = 0; kk < (long long)K; kk++) {
    const size_t k = (size_t)kk;
    const u64* w = inputs + k * l.in_words;
    std::vector<u64>&in = tuples[0][k], &out = tuples[1][k];
    u64 r[16];
    const int st = native_output(kind, w, r);
    if (st) {
#pragma omp critical
      if (k < err_k) {
        err_k = k;
        err_status = st;
      }
      continue;
    }
    for (int c = 4; c < l.in_words; c += 4) push_limbs(in, w + c);  // x (and the offset)
    push_limbs(in, w);                                                // s as 16 limbs
    for (int c = 0; c < out_words; c += 4) push_limbs(out, r + c);
    in.push_back(ts[k] % gl::P);
    out.push_back(ts[k] % gl::P);
  }
  if (err_status) throw native_error(err_status);
}

// ---- Merkle ------------------------------------------------------------------------------------------
// hash_or_noop of the leaf v[0..n), then the path of `depth` siblings up to the cap entry; true if they agree. Every
// word must be canonical (the walk has checked the whole blob): the device permutation requires canonical inputs.
PB_HD void hash_or_noop(const u64* v, size_t n, u64 d[4]) {
  if (n <= 4) {
#pragma unroll
    for (int i = 0; i < 4; i++) d[i] = (size_t)i < n ? v[i] : 0;
    return;
  }
  u64 s[12];
#pragma unroll
  for (int i = 0; i < 12; i++) s[i] = 0;
#pragma unroll 1
  for (size_t c = 0; c < n; c += 8) {
#pragma unroll
    for (int k = 0; k < 8; k++)
      if (c + k < n) s[k] = v[c + k];
    poseidon::permute(s);
  }
#pragma unroll
  for (int i = 0; i < 4; i++) d[i] = s[i];
}
PB_HD bool merkle_path_ok(const u64* leaf, size_t leaf_len, size_t index, const u64* siblings, int depth,
                          const u64* cap) {
  Digest cur;
  hash_or_noop(leaf, leaf_len, cur.e);
#pragma unroll 1
  for (int lv = 0; lv < depth; lv++) {
    Digest sib;
#pragma unroll
    for (int i = 0; i < 4; i++) sib.e[i] = siblings[4 * lv + i];
    const bool right = index & 1;
    cur = poseidon::two_to_one(right ? sib : cur, right ? cur : sib);
    index >>= 1;
  }
  bool same = true;
#pragma unroll
  for (int i = 0; i < 4; i++) same &= cur.e[i] == cap[4 * index + i];
  return same;
}

// ---- the two heavy parts of verification -----------------------------------------------------------
// What verify_walk knows once the transcript has run: the caller's batch, the proof and its layout, the CTL
// challenges and the query indices.
struct Job {
  int kind, nch, logN, cap_h;
  const u64* blob;
  size_t words;
  const pb254_proof_layout* lay;
  const u64 *inputs, *timestamps;
  size_t K;
  const aux::Challenges* chal;
  const std::vector<u64>* idx;
  const std::vector<unsigned>* arities;
};
struct CtlResults {
  int code = 0;               // the lowest failing instance's native error (0: none) ...
  std::string msg;            // ... and its message
  std::vector<uint8_t> zero;  // [c * nch + j]: some combination of CTL c under challenge j is zero
  std::vector<u64> sum;       // [c * nch + j]: the sum of the inverses of those combinations
};
// Tree t of a query: 0 trace, 1 auxiliary, 2 quotient, 3 + i FRI layer i.
struct Checks {
  virtual ~Checks() {}
  virtual void start(const Job& job) = 0;  // called once, before the quotient identity is evaluated
  virtual void ctl(CtlResults& out) = 0;
  virtual bool merkle_ok(size_t q, int tree, const u64* leaf, size_t leaf_len, size_t index, const u64* siblings,
                         int depth, const u64* cap) = 0;
};

// pb254_verify: both parts computed here on the CPU, the Merkle paths when the walk asks for them
struct HostChecks : Checks {
  Job job;
  void start(const Job& j) override { job = j; }
  void ctl(CtlResults& o) override {
    const int nch = job.nch;
    std::vector<std::vector<u64>> tuples[2];
    try {
      ctl_tuples(job.kind, job.inputs, job.timestamps, job.K, tuples);
    } catch (const Pb254Error& e) {
      o.code = e.code;
      o.msg = e.what();
      return;
    }
    o.zero.assign(2 * nch, 0);
    o.sum.assign(2 * nch, 0);
    for (int c = 0; c < 2; c++)
      for (int j = 0; j < nch; j++) {
        u64 sum = 0;
        for (size_t k = 0; k < job.K; k++) {
          const std::vector<u64>& t = tuples[c][k];
          u64 comb = 0;
          for (size_t i = t.size(); i-- > 0;) comb = gl::add(gl::mul(comb, job.chal->beta[j]), t[i]);
          comb = gl::add(comb, job.chal->gamma[j]);
          if (comb == 0) {
            o.zero[c * nch + j] = 1;
            break;
          }
          sum = gl::add(sum, gl::inv(comb));
        }
        o.sum[c * nch + j] = sum;
      }
  }
  bool merkle_ok(size_t, int, const u64* leaf, size_t leaf_len, size_t index, const u64* siblings, int depth,
                 const u64* cap) override {
    return merkle_path_ok(leaf, leaf_len, index, siblings, depth, cap);
  }
};

// ---- the verifier -------------------------------------------------------------------------------------
// `kind` and `cfg` are the CALLER's (the reference's verify(stark, config, ...) takes the StarkConfig from the caller,
// src/starks/common/verifier.rs:32-45): every security parameter stamped into the blob header must equal them, only
// degree_bits is read from the proof. `inputs` holds K rows of in_words(kind) words.
static inline void verify_walk(int kind, const pb254_config& cfg, const u64* blob, size_t words, const u64* inputs,
                               const u64* timestamps, size_t K, Checks& checks) {
  if (kind < 0 || kind > 2) throw Pb254Error(PB254_E_BAD_ARG, "unknown STARK kind");
  prover::validate_config(cfg);
  if (words < 22 || blob[0] != prover::PROOF_MAGIC) throw VerifyError("not a pb254 proof blob");
  if (blob[1] != (u64)kind) throw VerifyError("proof header: STARK kind differs from the caller's");
  const u64 want[7] = {cfg.rate_bits, cfg.cap_height, cfg.num_challenges, cfg.num_query_rounds,
                       cfg.pow_bits,  cfg.arity_bits, cfg.final_poly_bits};
  for (int i = 0; i < 7; i++)
    if (blob[3 + i] != want[i]) throw VerifyError("proof header: StarkConfig differs from the caller's");
  if (blob[2] < 16 || blob[2] > 26) throw VerifyError("proof header: degree_bits");
  const int L = (int)blob[2];
  if (K > (((size_t)1 << L) >> 9)) throw VerifyError("more public instances than the trace has periods");
  const tg::Layout l = tg::layout_for(kind);
  const int nch = (int)cfg.num_challenges, W = l.width, NH = aux::num_helpers(l), A = aux::num_aux(l, nch), Q = 2 * nch,
            nlk = (NH + 1) * nch, r = (int)cfg.rate_bits, logN = L + r, cap_h = (int)cfg.cap_height;
  const size_t n = (size_t)1 << L, N = n << r, ncap = (size_t)1 << cap_h, capw = ncap * 4;
  if (cap_h > logN) throw VerifyError("cap height");
  const std::vector<unsigned> arities = prover::fri_arities(cfg, (unsigned)L);
  // ---- layout (proofview.cuh) -----------------------------------------------------------------------
  pb254_proof_layout lay;
  try {
    proofview::parse(blob, words, lay);
  } catch (const Pb254Error& e) {
    throw VerifyError(std::string(e.what()));
  }
  const u64* state = blob + lay.init_challenger_state;
  const u64* caps = blob + lay.trace_cap;  // trace, auxiliary, quotient caps are consecutive
  const u64* op_tr = blob + lay.local_values;     // local | next
  const u64* op_ax = blob + lay.auxiliary_polys;  // aux | aux_next
  const u64* zs_first = blob + lay.ctl_zs_first;
  const u64* op_q = blob + lay.quotient_polys;
  const u64* fri_caps = blob + lay.commit_phase_merkle_caps;
  const size_t nq = cfg.num_query_rounds;
  const int nsib = (int)lay.initial_path_words;
  const size_t rec = lay.query_words;
  const u64* queries = blob + lay.query_round_proofs;
  const size_t keep = lay.final_poly_words / 2;  // coefficients of the final polynomial (len >> rate_bits)
  int log_final = 0;
  while (((size_t)1 << log_final) < keep) log_final++;
  const u64* final_poly = blob + lay.final_poly;
  const u64 pow_witness = blob[lay.pow_witness];
  for (size_t i = 22; i < words; i++)
    if (blob[i] >= gl::P) throw VerifyError("non-canonical field element");

  // ---- transcript (verifier.rs:47-78, get_challenges) ---------------------------------------------
  prover::Challenger ch;
  ch.observe_n(caps, capw);
  aux::Challenges chal;
  chal.nch = nch;
  for (int j = 0; j < nch; j++) {
    chal.beta[j] = ch.challenge();
    chal.gamma[j] = ch.challenge();
  }
  u64 st[12];
  ch.compact(st);
  if (memcmp(st, state, sizeof st) != 0) throw VerifyError("init_challenger_state");
  ch.observe_n(caps + capw, capw);
  Consumer y;
  for (int j = 0; j < nch; j++) y.alphas.push_back(ch.challenge());
  ch.observe_n(caps + 2 * capw, capw);
  const E2 zeta = ch.ext_challenge();
  ch.observe_n(op_tr, 2 * (size_t)W);
  ch.observe_n(op_ax, 2 * (size_t)A);
  ch.observe_n(op_q, 2 * (size_t)Q);
  ch.observe_n(op_tr + 2 * W, 2 * (size_t)W);
  ch.observe_n(op_ax + 2 * A, 2 * (size_t)A);
  for (int k = 0; k < 2 * nch; k++) {
    ch.observe(zs_first[k]);
    ch.observe(0);
  }
  const E2 fri_alpha = ch.ext_challenge();
  std::vector<E2> fri_betas;
  for (size_t i = 0; i < arities.size(); i++) {
    ch.observe_n(fri_caps + i * capw, capw);
    fri_betas.push_back(ch.ext_challenge());
  }
  ch.observe_n(final_poly, 2 * keep);
  ch.observe(pow_witness);
  const u64 pow_resp = ch.challenge();
  if (cfg.pow_bits && (pow_resp >> (64 - cfg.pow_bits)) != 0) throw VerifyError("proof of work");
  std::vector<u64> idx(nq);
  for (auto& x : idx) x = ch.challenge() % (u64)N;
  {
    const Job job{kind, nch, logN, cap_h, blob, words, &lay, inputs, timestamps, K, &chal, &idx, &arities};
    checks.start(job);
  }

  // ---- quotient identity at zeta -------------------------------------------------------------------
  const u64 g = gl::root_of_unity(L);
  E2 zeta_pow_n = zeta;
  for (int i = 0; i < L; i++) zeta_pow_n = zeta_pow_n * zeta_pow_n;
  const E2 z_h = zeta_pow_n - X(1);
  if (z_h == X(0)) throw VerifyError("zeta in the trace subgroup");
  const u64 n_inv = gl::inv((u64)n % gl::P);
  y.z_last = zeta - X(gl::inv(g));
  y.l_first = gl::emul_base(z_h, n_inv) * gl::einv(zeta - X(1));
  y.l_last = gl::emul_base(z_h, n_inv) * gl::einv(gl::emul_base(zeta, g) - X(1));
  y.acc.assign(nch, X(0));
  auto exts = [](const u64* p, size_t cnt) {
    std::vector<E2> v(cnt);
    for (size_t i = 0; i < cnt; i++) v[i] = gl::e2(p[2 * i], p[2 * i + 1]);
    return v;
  };
  const std::vector<E2> lv = exts(op_tr, W), nv = exts(op_tr + 2 * W, W), av = exts(op_ax, A), anv = exts(op_ax + 2 * A, A),
                        qv = exts(op_q, Q);
  Rows R{lv.data(), nv.data(), av.data(), anv.data()};
  eval_all(y, kind, R, chal);
  if ((int)y.count != quot::num_constraints(kind, nch)) throw VerifyError("internal: constraint count");
  for (int j = 0; j < nch; j++) {
    const E2 rhs = z_h * (qv[2 * j] + zeta_pow_n * qv[2 * j + 1]);
    if (!(y.acc[j] == rhs)) throw VerifyError("quotient identity at zeta");
  }

  // ---- cross-table lookup sums (verifier.rs:88-95, ctl_values.rs:28-47) ----------------------------
  {
    CtlResults ctl;
    checks.ctl(ctl);
    if (ctl.code) throw Pb254Error(ctl.code, ctl.msg);
    for (int c = 0; c < 2; c++)
      for (int j = 0; j < nch; j++) {
        if (ctl.zero[c * nch + j]) throw VerifyError("CTL combination is zero");
        if (ctl.sum[c * nch + j] != zs_first[c * nch + j]) throw VerifyError("cross-table lookup sum");
      }
  }

  // ---- FRI (verify_fri_proof) ------------------------------------------------------------------------
  const int NP = W + A + Q;
  std::vector<E2> apow(NP + 1);
  apow[0] = X(1);
  for (int i = 1; i <= NP; i++) apow[i] = apow[i - 1] * fri_alpha;
  E2 O0 = X(0), O1 = X(0), O2 = X(0);
  for (int i = 0; i < W; i++) {
    O0 = O0 + apow[i] * lv[i];
    O1 = O1 + apow[i] * nv[i];
  }
  for (int i = 0; i < A; i++) {
    O0 = O0 + apow[W + i] * av[i];
    O1 = O1 + apow[W + i] * anv[i];
  }
  for (int i = 0; i < Q; i++) O0 = O0 + apow[W + A + i] * qv[i];
  for (int k = 0; k < 2 * nch; k++) O2 = O2 + gl::emul_base(apow[k], zs_first[k]);
  const E2 zeta_next = gl::emul_base(zeta, g);
  const u64 wN = gl::root_of_unity(logN);
  for (size_t q = 0; q < nq; q++) {
    const u64* rp = queries + q * rec;
    size_t x_index = (size_t)idx[q];
    const u64 *row_tr = rp, *sib_tr = rp + W, *row_ax = sib_tr + nsib, *sib_ax = row_ax + A, *row_q = sib_ax + nsib,
              *sib_q = row_q + Q;
    if (!checks.merkle_ok(q, 0, row_tr, W, x_index, sib_tr, logN - cap_h, caps))
      throw VerifyError("Merkle path of the trace tree");
    if (!checks.merkle_ok(q, 1, row_ax, A, x_index, sib_ax, logN - cap_h, caps + capw))
      throw VerifyError("Merkle path of the auxiliary tree");
    if (!checks.merkle_ok(q, 2, row_q, Q, x_index, sib_q, logN - cap_h, caps + 2 * capw))
      throw VerifyError("Merkle path of the quotient tree");
    const u64 x = gl::mul(gl::COSET_SHIFT, gl::pow(wN, gl::brev32((u32)x_index, logN)));
    E2 f0 = X(0), f1 = X(0), f2 = X(0);
    for (int c = 0; c < W; c++) f1 = f1 + gl::emul_base(apow[c], row_tr[c]);
    for (int c = 0; c < A; c++) {
      f1 = f1 + gl::emul_base(apow[W + c], row_ax[c]);
      if (c >= nlk) f2 = f2 + gl::emul_base(apow[c - nlk], row_ax[c]);
    }
    f0 = f1;
    for (int c = 0; c < Q; c++) f0 = f0 + gl::emul_base(apow[W + A + c], row_q[c]);
    const E2 t0 = (f0 - O0) * gl::einv(X(x) - zeta);
    const E2 t1 = (f1 - O1) * gl::einv(X(x) - zeta_next);
    const E2 t2 = gl::emul_base(f2 - O2, gl::inv(gl::sub(x, 1)));
    E2 cur = (t0 * apow[W + A] + t1) * apow[2 * nch] + t2;
    const u64* lp = sib_q + nsib;
    int log_len = logN;
    u64 shift = gl::COSET_SHIFT;
    for (size_t li = 0; li < arities.size(); li++) {
      const int ab = (int)arities[li], arity = 1 << ab, log_leaves = log_len - ab;
      const u64* evals = lp;
      const u64* sib = lp + 2 * arity;
      const size_t coset = x_index >> ab, within = x_index & (size_t)(arity - 1);
      if (!(gl::e2(evals[2 * within], evals[2 * within + 1]) == cur)) throw VerifyError("FRI layer consistency");
      if (!checks.merkle_ok(q, 3 + (int)li, evals, 2 * (size_t)arity, coset, sib, log_leaves - cap_h, fri_caps + li * capw))
        throw VerifyError("Merkle path of the FRI layer tree");
      // fold (same formula as fri::FoldK)
      const u64 x0inv = gl::mul(gl::inv(shift), gl::pow(gl::inv(gl::root_of_unity(log_len)),
                                                         gl::brev32((u32)coset, log_leaves)));
      const E2 yb = gl::emul_base(fri_betas[li], x0inv);
      const u64 h_inv = gl::inv(gl::root_of_unity(ab));
      u64 hm = 1;
      E2 acc = X(0);
      for (int m = 0; m < arity; m++) {
        const E2 tm = gl::emul_base(yb, hm);
        E2 gsum = X(1) + tm, pw = tm;
        for (int k = 1; k < ab; k++) {
          pw = pw * pw;
          gsum = gsum * (X(1) + pw);
        }
        const size_t e = gl::brev32((u32)m, ab);
        acc = acc + gl::e2(evals[2 * e], evals[2 * e + 1]) * gsum;
        hm = gl::mul(hm, h_inv);
      }
      cur = gl::emul_base(acc, gl::inv((u64)arity));
      lp = sib + 4 * (log_leaves - cap_h);
      x_index = coset;
      log_len = log_leaves;
      shift = gl::pow(shift, (u64)arity);
    }
    // final polynomial at this query's point of the last layer
    const u64 xf = gl::mul(shift, gl::pow(gl::root_of_unity(log_len), gl::brev32((u32)x_index, log_len)));
    E2 ev = X(0);
    for (size_t i = keep; i-- > 0;) ev = gl::emul_base(ev, xf) + gl::e2(final_poly[2 * i], final_poly[2 * i + 1]);
    if (!(ev == cur)) throw VerifyError("FRI final polynomial");
  }
}

static inline void verify_proof(int kind, const pb254_config& cfg, const u64* blob, size_t words, const u64* inputs,
                                const u64* timestamps, size_t K) {
  HostChecks host;
  verify_walk(kind, cfg, blob, words, inputs, timestamps, K, host);
}

}  // namespace verify
