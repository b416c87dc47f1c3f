// K1/K2 kernels and their host driver; see tracegen.h for the interface.
#include "tracegen.h"
#include "curve_io.cuh"
#include "gl.cuh"

namespace tg {

PB_HD void atomic_add_u64(u64* p, u64 v) {
#ifdef __CUDA_ARCH__
  atomicAdd((unsigned long long*)p, (unsigned long long)v);
#else
  __atomic_fetch_add(p, v, __ATOMIC_RELAXED);
#endif
}

// column-major trace writer for one row
struct RowW {
  u64* base;
  size_t stride, row;
  PB_HD void put(int col, u64 v) const { base[(size_t)col * stride + row] = v; }
};

// ---------------- limb-polynomial witnesses ---------------------------------------------------
#define TG_P16 {64839, 55420, 35862, 15392, 51853, 26737, 27281, 38785, 22621, 33153, 17846, 47184, 41001, 57649, 20082, 12388}
// p^-1 mod 2^272 in 16-bit digits
#define TG_PINV16 {40055, 7033, 63613, 30765, 38198, 57653, 33434, 24865, 9599, 59340, 13359, 10064, 29588, 28279, 56648, 2693, 54160}

#if PB_HOSTSIM
#define TG_NOINLINE static
#else
#define TG_NOINLINE static __host__ __device__ __noinline__
#endif

// 16 x 16 -> 31 signed limb product, accumulated into r (r must be initialised)
PB_HD void pol_mac(const int a[16], const int b[16], i64 r[31], int scale) {
#pragma unroll
  for (int i = 0; i < 16; i++) {
    const i64 ai = (i64)a[i] * scale;
#pragma unroll
    for (int j = 0; j < 16; j++) r[i + j] += ai * b[j];
  }
}

// generate_modulus_zero: input = 31 signed coefficients whose value at 2^16 is divisible by p.
// Writes 80 cells at columns [col, col + 80): sign | quot_abs[17] | aux_lo[31] | aux_hi[31].
// The quotient is obtained without a division: q = V * p^-1 mod 2^272 (exact, two's complement).
TG_NOINLINE void gen_modulus_zero(const i64* input, const RowW w, int col, int* err) {
  const int P16[16] = TG_P16;
  const int PINV[17] = TG_PINV16;
  // low 17 digits of V in two's complement
  int d[17];
  {
    i64 carry = 0;
#pragma unroll
    for (int i = 0; i < 17; i++) {
      i64 t = input[i] + carry;
      d[i] = (int)(t & 0xffff);
      carry = t >> 16;
    }
  }
  int q[17];
  {
    u64 carry = 0;
#pragma unroll
    for (int k = 0; k < 17; k++) {
      u64 s = carry;
#pragma unroll
      for (int i = 0; i <= k; i++) s += (u64)((u32)d[i] * (u32)PINV[k - i]);
      q[k] = (int)(s & 0xffff);
      carry = s >> 16;
    }
  }
  const bool neg = q[16] >= 0x8000;
  if (neg) {
    int carry = 1;
#pragma unroll
    for (int k = 0; k < 17; k++) {
      int t = (0xffff - q[k]) + carry;
      q[k] = t & 0xffff;
      carry = t >> 16;
    }
  }
  int any = 0;
#pragma unroll
  for (int k = 0; k < 17; k++) any |= q[k];
  w.put(col, (any != 0 && !neg) ? 1 : 0);
#pragma unroll
  for (int k = 0; k < 17; k++) w.put(col + 1 + k, (u64)q[k]);
  // constr = (input | 0) - qs (*) m ; aux = constr / (x - 2^16)
  const int sgn = neg ? -1 : 1;
  i64 prev = 0;
#pragma unroll
  for (int k = 0; k < 32; k++) {
    i64 c = k < 31 ? input[k] : 0;
#pragma unroll
    for (int i = 0; i < 17; i++) {
      const int j = k - i;
      if (j >= 0 && j < 16) c -= (i64)(sgn * q[i]) * P16[j];
    }
    if (k < 31) {
      i64 a = k == 0 ? -(c >> 16) : ((prev - c) >> 16);
      // exactness of the shift (the reference relies on it; a failure means input != 0 mod p)
      i64 chk = k == 0 ? -c : (prev - c);
      if (chk & 0xffff) set_err(err, ERR_INTERNAL);
      prev = a;
      i64 t = a + ((i64)1 << 29);
      if (t < 0 || t > ((i64)1 << 30)) set_err(err, ERR_INTERNAL);
      w.put(col + 18 + k, (u64)(t & 0xffff));
      w.put(col + 49 + k, (u64)((t >> 16) & 0xffff));
    } else {
      if (prev - c != 0) set_err(err, ERR_INTERNAL);
    }
  }
}

// generate_is_modulus_zero: input 16 signed limbs (a difference of canonical values), inv16 = limbs
// of its inverse mod p (or 0), is_zero. Writes 96 cells at [col, col+96): inv[16] | ModulusZeroAux.
PB_HD void gen_is_modulus_zero(const int input[16], const int inv16[16], int is_zero, const RowW w, int col,
                               int* err) {
  i64 diff[31];
#pragma unroll
  for (int i = 0; i < 31; i++) diff[i] = 0;
  pol_mac(input, inv16, diff, 1);
  diff[0] += is_zero - 1;
#pragma unroll
  for (int i = 0; i < 16; i++) w.put(col + i, (u64)inv16[i]);
  gen_modulus_zero(diff, w, col + 16, err);
}

PB_HD void put_limbs(const RowW w, int col, const int l[16]) {
#pragma unroll
  for (int i = 0; i < 16; i++) w.put(col + i, (u64)l[i]);
}

// round flags table: rf[r] = {is_first, is_last, counter, inv_counter, inv_counter_prime}
struct RoundFlagsK {
  u64* table;  // PERIOD x 5
  PB_HD void operator()(size_t r) const {
    u64 counter = (u64)r, cprime = gl::sub(counter, (u64)(PERIOD - 1));
    table[r * 5 + 0] = counter == 0;
    table[r * 5 + 1] = cprime == 0;
    table[r * 5 + 2] = counter;
    table[r * 5 + 3] = counter ? gl::inv(counter) : 0;
    table[r * 5 + 4] = cprime ? gl::inv(cprime) : 0;
  }
};

PB_HD void put_common(const Layout& l, const RowW w, int r, const u64* scalar_words, const u64* rf_table, u64 ts) {
  const int shift = r >> 1;
  for (int i = 0; i < NBITS; i++) {
    int bi = (i + shift) & (NBITS - 1);
    w.put(l.bits + i, (scalar_words[bi >> 6] >> (bi & 63)) & 1);
  }
#pragma unroll
  for (int i = 0; i < 5; i++) w.put(l.rf + i, rf_table[r * 5 + i]);
  w.put(l.ts, ts);
  const bool adding = (r & 1) == 0;
  w.put(l.flag_op, adding ? 1 : 0);
  w.put(l.flag_sq_nl, adding ? 0 : (r == PERIOD - 1 ? 0 : 1));
  w.put(l.filter, 1);
  w.put(l.freq, 0);
}

// ---------------- curve STARKs (G1: F = bn::F1, G2: F = bn::F2) ------------------------------
template <class F>
struct CurveBufs {
  bn::Aff<F>* D;    // [257][K] affine doubles (Montgomery form), D[0] = x
  bn::Aff<F>* T;    // [256][K] affine T_j
  bn::Jac<F>* tmp;  // [256][K] Jacobian scratch
  typename F::T* pref;  // [256][K] prefix products scratch
  bn::Aff<F>* off;  // [K] offsets
  short* sidx;      // [256][K] index of the T giving S_j, or -1 for the offset
  bn::Fq* den;      // [NDEN][512][K] slope denominators then their inverses
  int* err;
};

// Jacobian -> affine for tmp[0..cnt) of instance k into dst[(j0 + j)][k] using one inversion
template <class F>
PB_HD void batch_to_affine(const CurveBufs<F>& B, size_t k, size_t K, int cnt, bn::Aff<F>* dst, int j0) {
  typedef typename F::T T;
  T acc = F::one();
  for (int j = 0; j < cnt; j++) {
    B.pref[(size_t)j * K + k] = acc;
    acc = F::mul(acc, B.tmp[(size_t)j * K + k].Z);
  }
  T inv = F::inv(acc);
  for (int j = cnt - 1; j >= 0; j--) {
    const bn::Jac<F> p = B.tmp[(size_t)j * K + k];
    T zi = F::mul(inv, B.pref[(size_t)j * K + k]);
    inv = F::mul(inv, p.Z);
    T zi2 = F::sqr(zi);
    bn::Aff<F> a;
    a.x = F::mul(p.X, zi2);
    a.y = F::mul(p.Y, F::mul(zi, zi2));
    dst[(size_t)(j0 + j) * K + k] = a;
  }
}

template <class F>
struct ChainsK {
  CurveBufs<F> B;
  const u64* inputs;  // [K][in_words]
  int in_words;
  size_t K;
  PB_HD void operator()(size_t k) const {
    typedef typename F::T T;
    const u64* w = inputs + k * in_words;
    const int FW = FieldIO<F>::WORDS;
    bn::Aff<F> x, off;
    bool ok = FieldIO<F>::load(w + 4, x.x) & FieldIO<F>::load(w + 4 + FW, x.y) &
              FieldIO<F>::load(w + 4 + 2 * FW, off.x) & FieldIO<F>::load(w + 4 + 3 * FW, off.y);
    if (!ok) {
      set_err(B.err, ERR_NOT_CANONICAL);
      return;
    }
    // G1Affine / G2Affine are points of the curve by construction in the reference; the step-parallel chains below
    // rely on the group law being associative, which only holds on the curve
    if (!FieldIO<F>::on_curve(x) || !FieldIO<F>::on_curve(off)) {
      set_err(B.err, ERR_NOT_ON_CURVE);
      return;
    }
    B.D[k] = x;
    B.off[k] = off;
    // doubling chain
    bn::Jac<F> p;
    p.X = x.x;
    p.Y = x.y;
    p.Z = F::one();
    for (int j = 0; j < 256; j++) {
      if (F::is_zero(p.Y)) set_err(B.err, ERR_INFINITY);  // 2-torsion: doubling gives infinity
      p = bn::jac_double<F>(p);
      B.tmp[(size_t)j * K + k] = p;
    }
    batch_to_affine<F>(B, k, K, 256, B.D, 1);
    // running-sum chain: T_j = S_(j-1) + D_j
    bn::Jac<F> s;
    s.X = off.x;
    s.Y = off.y;
    s.Z = F::one();
    short cur = -1;
    for (int j = 0; j < 256; j++) {
      int st;
      bn::Jac<F> t = bn::jac_add_mixed<F>(s, B.D[(size_t)j * K + k], st);
      if (st == 2) {
        set_err(B.err, ERR_INFINITY);
        t = s;  // keep Z != 0 so that the batched inversion stays well defined
      }
      if (st == 1 && F::is_zero(s.Y)) set_err(B.err, ERR_INFINITY);
      B.tmp[(size_t)j * K + k] = t;
      if (scalar_bit(w, j)) {
        s = t;
        cur = (short)j;
      }
      B.sidx[(size_t)j * K + k] = cur;
    }
    batch_to_affine<F>(B, k, K, 256, B.T, 0);
  }
};

#if !PB_HOSTSIM
// ---- the same chains with instance- AND step-level parallelism (device build) -----------------------------
// ChainsK walks both 256-step chains of an instance in one thread: with 2^10 instances that is 32 warps on a
// 148-SM machine, purely latency-bound (9.6 ms for G1, 48 ms for G2). Only the doubling chain is inherently
// sequential. The running sums S_j = offset + sum_{i <= j, bit_i} D_i are a prefix sum in the curve group, so
// they are computed by a 256-thread block per instance with an 8-step scan of complete Jacobian additions; the
// row values T_j = S_(j-1) + D_j are then one mixed addition per thread - the reference's own addition, with
// its status checks - and every Jacobian -> affine conversion is an independent Fermat inversion per thread.
// Affine coordinates are unique, so the trace is bit-identical to the sequential walk.
template <class F>
__global__ void __launch_bounds__(32) k_dbl_chain(CurveBufs<F> B, const u64* __restrict__ inputs, int in_words, size_t K) {
  const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const u64* w = inputs + k * in_words;
  const int FW = FieldIO<F>::WORDS;
  bn::Aff<F> x, off;
  bool ok = FieldIO<F>::load(w + 4, x.x) & FieldIO<F>::load(w + 4 + FW, x.y) &
            FieldIO<F>::load(w + 4 + 2 * FW, off.x) & FieldIO<F>::load(w + 4 + 3 * FW, off.y);
  if (!ok) {
    set_err(B.err, ERR_NOT_CANONICAL);
    x.x = x.y = off.x = off.y = F::one();  // keep the later kernels well defined; the error word wins
  } else if (!FieldIO<F>::on_curve(x) || !FieldIO<F>::on_curve(off)) {
    // the prefix scan of k_sum_scan re-associates the additions: only valid in the curve group
    set_err(B.err, ERR_NOT_ON_CURVE);
    x.x = x.y = off.x = off.y = F::one();
  }
  B.D[k] = x;
  B.off[k] = off;
  bn::Jac<F> p;
  p.X = x.x;
  p.Y = x.y;
  p.Z = F::one();
  for (int j = 0; j < 256; j++) {
    if (F::is_zero(p.Y)) set_err(B.err, ERR_INFINITY);  // 2-torsion: doubling gives infinity
    p = bn::jac_double<F>(p);
    B.tmp[(size_t)j * K + k] = p;
  }
}

template <class F>
__global__ void __launch_bounds__(256) k_sum_scan(CurveBufs<F> B, bn::Jac<F>* __restrict__ ping, bn::Jac<F>* __restrict__ pong,
                                                  const u64* __restrict__ inputs, int in_words, size_t K) {
  const size_t k = blockIdx.x;
  const int j = threadIdx.x;  // 0..255
  const u64* w = inputs + k * in_words;
  const bool bit = scalar_bit(w, j);
  bn::Jac<F> e;
  if (bit) {
    const bn::Aff<F> d = B.D[(size_t)j * K + k];
    e.X = d.x;
    e.Y = d.y;
    e.Z = F::one();
  } else {
    e.X = F::one();
    e.Y = F::one();
    e.Z = F::zero();
  }
  // inclusive Hillis-Steele scan over the 256 steps of this instance (global ping-pong buffers, [j][K] layout)
  bn::Jac<F>* cur = ping;
  bn::Jac<F>* nxt = pong;
  cur[(size_t)j * K + k] = e;
  __syncthreads();
  for (int d = 1; d < 256; d <<= 1) {
    bn::Jac<F> v = cur[(size_t)j * K + k];
    if (j >= d) v = bn::jac_add_complete<F>(cur[(size_t)(j - d) * K + k], v);
    nxt[(size_t)j * K + k] = v;
    __syncthreads();
    bn::Jac<F>* t = cur;
    cur = nxt;
    nxt = t;
  }
  // S_(j-1) = offset + P_(j-1)
  const bn::Aff<F> off = B.off[k];
  bn::Jac<F> sprev;
  sprev.X = off.x;
  sprev.Y = off.y;
  sprev.Z = F::one();
  if (j > 0) sprev = bn::jac_add_complete<F>(cur[(size_t)(j - 1) * K + k], sprev);
  if (F::is_zero(sprev.Z)) {  // an earlier row produced the point at infinity (flagged there as well)
    set_err(B.err, ERR_INFINITY);
    sprev.X = off.x;
    sprev.Y = off.y;
    sprev.Z = F::one();
  }
  int st;
  bn::Jac<F> t = bn::jac_add_mixed<F>(sprev, B.D[(size_t)j * K + k], st);
  if (st == 2) {
    set_err(B.err, ERR_INFINITY);
    t = sprev;
  }
  if (st == 1 && F::is_zero(sprev.Y)) set_err(B.err, ERR_INFINITY);
  __syncthreads();  // everyone has read the scan result before it is overwritten with T
  nxt[(size_t)j * K + k] = t;  // Jacobian T_j; k_to_affine turns it into B.T
  // index of the T that gives S_j: the last set bit at or below j, or -1 (the offset)
  int last = -1;
  for (int wi = j >> 6; wi >= 0 && last < 0; wi--) {
    u64 m = w[wi];
    if (wi == (j >> 6) && (j & 63) != 63) m &= (((u64)2) << (j & 63)) - 1;
    if (m) last = wi * 64 + 63 - __clzll((long long)m);
  }
  B.sidx[(size_t)j * K + k] = (short)last;
}
#endif

// operands of row r of instance k
template <class F>
PB_HD void row_operands(const CurveBufs<F>& B, size_t k, size_t K, int r, bn::Aff<F>& a, bn::Aff<F>& b) {
  const int j = r >> 1;
  b = B.D[(size_t)j * K + k];
  if (r & 1) {
    a = b;
  } else {
    short si = j == 0 ? (short)-1 : B.sidx[(size_t)(j - 1) * K + k];
    a = si < 0 ? B.off[k] : B.T[(size_t)si * K + k];
  }
}

// den[0] = slope denominator; G2 additionally den[1], den[2] = delta_x.c0, delta_x.c1 (zero -> 1)
template <class F>
struct DensK;
template <>
struct DensK<bn::F1> {
  CurveBufs<bn::F1> B;
  size_t K;
  PB_HD void operator()(size_t gid) const {
    size_t k = gid / PERIOD;
    int r = (int)(gid % PERIOD);
    bn::Aff<bn::F1> a, b;
    row_operands<bn::F1>(B, k, K, r, a, b);
    bn::Fq dx = bn::sub(b.x, a.x);
    bn::Fq den = bn::is_zero(dx) ? bn::dbl(a.y) : dx;
    if (bn::is_zero(den)) {
      set_err(B.err, ERR_INFINITY);
      den = bn::one();
    }
    B.den[(size_t)r * K + k] = den;
  }
};
template <>
struct DensK<bn::F2> {
  CurveBufs<bn::F2> B;
  size_t K;
  PB_HD void operator()(size_t gid) const {
    size_t k = gid / PERIOD;
    int r = (int)(gid % PERIOD);
    bn::Aff<bn::F2> a, b;
    row_operands<bn::F2>(B, k, K, r, a, b);
    bn::Fq2 dx = bn::F2::sub(b.x, a.x);
    bn::Fq2 d2 = bn::F2::is_zero(dx) ? bn::F2::dbl(a.y) : dx;
    bn::Fq norm = bn::add(bn::sqr(d2.c0), bn::sqr(d2.c1));
    if (bn::is_zero(norm)) {
      set_err(B.err, ERR_INFINITY);
      norm = bn::one();
    }
    const size_t plane = (size_t)PERIOD * K;
    B.den[(size_t)r * K + k] = norm;
    B.den[plane + (size_t)r * K + k] = bn::is_zero(dx.c0) ? bn::one() : dx.c0;
    B.den[2 * plane + (size_t)r * K + k] = bn::is_zero(dx.c1) ? bn::one() : dx.c1;
  }
};

// in-place batched inversion of non-zero Montgomery-form elements, 16 per thread
struct BatchInvK {
  bn::Fq* v;
  size_t n;
  PB_HD void operator()(size_t t) const {
    const int CH = 16;
    size_t base = t * CH;
    int cnt = (int)((n - base) < (size_t)CH ? (n - base) : (size_t)CH);
    bn::Fq pref[CH];
    bn::Fq acc = bn::one();
    for (int i = 0; i < cnt; i++) {
      pref[i] = acc;
      acc = bn::mul(acc, v[base + i]);
    }
    bn::Fq inv = bn::inv(acc);
    for (int i = cnt - 1; i >= 0; i--) {
      bn::Fq x = v[base + i];
      v[base + i] = bn::mul(inv, pref[i]);
      inv = bn::mul(inv, x);
    }
  }
};

PB_HD void fq_limbs(const bn::Fq& mont, int out[16]) { bn::to_limbs16(bn::from_mont(mont), out); }

// G1 rows
struct RowsG1K {
  CurveBufs<bn::F1> B;
  Layout l;
  const u64* inputs;
  const u64* timestamps;
  const u64* rf_table;
  u64* trace;
  size_t n_rows, K;
  PB_HD void operator()(size_t gid) const {
    const size_t k = gid / PERIOD;
    const int r = (int)(gid % PERIOD), j = r >> 1;
    RowW w{trace, n_rows, gid};
    bn::Aff<bn::F1> a, b;
    row_operands<bn::F1>(B, k, K, r, a, b);
    const bn::Fq dinv = B.den[(size_t)r * K + k];
    const bn::Fq dxm = bn::sub(b.x, a.x);
    const int is_x_eq = bn::is_zero(dxm) ? 1 : 0;
    if (is_x_eq && !bn::eq(a.y, b.y)) set_err(B.err, ERR_INFINITY);  // a = -b (g1/add.rs:76-78)
    bn::Fq lam;
    if (is_x_eq) {
      bn::Fq x2 = bn::sqr(a.x);
      lam = bn::mul(bn::add(bn::dbl(x2), x2), dinv);
    } else {
      lam = bn::mul(bn::sub(b.y, a.y), dinv);
    }
    bn::Aff<bn::F1> c;
    c.x = bn::sub(bn::sub(bn::sqr(lam), a.x), b.x);
    c.y = bn::sub(bn::mul(lam, bn::sub(a.x, c.x)), a.y);
    int ax[16], ay[16], bx[16], by[16], cx[16], cy[16], lm[16], iv[16], t16[16];
    fq_limbs(a.x, ax);
    fq_limbs(a.y, ay);
    fq_limbs(b.x, bx);
    fq_limbs(b.y, by);
    fq_limbs(c.x, cx);
    fq_limbs(c.y, cy);
    fq_limbs(lam, lm);
    if (is_x_eq) {
#pragma unroll
      for (int i = 0; i < 16; i++) iv[i] = 0;
    } else {
      fq_limbs(dinv, iv);
    }
    // registers
    put_limbs(w, l.a, ax);
    put_limbs(w, l.a + 16, ay);
    put_limbs(w, l.b, bx);
    put_limbs(w, l.b + 16, by);
    put_limbs(w, l.c, cx);
    put_limbs(w, l.c + 16, cy);
    // double: adding row -> D_j (= b); doubling row -> D_(j+1) (= c)
    if (r & 1) {
      put_limbs(w, l.reg0, cx);
      put_limbs(w, l.reg0 + 16, cy);
    } else {
      put_limbs(w, l.reg0, bx);
      put_limbs(w, l.reg0 + 16, by);
    }
    // sum: S_j
    {
      const u64* sw = inputs + k * l.in_words;
      bool take_c = !(r & 1) && scalar_bit(sw, j);
      if (take_c) {
        put_limbs(w, l.reg1, cx);
        put_limbs(w, l.reg1 + 16, cy);
      } else if (!(r & 1)) {
        put_limbs(w, l.reg1, ax);
        put_limbs(w, l.reg1 + 16, ay);
      } else {
        short si = B.sidx[(size_t)j * K + k];
        bn::Aff<bn::F1> s = si < 0 ? B.off[k] : B.T[(size_t)si * K + k];
        fq_limbs(s.x, t16);
        put_limbs(w, l.reg1, t16);
        fq_limbs(s.y, t16);
        put_limbs(w, l.reg1 + 16, t16);
      }
      put_common(l, w, r, sw, rf_table, timestamps[k]);
    }
    // add_aux
    const int A = l.aux;
    int dx[16];
#pragma unroll
    for (int i = 0; i < 16; i++) dx[i] = bx[i] - ax[i];
    w.put(A, (u64)is_x_eq);
    gen_is_modulus_zero(dx, iv, is_x_eq, w, A + 1, B.err);
    w.put(A + 97, (u64)is_x_eq);
    put_limbs(w, A + 98, lm);
    i64 diff[31];
#pragma unroll
    for (int i = 0; i < 31; i++) diff[i] = 0;
    if (!is_x_eq) {
      pol_mac(lm, dx, diff, 1);
#pragma unroll
      for (int i = 0; i < 16; i++) diff[i] -= by[i] - ay[i];
    } else {
      pol_mac(lm, ay, diff, 2);
      pol_mac(ax, ax, diff, -3);
    }
    gen_modulus_zero(diff, w, A + 114, B.err);
#pragma unroll
    for (int i = 0; i < 31; i++) diff[i] = 0;
    pol_mac(lm, lm, diff, 1);
#pragma unroll
    for (int i = 0; i < 16; i++) diff[i] -= ax[i] + bx[i] + cx[i];
    gen_modulus_zero(diff, w, A + 194, B.err);
#pragma unroll
    for (int i = 0; i < 31; i++) diff[i] = 0;
#pragma unroll
    for (int i = 0; i < 16; i++) t16[i] = cx[i] - ax[i];
    pol_mac(lm, t16, diff, 1);
#pragma unroll
    for (int i = 0; i < 16; i++) diff[i] += cy[i] + ay[i];
    gen_modulus_zero(diff, w, A + 274, B.err);
  }
};

// ---- G2 ------------------------------------------------------------------------------------
struct Ext16 {
  int c0[16], c1[16];
};
PB_HD Ext16 fq2_limbs(const bn::Fq2& m) {
  Ext16 r;
  fq_limbs(m.c0, r.c0);
  fq_limbs(m.c1, r.c1);
  return r;
}
PB_HD void put_ext(const RowW w, int col, const Ext16& e) {
  put_limbs(w, col, e.c0);
  put_limbs(w, col + 16, e.c1);
}
// (x * y) in Fq2 on limb polynomials, scaled: c0 += s (x0 y0 - x1 y1), c1 += s (x0 y1 + x1 y0)
PB_HD void ext_mac(const Ext16& x, const Ext16& y, i64 c0[31], i64 c1[31], int s) {
  pol_mac(x.c0, y.c0, c0, s);
  pol_mac(x.c1, y.c1, c0, -s);
  pol_mac(x.c0, y.c1, c1, s);
  pol_mac(x.c1, y.c0, c1, s);
}

struct RowsG2K {
  CurveBufs<bn::F2> B;
  Layout l;
  const u64* inputs;
  const u64* timestamps;
  const u64* rf_table;
  u64* trace;
  size_t n_rows, K;
  PB_HD void operator()(size_t gid) const {
    typedef bn::F2 F;
    const size_t k = gid / PERIOD;
    const int r = (int)(gid % PERIOD), j = r >> 1;
    RowW w{trace, n_rows, gid};
    bn::Aff<F> a, b;
    row_operands<F>(B, k, K, r, a, b);
    const size_t plane = (size_t)PERIOD * K;
    const bn::Fq ninv = B.den[(size_t)r * K + k];
    const bn::Fq i0 = B.den[plane + (size_t)r * K + k], i1 = B.den[2 * plane + (size_t)r * K + k];
    const bn::Fq2 dxm = F::sub(b.x, a.x);
    const int z0 = bn::is_zero(dxm.c0) ? 1 : 0, z1 = bn::is_zero(dxm.c1) ? 1 : 0;
    const int is_x_eq = z0 & z1;
    if (is_x_eq && !(bn::eq(a.y.c0, b.y.c0) && bn::eq(a.y.c1, b.y.c1))) set_err(B.err, ERR_INFINITY);
    // 1/d = conj(d) / norm(d) with d = delta_x or 2 a.y
    bn::Fq2 d = is_x_eq ? F::dbl(a.y) : dxm;
    bn::Fq2 dinv = bn::Fq2{bn::mul(d.c0, ninv), bn::mul(bn::neg(d.c1), ninv)};
    bn::Fq2 lam;
    if (is_x_eq) {
      bn::Fq2 x2 = F::sqr(a.x);
      lam = F::mul(F::add(F::dbl(x2), x2), dinv);
    } else {
      lam = F::mul(F::sub(b.y, a.y), dinv);
    }
    bn::Aff<F> c;
    c.x = F::sub(F::sub(F::sqr(lam), a.x), b.x);
    c.y = F::sub(F::mul(lam, F::sub(a.x, c.x)), a.y);
    Ext16 ax = fq2_limbs(a.x), ay = fq2_limbs(a.y), bx = fq2_limbs(b.x), by = fq2_limbs(b.y);
    Ext16 cx = fq2_limbs(c.x), cy = fq2_limbs(c.y), lm = fq2_limbs(lam);
    put_ext(w, l.a, ax);
    put_ext(w, l.a + 32, ay);
    put_ext(w, l.b, bx);
    put_ext(w, l.b + 32, by);
    put_ext(w, l.c, cx);
    put_ext(w, l.c + 32, cy);
    if (r & 1) {
      put_ext(w, l.reg0, cx);
      put_ext(w, l.reg0 + 32, cy);
    } else {
      put_ext(w, l.reg0, bx);
      put_ext(w, l.reg0 + 32, by);
    }
    {
      const u64* sw = inputs + k * l.in_words;
      bool take_c = !(r & 1) && scalar_bit(sw, j);
      if (take_c) {
        put_ext(w, l.reg1, cx);
        put_ext(w, l.reg1 + 32, cy);
      } else if (!(r & 1)) {
        put_ext(w, l.reg1, ax);
        put_ext(w, l.reg1 + 32, ay);
      } else {
        short si = B.sidx[(size_t)j * K + k];
        bn::Aff<F> s = si < 0 ? B.off[k] : B.T[(size_t)si * K + k];
        put_ext(w, l.reg1, fq2_limbs(s.x));
        put_ext(w, l.reg1 + 32, fq2_limbs(s.y));
      }
      put_common(l, w, r, sw, rf_table, timestamps[k]);
    }
    const int A = l.aux;
    Ext16 dx;
#pragma unroll
    for (int i = 0; i < 16; i++) {
      dx.c0[i] = bx.c0[i] - ax.c0[i];
      dx.c1[i] = bx.c1[i] - ax.c1[i];
    }
    int iv0[16], iv1[16];
    if (z0) {
#pragma unroll
      for (int i = 0; i < 16; i++) iv0[i] = 0;
    } else {
      fq_limbs(i0, iv0);
    }
    if (z1) {
#pragma unroll
      for (int i = 0; i < 16; i++) iv1[i] = 0;
    } else {
      fq_limbs(i1, iv1);
    }
    w.put(A, (u64)is_x_eq);
    w.put(A + 1, (u64)z0);
    w.put(A + 2, (u64)z1);
    gen_is_modulus_zero(dx.c0, iv0, z0, w, A + 3, B.err);
    gen_is_modulus_zero(dx.c1, iv1, z1, w, A + 99, B.err);
    w.put(A + 195, (u64)is_x_eq);
    put_ext(w, A + 196, lm);
    i64 d0[31], d1[31];
#pragma unroll
    for (int i = 0; i < 31; i++) d0[i] = d1[i] = 0;
    if (!is_x_eq) {
      ext_mac(lm, dx, d0, d1, 1);
#pragma unroll
      for (int i = 0; i < 16; i++) {
        d0[i] -= by.c0[i] - ay.c0[i];
        d1[i] -= by.c1[i] - ay.c1[i];
      }
    } else {
      ext_mac(lm, ay, d0, d1, 2);
      ext_mac(ax, ax, d0, d1, -3);
    }
    gen_modulus_zero(d0, w, A + 228, B.err);
    gen_modulus_zero(d1, w, A + 308, B.err);
#pragma unroll
    for (int i = 0; i < 31; i++) d0[i] = d1[i] = 0;
    ext_mac(lm, lm, d0, d1, 1);
#pragma unroll
    for (int i = 0; i < 16; i++) {
      d0[i] -= ax.c0[i] + bx.c0[i] + cx.c0[i];
      d1[i] -= ax.c1[i] + bx.c1[i] + cx.c1[i];
    }
    gen_modulus_zero(d0, w, A + 388, B.err);
    gen_modulus_zero(d1, w, A + 468, B.err);
#pragma unroll
    for (int i = 0; i < 31; i++) d0[i] = d1[i] = 0;
    Ext16 t;
#pragma unroll
    for (int i = 0; i < 16; i++) {
      t.c0[i] = cx.c0[i] - ax.c0[i];
      t.c1[i] = cx.c1[i] - ax.c1[i];
    }
    ext_mac(lm, t, d0, d1, 1);
#pragma unroll
    for (int i = 0; i < 16; i++) {
      d0[i] += cy.c0[i] + ay.c0[i];
      d1[i] += cy.c1[i] + ay.c1[i];
    }
    gen_modulus_zero(d0, w, A + 548, B.err);
    gen_modulus_zero(d1, w, A + 628, B.err);
  }
};

// ---- Fq exponentiation ------------------------------------------------------------------------
struct FqBufs {
  bn::Fq* SQ;   // [257][K]  x^(2^j), Montgomery form
  bn::Fq* T;    // [256][K]  product_(j-1) * square_j
  short* sidx;  // [256][K]
  int* err;
};
struct FqChainsK {
  FqBufs B;
  const u64* inputs;
  size_t K;
  PB_HD void operator()(size_t k) const {
    const u64* w = inputs + k * 8;
    if (!words_lt_p(w + 4)) {
      set_err(B.err, ERR_NOT_CANONICAL);
      return;
    }
    bn::Fq sq = bn::to_mont(bn::from_words(w + 4));
    bn::Fq prod = bn::one();
    short cur = -1;
    B.SQ[k] = sq;
    for (int j = 0; j < 256; j++) {
      bn::Fq t = bn::mul(prod, sq);
      B.T[(size_t)j * K + k] = t;
      if (scalar_bit(w, j)) {
        prod = t;
        cur = (short)j;
      }
      B.sidx[(size_t)j * K + k] = cur;
      sq = bn::sqr(sq);
      B.SQ[(size_t)(j + 1) * K + k] = sq;
    }
  }
};
struct RowsFqK {
  FqBufs B;
  Layout l;
  const u64* inputs;
  const u64* timestamps;
  const u64* rf_table;
  u64* trace;
  size_t n_rows, K;
  PB_HD void operator()(size_t gid) const {
    const size_t k = gid / PERIOD;
    const int r = (int)(gid % PERIOD), j = r >> 1;
    RowW w{trace, n_rows, gid};
    const u64* sw = inputs + k * l.in_words;
    bn::Fq b = B.SQ[(size_t)j * K + k], a, c, prod;
    short si_prev = j == 0 ? (short)-1 : B.sidx[(size_t)(j - 1) * K + k];
    short si = B.sidx[(size_t)j * K + k];
    bn::Fq s_prev = si_prev < 0 ? bn::one() : B.T[(size_t)si_prev * K + k];
    bn::Fq s_cur = si < 0 ? bn::one() : B.T[(size_t)si * K + k];
    if (r & 1) {
      a = b;
      c = B.SQ[(size_t)(j + 1) * K + k];
      prod = s_cur;
    } else {
      a = s_prev;
      c = B.T[(size_t)j * K + k];
      prod = s_cur;
    }
    int al[16], bl[16], cl[16], t16[16];
    fq_limbs(a, al);
    fq_limbs(b, bl);
    fq_limbs(c, cl);
    put_limbs(w, l.a, al);
    put_limbs(w, l.b, bl);
    put_limbs(w, l.c, cl);
    if (r & 1)
      put_limbs(w, l.reg0, cl);
    else
      put_limbs(w, l.reg0, bl);
    fq_limbs(prod, t16);
    put_limbs(w, l.reg1, t16);
    put_common(l, w, r, sw, rf_table, timestamps[k]);
    i64 diff[31];
#pragma unroll
    for (int i = 0; i < 31; i++) diff[i] = 0;
    pol_mac(al, bl, diff, 1);
#pragma unroll
    for (int i = 0; i < 16; i++) diff[i] -= cl[i];
    gen_modulus_zero(diff, w, l.aux, B.err);
  }
};

// ---- padding, range counter, range-check histogram -----------------------------------------
struct ZeroPadK {  // zero rows [used, n) of every column
  u64* trace;
  size_t n_rows, used, pad;
  PB_HD void operator()(size_t gid) const {
    size_t col = gid / pad, i = gid % pad;
    trace[col * n_rows + used + i] = 0;
  }
};
struct RangeCounterK {
  u64* col;
  size_t row0;  // index of local row 0 in the whole trace (row-block form)
  PB_HD void operator()(size_t i) const { col[i] = row0 + i < 65536 ? (u64)(row0 + i) : 65535; }
};
struct HistK {  // one thread per used row: frequency[v] += 1 for every range-checked cell
  const u64* trace;
  u64* freq;
  size_t n_rows;
  int rc_lo, rc_hi;
  int* err;
  PB_HD void operator()(size_t row) const {
    for (int c = rc_lo; c < rc_hi; c++) {
      u64 v = trace[(size_t)c * n_rows + row];
      if (v >= 65536) {
        set_err(err, ERR_INTERNAL);
        continue;
      }
      atomic_add_u64(freq + v, 1);
    }
  }
};
#if !PB_HOSTSIM
// K2 on the device: the 2^16-bin histogram lives in shared memory, half of the bins per CTA (32768 x u32 =
// 128 KB), so the (rc_hi - rc_lo) x used cells cost shared-memory atomics instead of global ones; every CTA
// of a half streams its row range of all range-checked columns (coalesced 8-byte loads, the matrix is read
// twice in total) and flushes its non-zero bins with one global atomic each. Zero cells - by far the most
// frequent value - are counted with a warp ballot.
__global__ void __launch_bounds__(1024) k_range_hist(const u64* __restrict__ trace, u64* __restrict__ freq, size_t n_rows,
                                                     size_t used, int rc_lo, int rc_hi, int* err) {
  extern __shared__ u32 hist[];
  const u32 half = blockIdx.y;
  for (int i = threadIdx.x; i < 32768; i += blockDim.x) hist[i] = 0;
  __syncthreads();
  const size_t per = ((used + gridDim.x - 1) / gridDim.x + 1023) & ~(size_t)1023;
  const size_t r0 = (size_t)blockIdx.x * per, r1 = r0 + per < used ? r0 + per : used;  // used is a multiple of 512
  const u32 lane = threadIdx.x & 31;
  bool bad = false;
  for (int c = rc_lo; c < rc_hi; c++) {
    const u64* col = trace + (size_t)c * n_rows;
    for (size_t base = r0 + (threadIdx.x & ~31u); base < r1; base += blockDim.x) {  // whole warps: 32 | r1
      const u64 v = col[base + lane];
      bad |= v >= 65536;
      const u32 zeros = __ballot_sync(0xffffffffu, v == 0);
      if (v == 0) {
        if (half == 0 && lane == (u32)(__ffs(zeros) - 1)) atomicAdd(&hist[0], (u32)__popc(zeros));
      } else if ((u32)(v >> 15) == half) {
        atomicAdd(&hist[(u32)v & 32767u], 1u);
      }
    }
  }
  if (bad) set_err(err, ERR_INTERNAL);
  __syncthreads();
  for (int i = threadIdx.x; i < 32768; i += blockDim.x) {
    const u32 h = hist[i];
    if (h) atomicAdd((unsigned long long*)(freq + half * 32768u + i), (unsigned long long)h);
  }
}
#endif
struct AddK {
  u64* p;
  u64 v;
  PB_HD void operator()(size_t) const { *p = gl::add(*p, v % gl::P); }
};

template <class F, class RowsK>
static inline void run_curve(Arena& ar, const Layout& l, const u64* d_inputs, const u64* d_ts, size_t K, size_t n_rows,
                             u64* d_trace, const u64* rf_table, int* d_err, pbStream s) {
  CurveBufs<F> B;
  B.D = ar.alloc_n<bn::Aff<F>>(257 * K);
  B.T = ar.alloc_n<bn::Aff<F>>(256 * K);
  B.tmp = ar.alloc_n<bn::Jac<F>>(256 * K);
  B.pref = ar.alloc_n<typename F::T>(256 * K);
  B.off = ar.alloc_n<bn::Aff<F>>(K);
  B.sidx = ar.alloc_n<short>(256 * K);
  const int nden = FieldIO<F>::NDEN;
  B.den = ar.alloc_n<bn::Fq>((size_t)nden * PERIOD * K);
  B.err = d_err;
#if PB_HOSTSIM
  pb_launch("tracegen chains", ChainsK<F>{B, d_inputs, l.in_words, K}, K, s, 32);
#else
  {
    bn::Jac<F>* pong = ar.alloc_n<bn::Jac<F>>(256 * K);
    k_dbl_chain<F><<<(unsigned)((K + 31) / 32), 32, 0, s>>>(B, d_inputs, l.in_words, K);
    k_to_affine<F><<<(unsigned)((256 * K / AFF_CH + 127) / 128), 128, 0, s>>>(B.tmp, B.D, 256 * K, K, d_err);
    // ping = B.tmp (free again), pong: the scan ends in ping after 8 swaps and the Jacobian T_j land in pong
    k_sum_scan<F><<<(unsigned)K, 256, 0, s>>>(B, B.tmp, pong, d_inputs, l.in_words, K);
    k_to_affine<F><<<(unsigned)((256 * K / AFF_CH + 127) / 128), 128, 0, s>>>(pong, B.T, 256 * K, 0, d_err);
    g_pb_launches += 4;
    pb_check_last("tracegen chains");
  }
#endif
  pb_launch("tracegen dens", DensK<F>{B, K}, K * PERIOD, s, 128);
  size_t nd = (size_t)nden * PERIOD * K;
  pb_launch("tracegen batchinv", BatchInvK{B.den, nd}, (nd + 15) / 16, s, 64);
  // 128 registers (a few spilled words) and twice the resident warps beat 255 registers: 2.4 -> 1.7 ms for 1024 G1 instances
  pb_launch_lb<64, 8>("tracegen rows", RowsK{B, l, d_inputs, d_ts, rf_table, d_trace, n_rows, K}, K * PERIOD, s);
}

void generate(Arena& ar, int kind, const u64* d_inputs, const u64* d_ts, size_t K, size_t n_rows,
                            u64* d_trace, int* d_err, pbStream s, size_t row0) {
  Layout l = layout_for(kind);
  const size_t used = K * PERIOD;
  u64* rf_table = ar.alloc_n<u64>(PERIOD * 5);
  pb_launch("round flags", RoundFlagsK{rf_table}, PERIOD, s, 64);
  if (used < n_rows) {
    size_t pad = n_rows - used;
    pb_launch("zero pad", ZeroPadK{d_trace, n_rows, used, pad}, pad * (size_t)l.width, s);
  }
  if (K > 0) {
    if (kind == 0) {
      run_curve<bn::F1, RowsG1K>(ar, l, d_inputs, d_ts, K, n_rows, d_trace, rf_table, d_err, s);
    } else if (kind == 1) {
      run_curve<bn::F2, RowsG2K>(ar, l, d_inputs, d_ts, K, n_rows, d_trace, rf_table, d_err, s);
    } else {
      FqBufs B;
      B.SQ = ar.alloc_n<bn::Fq>(257 * K);
      B.T = ar.alloc_n<bn::Fq>(256 * K);
      B.sidx = ar.alloc_n<short>(256 * K);
      B.err = d_err;
      pb_launch("tracegen fq chains", FqChainsK{B, d_inputs, K}, K, s, 32);
      pb_launch("tracegen fq rows", RowsFqK{B, l, d_inputs, d_ts, rf_table, d_trace, n_rows, K}, K * PERIOD, s, 64);
    }
  }
  pb_launch("range counter", RangeCounterK{d_trace + (size_t)l.range_counter * n_rows, row0}, n_rows, s);
  u64* freq = d_trace + (size_t)l.freq * n_rows;
#if PB_HOSTSIM
  if (used > 0) pb_launch("range histogram", HistK{d_trace, freq, n_rows, l.rc_lo, l.rc_hi, d_err}, used, s, 128);
#else
  if (used > 0) {
    static bool attr_set[64] = {};  // per device
    static std::mutex attr_mutex;
    int dev = 0;
    PB_CUDA(cudaGetDevice(&dev));
    if (dev < 0 || dev >= 64) dev = 63;
    {
      std::lock_guard<std::mutex> lock(attr_mutex);
      if (!attr_set[dev]) {
        PB_CUDA(cudaFuncSetAttribute(k_range_hist, cudaFuncAttributeMaxDynamicSharedMemorySize, 32768 * 4));
        attr_set[dev] = true;
      }
    }
    size_t bx = (used + 1023) / 1024;
    if (bx > 74) bx = 74;  // 2 halves x 74 = one CTA per SM
    k_range_hist<<<dim3((unsigned)bx, 2), 1024, 32768 * 4, s>>>(d_trace, freq, n_rows, used, l.rc_lo, l.rc_hi, d_err);
    g_pb_launches++;
    pb_check_last("range histogram");
  }
#endif
  if (used < n_rows) {
    // padding rows are all zero: (rc_hi - rc_lo) look-ups of the value 0 each
    u64 extra = (u64)(n_rows - used) * (u64)(l.rc_hi - l.rc_lo);
    pb_launch("pad frequency", AddK{freq, extra}, 1, s, 32);
  }
}

}  // namespace tg
