// K13 `scalar_mul_chains`: the chained scalar multiplications of G1SingleGenerator / G2SingleGenerator
// (src/generators/g1/single.rs:48-52) and g1_msm (src/utils/g1_msm.rs:22-36), batched on the device.
//
// Terms (s_i, x_i) come in consecutive chains c = [starts[c], starts[c+1]) with one affine offset each. For a chain,
// acc = offset, then for each of its terms: row i = (s_i, x_i, acc), acc = s_i x_i + acc; sums[c] = acc. All products
// P_i = s_i x_i are independent, and the accumulators are an inclusive segmented prefix sum in the curve group over
// n_terms + n_chains elements: chain c's offset (a segment head) at position starts[c] + c, followed by its P_i, so
// that term i sits at e = i + c + 1 and its row takes acc_i from e - 1.
//   1. products  one thread per term: the doublings D_j = 2^j x (the only sequential part, 256 steps); then one warp
//                per term sums the D_j of the set bits of s, 8 per lane, and a 5-level tree adds the lanes;
//                a thread per chain writes the heads
//   2. scan      block-level Hillis-Steele scan in shared memory with complete additions and segment-head flags,
//                applied recursively to the block aggregates, whose scan is then added back into every element that
//                has no head before it in its block
//   3. affine    k_to_affine (Montgomery-trick batch inversion), then canonical words into the wire rows and sums
// Affine coordinates are unique, so every output equals the serial reference walk. An accumulator at infinity
// (s_i x_i = -acc_i) is an error, as in the reference (g1_msm.rs:20-21); the lowest such element is reported.
#pragma once
#include "curve_io.cuh"

namespace chains {

using tg::FieldIO;

static constexpr size_t MAX_TERMS = (size_t)1 << 17;  // the largest batch one proof holds: 2^26 rows / 512
static constexpr size_t MAX_CHAINS = (size_t)1 << 17;
static constexpr unsigned NO_INF = 0xffffffffu;

template <class F>
struct Bufs {
  const u64* terms;    // [n_terms][4 + 2 FW]: s, x
  const u64* starts;   // [n_chains + 1]
  const u64* offsets;  // [n_chains][2 FW]
  bn::Jac<F>* D;       // [256][n_terms]: 2^j x_i, written only where bit j of s_i is set
  bn::Jac<F>* E;       // [n_elems]: scan elements, then the inclusive segmented scan
  int* head;           // [n_elems]: segment-head flags, then (per scan block) "a head at or before this element"
  bn::Aff<F>* A;       // [n_elems]: affine scan
  int* err;            // tg::ERR_* (maximum wins)
  unsigned* first_inf; // lowest element at infinity, NO_INF if none
  size_t n_terms, n_chains;
};

// the chain of term i: the largest c with starts[c] <= i (empty chains share their start with the next one)
PB_HD size_t chain_of_term(const u64* starts, size_t n_chains, size_t i) {
  size_t lo = 0, hi = n_chains;  // starts[lo] <= i < starts[hi]
  while (hi - lo > 1) {
    const size_t mid = (lo + hi) / 2;
    if (starts[mid] <= i) lo = mid; else hi = mid;
  }
  return lo;
}

template <class F>
PB_HD bn::Jac<F> infinity() {
  bn::Jac<F> p;
  p.X = F::one();
  p.Y = F::one();
  p.Z = F::zero();
  return p;
}

// load and check the affine point at w (2 FW words); false after flagging the error word
template <class F>
PB_HD bool load_point(const u64* w, bn::Aff<F>& p, int* err) {
  const int FW = FieldIO<F>::WORDS;
  if (!(FieldIO<F>::load(w, p.x) & FieldIO<F>::load(w + FW, p.y))) {
    tg::set_err(err, tg::ERR_NOT_CANONICAL);
    return false;
  }
  // the scan re-associates the additions: only valid in the curve group
  if (!FieldIO<F>::on_curve(p)) {
    tg::set_err(err, tg::ERR_NOT_ON_CURVE);
    return false;
  }
  return true;
}

PB_HD void put_fq(u64* w, const bn::Fq& mont) {
  const bn::Fq r = bn::from_mont(mont);
#pragma unroll
  for (int k = 0; k < 4; k++) w[k] = (u64)r.l[2 * k] | ((u64)r.l[2 * k + 1] << 32);
}
PB_HD void put_coord(u64* w, const bn::Fq& v) { put_fq(w, v); }
PB_HD void put_coord(u64* w, const bn::Fq2& v) {
  put_fq(w, v.c0);
  put_fq(w + 4, v.c1);
}

// 1a. the doubling chain of term i
template <class F>
struct DblK {
  Bufs<F> B;
  PB_HD void operator()(size_t i) const {
    const int FW = FieldIO<F>::WORDS;
    const u64* w = B.terms + i * (4 + 2 * FW);
    bn::Aff<F> x;
    if (!load_point<F>(w + 4, x, B.err)) x.x = x.y = F::one();  // keep the later kernels well defined
    bn::Jac<F> p;
    p.X = x.x;
    p.Y = x.y;
    p.Z = F::one();
    for (int j = 0; j < 256; j++) {
      if (tg::scalar_bit(w, j)) B.D[(size_t)j * B.n_terms + i] = p;
      if (j < 255) p = bn::jac_double<F>(p);  // a point of order two doubles to Z = 0, which the additions handle
    }
  }
};

// 1c. segment heads: chain c's offset at e = starts[c] + c
template <class F>
struct HeadsK {
  Bufs<F> B;
  PB_HD void operator()(size_t c) const {
    const size_t e = B.starts[c] + c;
    bn::Aff<F> off;
    if (!load_point<F>(B.offsets + c * 2 * FieldIO<F>::WORDS, off, B.err)) off.x = off.y = F::one();
    B.E[e].X = off.x;
    B.E[e].Y = off.y;
    B.E[e].Z = F::one();
    B.head[e] = 1;
  }
};

// 2b. the lowest accumulator at infinity (heads are offsets, never at infinity)
template <class F>
struct FindInfK {
  Bufs<F> B;
  PB_HD void operator()(size_t e) const {
    if (F::is_zero(B.E[e].Z)) tg::set_lowest(B.first_inf, (unsigned)e);
  }
};

// 3b. wire row i = (s_i, x_i, acc_i), acc_i = A[i + c]
template <class F>
struct RowsK {
  Bufs<F> B;
  u64* rows;  // [n_terms][4 + 4 FW]
  PB_HD void operator()(size_t i) const {
    const int FW = FieldIO<F>::WORDS, TW = 4 + 2 * FW;
    const size_t c = chain_of_term(B.starts, B.n_chains, i);
    u64* o = rows + i * (TW + 2 * FW);
    for (int k = 0; k < TW; k++) o[k] = B.terms[i * TW + k];
    const bn::Aff<F> a = B.A[i + c];
    put_coord(o + TW, a.x);
    put_coord(o + TW + FW, a.y);
  }
};
// 3c. sums[c] = the last element of chain c's segment
template <class F>
struct SumsK {
  Bufs<F> B;
  u64* sums;  // [n_chains][2 FW]
  PB_HD void operator()(size_t c) const {
    const int FW = FieldIO<F>::WORDS;
    const bn::Aff<F> a = B.A[B.starts[c + 1] + c];
    put_coord(sums + c * 2 * FW, a.x);
    put_coord(sums + c * 2 * FW + FW, a.y);
  }
};

#if PB_HOSTSIM
// ---- the same stages, one work item per thread, for the host-simulation build ---------------------------------
template <class F>
struct SumK {  // P_i into its element
  Bufs<F> B;
  PB_HD void operator()(size_t i) const {
    const u64* w = B.terms + i * (4 + 2 * FieldIO<F>::WORDS);
    bn::Jac<F> acc = infinity<F>();
    for (int j = 0; j < 256; j++)
      if (tg::scalar_bit(w, j)) acc = bn::jac_add_complete<F>(acc, B.D[(size_t)j * B.n_terms + i]);
    const size_t e = i + chain_of_term(B.starts, B.n_chains, i) + 1;
    B.E[e] = acc;
    B.head[e] = 0;
  }
};
template <class F>
struct ScanK {  // one chain, serially
  Bufs<F> B;
  PB_HD void operator()(size_t c) const {
    const size_t e0 = B.starts[c] + c, e1 = B.starts[c + 1] + c;
    for (size_t e = e0 + 1; e <= e1; e++) B.E[e] = bn::jac_add_complete<F>(B.E[e - 1], B.E[e]);
  }
};
template <class F>
struct AffK {
  const bn::Jac<F>* src;
  bn::Aff<F>* dst;
  int* err;
  PB_HD void operator()(size_t e) const {
    const bn::Jac<F> p = src[e];
    if (F::is_zero(p.Z)) {
      tg::set_err(err, tg::ERR_INFINITY);
      dst[e].x = dst[e].y = F::zero();
      return;
    }
    const typename F::T zi = F::inv(p.Z), zi2 = F::sqr(zi);
    dst[e].x = F::mul(p.X, zi2);
    dst[e].y = F::mul(p.Y, F::mul(zi, zi2));
  }
};
#else
// ---- device-only block code -------------------------------------------------------------------------------------
// The sum over the set bits of a 256-bit scalar w of the table points D[j * stride], one warp per scalar: lane l adds
// the entries of bits 8l .. 8l+7, then a 5-level tree adds the lanes; the sum is left in p[0]. The partial sums live
// in shared memory (p: 32 entries of this warp), so that an addition's operands are loaded as it needs them (F2: no
// spills at 255 registers).
template <class F>
__device__ __forceinline__ void warp_bit_sum(bn::Jac<F>* p, const u64* w, const bn::Jac<F>* D, size_t stride) {
  const int lane = threadIdx.x & 31;
  const u32 bits = (u32)(w[lane >> 3] >> ((lane & 7) * 8)) & 0xffu;
  p[lane] = infinity<F>();
#pragma unroll 1
  for (int t = 0; t < 8; t++)
    if ((bits >> t) & 1) p[lane] = bn::jac_add_complete<F>(p[lane], D[(size_t)(8 * lane + t) * stride]);
  __syncwarp();
#pragma unroll 1
  for (int d = 16; d >= 1; d >>= 1) {
    if (lane < d) p[lane] = bn::jac_add_complete<F>(p[lane], p[lane + d]);
    __syncwarp();
  }
}

// 1b. one warp per term: s_i x_i from the doublings D_j = 2^j x_i of the set bits of s_i
static constexpr int SUM_WARPS = 4;
template <class F>
__global__ void __launch_bounds__(32 * SUM_WARPS) k_chain_sum(Bufs<F> B) {
  __shared__ bn::Jac<F> part[SUM_WARPS][32];
  const size_t i = (size_t)blockIdx.x * SUM_WARPS + (threadIdx.x >> 5);
  if (i >= B.n_terms) return;  // whole warps
  bn::Jac<F>* p = part[threadIdx.x >> 5];
  warp_bit_sum<F>(p, B.terms + i * (4 + 2 * FieldIO<F>::WORDS), B.D + i, B.n_terms);
  if ((threadIdx.x & 31) == 0) {
    const size_t e = i + chain_of_term(B.starts, B.n_chains, i) + 1;
    B.E[e] = p[0];
    B.head[e] = 0;
  }
}

// 2a. inclusive segmented scan of v[0..n) within blocks of SCAN_B: (head_a, a) . (head_b, b) = (head_a | head_b,
// head_b ? b : a + b). head[e] becomes "a head at or before e in its block"; the block's total goes to agg / agg_head.
static constexpr int SCAN_B = 128;
template <class F>
__global__ void __launch_bounds__(SCAN_B, 1) k_seg_scan_block(bn::Jac<F>* __restrict__ v, int* __restrict__ head, size_t n,
                                                           bn::Jac<F>* __restrict__ agg, int* __restrict__ agg_head) {
  __shared__ bn::Jac<F> sv[SCAN_B];
  __shared__ int sh[SCAN_B];
  const int t = threadIdx.x;
  const size_t e = (size_t)blockIdx.x * SCAN_B + t;
  bn::Jac<F> x = e < n ? v[e] : infinity<F>();
  int h = e < n ? head[e] : 0;
#pragma unroll 1
  for (int d = 1; d < SCAN_B; d <<= 1) {
    sv[t] = x;
    sh[t] = h;
    __syncthreads();
    if (t >= d && !h) {
      x = bn::jac_add_complete<F>(sv[t - d], x);
      h = sh[t - d];
    }
    __syncthreads();
  }
  if (e < n) {
    v[e] = x;
    head[e] = h;
  }
  if (t == SCAN_B - 1 && agg) {
    agg[blockIdx.x] = x;
    agg_head[blockIdx.x] = h;
  }
}
// 2c. element e of block b > 0 without a head before it in its block continues the scan of blocks 0 .. b-1
template <class F>
__global__ void __launch_bounds__(128) k_seg_scan_fix(bn::Jac<F>* __restrict__ v, const int* __restrict__ head, size_t n,
                                                      const bn::Jac<F>* __restrict__ agg_scan) {
  const size_t e = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= n || e < (size_t)SCAN_B || head[e]) return;
  v[e] = bn::jac_add_complete<F>(agg_scan[e / SCAN_B - 1], v[e]);
}

template <class F>
void seg_scan(Arena& ar, bn::Jac<F>* v, int* head, size_t n, pbStream s) {
  const size_t nb = (n + SCAN_B - 1) / SCAN_B;
  bn::Jac<F>* agg = nb > 1 ? ar.alloc_n<bn::Jac<F>>(nb) : nullptr;
  int* agg_head = nb > 1 ? ar.alloc_n<int>(nb) : nullptr;
  k_seg_scan_block<F><<<(unsigned)nb, SCAN_B, 0, s>>>(v, head, n, agg, agg_head);
  g_pb_launches++;
  pb_check_last("chains scan block");
  if (nb > 1) {
    seg_scan<F>(ar, agg, agg_head, nb, s);
    k_seg_scan_fix<F><<<(unsigned)((n + 127) / 128), 128, 0, s>>>(v, head, n, agg);
    g_pb_launches++;
    pb_check_last("chains scan fix");
  }
}
#endif

// dst[e] = affine(src[e]), e < n; a point at infinity flags tg::ERR_INFINITY
template <class F>
void to_affine(const bn::Jac<F>* src, bn::Aff<F>* dst, size_t n, int* err, pbStream s) {
#if PB_HOSTSIM
  pb_launch("to affine", AffK<F>{src, dst, err}, n, s);
#else
  const size_t threads = (n + tg::AFF_CH - 1) / tg::AFF_CH;
  if (!threads) return;
  tg::k_to_affine<F><<<(unsigned)((threads + 127) / 128), 128, 0, s>>>(src, dst, n, 0, err);
  g_pb_launches++;
  pb_check_last("to affine");
#endif
}

// scratch bytes for n_terms / n_chains (the scan's aggregate levels included)
template <class F>
size_t scratch_bytes(size_t n_terms, size_t n_chains) {
  const size_t n = n_terms + n_chains, jac = sizeof(bn::Jac<F>), aff = sizeof(bn::Aff<F>);
  return 256 * n_terms * jac + n * (2 * jac + aff + 2 * sizeof(int)) + 64 * 256;
}

// Runs the three stages on device buffers. Errors land in *B.err / *B.first_inf.
template <class F>
void run(pb254_ctx* c, Bufs<F> B, u64* d_rows, u64* d_sums) {
  const pbStream s = c->stream;
  const size_t n = B.n_terms + B.n_chains;
  int t0 = c->times.begin("chains products", s);
  pb_launch("chains doublings", DblK<F>{B}, B.n_terms, s, 32);
#if PB_HOSTSIM
  pb_launch("chains sums", SumK<F>{B}, B.n_terms, s);
#else
  if (B.n_terms) {
    k_chain_sum<F><<<(unsigned)((B.n_terms + SUM_WARPS - 1) / SUM_WARPS), 32 * SUM_WARPS, 0, s>>>(B);
    g_pb_launches++;
    pb_check_last("chains sums");
  }
#endif
  pb_launch("chains heads", HeadsK<F>{B}, B.n_chains, s, 128);
  c->times.end(t0, s);
  int t1 = c->times.begin("chains scan", s);
#if PB_HOSTSIM
  pb_launch("chains scan", ScanK<F>{B}, B.n_chains, s);
#else
  seg_scan<F>(c->arena, B.E, B.head, n, s);
#endif
  pb_launch("chains infinity", FindInfK<F>{B}, n, s, 128);
  c->times.end(t1, s);
  int t2 = c->times.begin("chains affine", s);
  to_affine<F>(B.E, B.A, n, B.err, s);
  pb_launch("chains rows", RowsK<F>{B, d_rows}, B.n_terms, s, 128);
  if (d_sums) pb_launch("chains sums out", SumsK<F>{B, d_sums}, B.n_chains, s, 128);
  c->times.end(t2, s);
}

}  // namespace chains
