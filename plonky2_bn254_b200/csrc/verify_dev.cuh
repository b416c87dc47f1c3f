// K15 `verify_device`: the two heavy parts of verify::verify_walk on the context's GPU (pb254_verify_device).
//   1. native CTL  NativeCtlK, one thread per instance: canonical loads, the native output with the shared ladder
//                  (verify::native_output), then per challenge j the input and output tuple combinations in the host's
//                  Horner order (last tuple element first, then + gamma), a zero flag per (c, j) or the inverse.
//                  The lowest failing instance and its status go into one word with tg::set_lowest. SumInvK /
//                  SumPartK add the inverses per (c, j); Goldilocks addition is exact, so any order gives the host sum.
//   2. Merkle      MerkleCheckK, one thread per (query, tree): verify::merkle_path_ok with the device permutation. The
//                  walk has rejected every blob word >= p before this runs, as the lazy permutation requires.
// The host uploads the blob and the batch after the transcript and evaluates the quotient identity while these run;
// the walk then reads the results in its own order, so every outcome equals pb254_verify's.
#pragma once
#include "verify.cuh"

namespace verify_dev {

// where the leaf and the path of tree t sit in a query record, and its cap in the blob (words)
struct Tree {
  u32 leaf, leaf_len, path, depth, shift;  // the leaf index is the query index >> shift
  u64 cap;
};
static constexpr int STATUS_BITS = 3;  // bad = (k << STATUS_BITS) | verify::NATIVE_*
static constexpr unsigned NO_BAD = 0xffffffffu;
static constexpr int SUM_CHUNK = 256;

// a = a * beta^4 + (the four 16-bit limbs of w, most significant first)
PB_HD u64 horner_word(u64 a, u64 w, u64 beta) {
#pragma unroll
  for (int q = 3; q >= 0; q--) a = gl::add(gl::mul(a, beta), (w >> (16 * q)) & 0xffff);
  return a;
}

template <int KIND>
struct NativeCtlK {
  static constexpr int IN = KIND == 0 ? 20 : KIND == 1 ? 36 : 8, OUT = KIND == 0 ? 8 : KIND == 1 ? 16 : 4;
  const u64* inputs;  // [K][IN]
  const u64* ts;      // [K]
  const u64* chal;    // beta[nch], gamma[nch]
  u64* inv;           // [2 nch][K]: 1 / combination, 0 where it is zero or the instance failed
  int* zero;          // [2 nch]
  unsigned* bad;      // the lowest (k << STATUS_BITS) | status
  size_t K;
  int nch;
  PB_HD void operator()(size_t k) const {
    const u64* w = inputs + k * IN;
    u64 out[OUT];
    const int st = verify::native_output<KIND>(w, out);
    if (st) tg::set_lowest(bad, (unsigned)(k << STATUS_BITS) | (unsigned)st);
    const u64 t = ts[k] % gl::P;
#pragma unroll 1
    for (int j = 0; j < nch; j++) {
      const u64 beta = chal[j], gamma = chal[nch + j];
      u64 a = 0, b = 0;
      if (!st) {
        // inputs: limbs of words 4 .. IN (x, offset), then of words 0 .. 4 (s), then t
        a = t;
#pragma unroll 1
        for (int i = 3; i >= 0; i--) a = horner_word(a, w[i], beta);
#pragma unroll 1
        for (int i = IN - 1; i >= 4; i--) a = horner_word(a, w[i], beta);
        a = gl::add(a, gamma);
        // outputs: limbs of the native output's words, then t
        b = t;
#pragma unroll
        for (int i = OUT - 1; i >= 0; i--) b = horner_word(b, out[i], beta);
        b = gl::add(b, gamma);
      }
      for (int c = 0; c < 2; c++) {
        const u64 v = c ? b : a;
        const size_t cj = (size_t)c * nch + j;
        if (!st && v == 0) zero[cj] = 1;
        inv[cj * K + k] = v ? gl::inv(v) : 0;
      }
    }
  }
};

// part[cj][p] = sum of inv[cj][p * SUM_CHUNK ..][..SUM_CHUNK]
struct SumInvK {
  const u64* inv;
  u64* part;
  size_t K, nparts;
  PB_HD void operator()(size_t gid) const {
    const size_t cj = gid / nparts, p = gid % nparts, end = (p + 1) * SUM_CHUNK < K ? (p + 1) * SUM_CHUNK : K;
    u64 s = 0;
    for (size_t k = p * SUM_CHUNK; k < end; k++) s = gl::add(s, inv[cj * K + k]);
    part[gid] = s;
  }
};
struct SumPartK {
  const u64* part;
  u64* sum;  // [2 nch]
  size_t nparts;
  PB_HD void operator()(size_t cj) const {
    u64 s = 0;
    for (size_t p = 0; p < nparts; p++) s = gl::add(s, part[cj * nparts + p]);
    sum[cj] = s;
  }
};

struct MerkleCheckK {
  const u64* blob;
  const Tree* trees;  // [T]
  const u64* idx;     // [num_query_rounds]
  u64 queries, rec;   // first query record and record length (words)
  int T;
  int* ok;  // [q][T]
  PB_HD void operator()(size_t gid) const {
    const size_t q = gid / T;
    const Tree tr = trees[gid % T];
    const u64* rp = blob + queries + q * rec;
    ok[gid] = verify::merkle_path_ok(rp + tr.leaf, tr.leaf_len, (size_t)(idx[q] >> tr.shift), rp + tr.path,
                                     (int)tr.depth, blob + tr.cap);
  }
};

// verify::Checks on the context's GPU: start() uploads and launches, ctl() and the first merkle_ok() wait for their
// results. The destructor waits for whatever is still running (a walk that fails early leaves kernels in flight).
struct DeviceChecks : verify::Checks {
  pb254_ctx* c;
  int nch = 0, T = 0;
  size_t K = 0, nparts = 0, nq = 0;
  unsigned* d_bad = nullptr;
  int *d_zero = nullptr, *d_ok = nullptr;
  u64* d_sum = nullptr;
  std::vector<int> ok;
  bool have_ok = false;
  explicit DeviceChecks(pb254_ctx* ctx) : c(ctx) {}
  ~DeviceChecks() override {
#if !PB_HOSTSIM
    (void)cudaStreamSynchronize(c->stream);  // errors of the stream are reported by the next call on the context
#endif
    c->times.resolve();
  }

  void start(const verify::Job& j) override {
    const tg::Layout l = tg::layout_for(j.kind);
    const pb254_proof_layout& lay = *j.lay;
    const pbStream s = c->stream;
    nch = j.nch;
    K = j.K;
    nparts = (K + SUM_CHUNK - 1) / SUM_CHUNK;
    nq = j.idx->size();
    const size_t ncj = 2 * (size_t)nch;
    T = 3 + (int)j.arities->size();
    // the trees of one query record (proofview.cuh)
    std::vector<Tree> trees(T);
    const u32 d0 = (u32)(j.logN - j.cap_h);
    trees[0] = Tree{lay.q_trace_leaf, lay.trace_width, lay.q_trace_path, d0, 0, lay.trace_cap};
    trees[1] = Tree{lay.q_aux_leaf, lay.aux_width, lay.q_aux_path, d0, 0, lay.auxiliary_polys_cap};
    trees[2] = Tree{lay.q_quotient_leaf, lay.quotient_width, lay.q_quotient_path, d0, 0, lay.quotient_polys_cap};
    u32 shift = 0;
    for (size_t i = 0; i < j.arities->size(); i++) {
      shift += (*j.arities)[i];
      trees[3 + i] = Tree{lay.q_step_evals[i], lay.q_step_evals_words[i], lay.q_step_path[i],
                          lay.q_step_path_words[i] / 4, shift, lay.commit_phase_merkle_caps + i * lay.cap_words};
    }
    std::vector<u64> chal(ncj);
    for (int i = 0; i < nch; i++) {
      chal[i] = j.chal->beta[i];
      chal[nch + i] = j.chal->gamma[i];
    }

    c->arena.reserve((j.words + K * l.in_words + K + ncj * (K + nparts + 2) + nq) * 8 + T * sizeof(Tree) +
                     nq * T * sizeof(int) + 16 * 256 + 65536);
    c->arena.reset();
    u64* d_blob = c->arena.alloc_n<u64>(j.words);
    u64* d_in = c->arena.alloc_n<u64>(K * l.in_words + 1);
    u64* d_ts = c->arena.alloc_n<u64>(K + 1);
    u64* d_chal = c->arena.alloc_n<u64>(ncj);
    u64* d_inv = c->arena.alloc_n<u64>(ncj * K + 1);
    u64* d_part = c->arena.alloc_n<u64>(ncj * nparts + 1);
    d_sum = c->arena.alloc_n<u64>(ncj);
    d_zero = c->arena.alloc_n<int>(ncj);
    d_bad = c->arena.alloc_n<unsigned>(1);
    u64* d_idx = c->arena.alloc_n<u64>(nq);
    Tree* d_trees = c->arena.alloc_n<Tree>(T);
    d_ok = c->arena.alloc_n<int>(nq * T);
    pb_h2d(d_blob, j.blob, j.words * 8, s);
    if (K) {
      pb_h2d(d_in, j.inputs, K * l.in_words * 8, s);
      pb_h2d(d_ts, j.timestamps, K * 8, s);
    }
    pb_h2d(d_chal, chal.data(), ncj * 8, s);
    pb_h2d(d_idx, j.idx->data(), nq * 8, s);
    pb_h2d(d_trees, trees.data(), T * sizeof(Tree), s);
    pb_memset(d_zero, 0, ncj * sizeof(int), s);
    pb_memset(d_bad, 0xff, sizeof(unsigned), s);

    int t = c->times.begin("verify native ctl", s);
    if (j.kind == 0)
      pb_launch("verify native ctl", NativeCtlK<0>{d_in, d_ts, d_chal, d_inv, d_zero, d_bad, K, nch}, K, s, 32);
    else if (j.kind == 1)
      pb_launch("verify native ctl", NativeCtlK<1>{d_in, d_ts, d_chal, d_inv, d_zero, d_bad, K, nch}, K, s, 32);
    else
      pb_launch("verify native ctl", NativeCtlK<2>{d_in, d_ts, d_chal, d_inv, d_zero, d_bad, K, nch}, K, s, 32);
    pb_launch("verify ctl sums", SumInvK{d_inv, d_part, K, nparts}, ncj * nparts, s, 128);
    pb_launch("verify ctl total", SumPartK{d_part, d_sum, nparts}, ncj, s, 32);
    c->times.end(t, s);
    t = c->times.begin("verify merkle", s);
    pb_launch("verify merkle", MerkleCheckK{d_blob, d_trees, d_idx, lay.query_round_proofs, lay.query_words, T, d_ok},
              nq * T, s, 32);
    c->times.end(t, s);
  }

  void ctl(verify::CtlResults& o) override {
    const size_t ncj = 2 * (size_t)nch;
    unsigned bad = 0;
    std::vector<int> zero(ncj);
    o.sum.assign(ncj, 0);
    pb_d2h(&bad, d_bad, sizeof bad, c->stream);
    pb_d2h(zero.data(), d_zero, ncj * sizeof(int), c->stream);
    pb_d2h(o.sum.data(), d_sum, ncj * 8, c->stream);
    pb_sync(c->stream);
    if (bad != NO_BAD) {
      const Pb254Error e = verify::native_error((int)(bad & ((1u << STATUS_BITS) - 1)));
      o.code = e.code;
      o.msg = e.what();
      return;
    }
    o.zero.assign(zero.begin(), zero.end());
  }

  bool merkle_ok(size_t q, int tree, const u64*, size_t, size_t, const u64*, int, const u64*) override {
    if (!have_ok) {
      ok.resize(nq * T);
      pb_d2h(ok.data(), d_ok, ok.size() * sizeof(int), c->stream);
      pb_sync(c->stream);
      have_ok = true;
    }
    return ok[q * T + tree] != 0;
  }
};

}  // namespace verify_dev
