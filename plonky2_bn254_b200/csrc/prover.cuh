// Host orchestration of one STARK proof on one GPU. Mirrors, step for step,
//   prove()                  src/starks/common/prover.rs:18-72
//   prove_with_commitment()  starky 0.4.0 prover.rs        (un-vendored dependency)
//   PolynomialBatch::prove_openings / fri_proof           plonky2 0.2.2 fri/{oracle,prover}.rs
// The Fiat-Shamir transcript (Challenger, plonky2 0.2.2 iop/challenger.rs) stays on the host: it is
// a strictly sequential chain of ~10^3 Poseidon permutations over caps and openings that have to
// cross to the host for the proof anyway (SURVEY.md 2.3). Everything that touches trace-sized data
// runs in CUDA kernels on the context's stream.
#pragma once
#include "../../include/pb254.h"
#include "context.cuh"
#include "ntt.cuh"
#include "merkle.cuh"
#include "tracegen.h"
#include "aux.cuh"
#include "quotient.h"
#include "fri.cuh"
#include "proofview.cuh"
#include <vector>

namespace prover {

using gl::E2;
using merkle::Digest;

// ---- host transcript ---------------------------------------------------------------------------
struct Challenger {
  u64 state[12];
  std::vector<u64> in, out;
  Challenger() { memset(state, 0, sizeof state); }
  void duplex() {
    for (size_t i = 0; i < in.size(); i++) state[i] = in[i];
    in.clear();
    poseidon::permute(state);
    out.assign(state, state + 8);
  }
  void observe(u64 x) {
    out.clear();
    in.push_back(x);
    if (in.size() == 8) duplex();
  }
  void observe_n(const u64* x, size_t n) {
    for (size_t i = 0; i < n; i++) observe(x[i]);
  }
  u64 challenge() {
    if (!in.empty() || out.empty()) duplex();
    u64 r = out.back();
    out.pop_back();
    return r;
  }
  E2 ext_challenge() {
    u64 a = challenge();
    u64 b = challenge();
    return gl::e2(a, b);
  }
  void compact(u64 dst[12]) {
    if (!in.empty()) duplex();
    out.clear();
    memcpy(dst, state, sizeof state);
  }
};

using proofview::fri_arities;
static const u64 PROOF_MAGIC = proofview::MAGIC;

struct ProofData {
  std::vector<u64> blob;
  std::vector<u64> dbg_aux, dbg_chunks, dbg_challenges, dbg_indices, dbg_groups;
};

static inline void validate_config(const pb254_config& c) {
  if (c.rate_bits < 1 || c.rate_bits > 3) throw Pb254Error(PB254_E_BAD_ARG, "rate_bits must be in 1..3");
  if (c.num_challenges < 1 || c.num_challenges > (unsigned)aux::MAXCH)
    throw Pb254Error(PB254_E_BAD_ARG, "num_challenges must be in 1..4");
  if (c.arity_bits < 1 || c.arity_bits > 4) throw Pb254Error(PB254_E_BAD_ARG, "arity_bits must be in 1..4");
  if (c.pow_bits > 40) throw Pb254Error(PB254_E_BAD_ARG, "pow_bits too large");
  if (c.num_query_rounds < 1 || c.num_query_rounds > 1024) throw Pb254Error(PB254_E_BAD_ARG, "num_query_rounds");
  if (c.cap_height > 16) throw Pb254Error(PB254_E_BAD_ARG, "cap_height must be <= 16");
  if (c.final_poly_bits > 16) throw Pb254Error(PB254_E_BAD_ARG, "final_poly_bits must be <= 16");
}

// device bytes needed by prove_device for an (kind, n, cfg) proof, excluding the trace values
static inline size_t workspace_bytes(int kind, size_t n, const pb254_config& cfg) {
  tg::Layout l = tg::layout_for(kind);
  size_t nch = cfg.num_challenges, W = l.width, A = aux::num_aux(l, (int)nch), Q = 2 * nch;
  size_t N = n << cfg.rate_bits;
  size_t words = (W + A + Q) * N            // LDEs
                 + (A + (W > A ? W : A)) * n  // aux values + NTT scratch
                 + 4 * nch * n * 2          // quotient values + coefficients
                 + 2 * nch * n + (nch << 16) + 4 * nch * (n / 256 + 16)  // aux build scratch
                 + 2 * n                    // barycentric weights
                 + (W > A ? W : A) * fri::PARTS * 4 + 4 * (W + A + Q) + 2 * (W + A + Q)
                 + 3 * N                    // FRI layer values (geometric series < 2.2 N words ext)
                 + 4 * (3 * 2 * N + 2 * N);  // digests: 3 initial trees + FRI layer trees
  return words * 8 + (size_t)quot::num_constraints(kind, (int)nch) * nch * 8 + (1u << 22);
}

// the same when the proof is spread over `world` ranks (prove_device with a communicator): row blocks instead of whole
// LDEs, plus the column-shard LDE, the exchange buffers and the gathered digests
static inline size_t workspace_bytes_sharded(int kind, size_t n, const pb254_config& cfg, size_t world) {
  tg::Layout l = tg::layout_for(kind);
  size_t nch = cfg.num_challenges, W = l.width, A = aux::num_aux(l, (int)nch), Q = 2 * nch;
  size_t N = n << cfg.rate_bits, halo = (size_t)1 << cfg.rate_bits, Nloc = N / world;
  size_t WA = W > A ? W : A, cper = (WA + world - 1) / world, Cpad = cper * world;
  size_t words = (W + A + 2 * world) * (Nloc + halo) + Q * N    // row blocks, quotient LDE
                 + cper * n + A * n                             // NTT scratch, aux values
                 + cper * N + Cpad * (Nloc + halo)                 // column-shard LDE, send buffer
                 + 3 * cper * n                                    // value column shards (trace, aux) + their exchange
                 + 4 * (Nloc + N)                               // digests of the own rows, of all rows
                 + 4 * nch * n * 2 + 2 * nch * n + (nch << 16) + 4 * nch * (n / 256 + 16) + 2 * n
                 + WA * fri::PARTS * 4 + 6 * (W + A + Q) + 3 * N + 2 * Nloc + 2 * N
                 + 4 * (3 * 2 * N + 2 * N);
  return words * 8 + (size_t)quot::num_constraints(kind, (int)nch) * nch * 8 + (1u << 22);
}

// out[i] = sum over `parts` records of in[p * words + i] (u64 wrap-around; exactly one rank holds a non-zero value)
struct SumRecordsK {
  const u64* in;
  u64* out;
  size_t words;
  int parts;
  PB_HD void operator()(size_t i) const {
    u64 v = 0;
    for (int p = 0; p < parts; p++) v += in[(size_t)p * words + i];
    out[i] = v;
  }
};

struct Stage {
  pb254_ctx* c;
  int id;
  Stage(pb254_ctx* c_, const char* name) : c(c_), id(c_->times.begin(name, c_->stream)) {}
  // a destructor must not throw (a sticky CUDA error, or unwinding from another throw): the failure is recorded
  // and surfaces at the next synchronisation of the stream
  ~Stage() { c->times.end_nothrow(id, c->stream); }
};

// d_trace: W x n column-major device matrix (trace values on H). Fills out.blob.
// comm != nullptr with world > 1: ONE proof across the ranks of `comm` (SURVEY.md 8e, include/pb254.h
// pb254_prove_sharded); every rank holds the whole trace, runs the same transcript and produces the same proof,
// the commitments, the quotient evaluation, the FRI combination and the query openings are sharded.
// trace_is_block (sharded only): d_trace is not the whole trace but this rank's row block [rank n / P, (rank + 1) n / P)
// of it, column-major [ceil(W / P) P columns][n / P] (instance-sharded trace generation, pb254.cu); the column shards
// the LDE and the openings need are then produced by one more all-to-all of VALUES, and the auxiliary columns are
// built per row block with the running sums carried across the ranks.
static inline void prove_device(pb254_ctx* c, int kind, const u64* d_trace, size_t n, const pb254_config& cfg,
                                ProofData& out, bool keep_debug, const pb254_comm* comm = nullptr,
                                bool trace_is_block = false) {
  validate_config(cfg);
  pbStream s = c->stream;
  Arena& ar = c->arena;
  const tg::Layout l = tg::layout_for(kind);
  const int nch = (int)cfg.num_challenges, W = l.width, NH = aux::num_helpers(l), A = aux::num_aux(l, nch),
            Q = 2 * nch, nlk = (NH + 1) * nch;
  int L = 0;
  while (((size_t)1 << L) < n) L++;
  if (((size_t)1 << L) != n || L < 8) throw Pb254Error(PB254_E_BAD_ARG, "trace height must be a power of two >= 256");
  const int r = (int)cfg.rate_bits, logN = L + r, cap_h = (int)cfg.cap_height;
  const size_t N = n << r, ncap = (size_t)1 << cap_h;
  if (cap_h > logN) throw Pb254Error(PB254_E_BAD_ARG, "cap_height too large");
  std::vector<unsigned> arities = fri_arities(cfg, (unsigned)L);
  const size_t WA = W > A ? W : A;
  const bool sharded = comm && comm->world > 1;
  const size_t P = sharded ? comm->world : 1, rk = sharded ? comm->rank : 0;
  const size_t Nloc = N / P, halo = (size_t)1 << r;  // LDE rows per rank; the next trace row is 2^r LDE rows further
  if (sharded && (Nloc < 256 || keep_debug))
    throw Pb254Error(PB254_E_BAD_ARG, "comm: too many ranks for this trace (or keep_debug set)");
  auto coll = [&](int rc, const char* what) {
    if (rc) throw Pb254Error(PB254_E_CUDA, std::string("collective failed: ") + what);
  };
  struct RowBlock {
    const u64* ptr;
    size_t stride;
  };
  const size_t nloc = n / P;  // trace rows per rank
  auto first_col = [&](int C) { return std::min((size_t)C, rk * (((size_t)C + P - 1) / P)); };
  // Row blocks of VALUES [ceil(C / P) P][nloc] -> this rank's column shard [ceil(C / P)][n]: chunk q of the all-to-all
  // is the contiguous slab of rank q's columns, the received slabs are laid side by side along the rows.
  auto to_column_shard = [&](const u64* rows, int C, const char* tag) -> const u64* {
    const size_t cper = ((size_t)C + P - 1) / P;
    u64* shard = ar.alloc_n<u64>(cper * n);
    const size_t mark = ar.off;
    Stage st(c, (std::string("values exchange ") + tag).c_str());
    u64* recv = ar.alloc_n<u64>(cper * n);
    coll(comm->all_to_all(comm->user, rows, recv, cper * nloc * 8), "all_to_all (values)");
    for (size_t p = 0; p < P; p++) pb_copy2d(shard + p * nloc, n * 8, recv + p * cper * nloc, nloc * 8, nloc * 8, cper, s);
    ar.off = mark;
    return shard;
  };
  // Inner levels of a tree whose leaf level is complete on every rank: rank q hashes the nodes [q m / P, (q + 1) m / P)
  // of a level (a contiguous node range at every level is one subtree) and the level is all-gathered, instead of
  // every rank hashing all of it; the top levels (fewer than 256 nodes per rank) are computed by everyone.
  // part: scratch for N / (2 P) digests.
  auto levels_sharded = [&](Digest* dig, Digest* part) {
    size_t off = 0;
    for (int lv = 0; lv < logN - cap_h; lv++) {
      const size_t m = (size_t)1 << (logN - lv), half = m / 2, per = half / P;
      Digest* child = dig + off;
      Digest* parent = dig + off + m;
      if (per >= 256) {
        merkle::launch_level(child + 2 * rk * per, part, per, s);
        coll(comm->all_gather(comm->user, part, parent, per * sizeof(Digest)), "all_gather (tree level)");
      } else {
        merkle::launch_level(child, parent, half, s);
      }
      off += m;
    }
  };
  // PolynomialBatch::from_values of one matrix across the ranks: LDE of this rank's column shard, one all-to-all into
  // row blocks (plus the next-row halo), leaf hashing of the own rows, all-gather of the digests, inner levels.
  // Returns this rank's rows [rk Nloc, (rk + 1) Nloc + halo) of all C columns; dig receives the whole tree.
  // shard: the values of this rank's columns [c0, c1), [nc][n].
  auto commit_sharded = [&](const u64* shard, int C, Digest* dig, u64* scratch_, const char* tag) -> RowBlock {
    const size_t cper = ((size_t)C + P - 1) / P, Cpad = cper * P;
    const size_t c0 = std::min((size_t)C, rk * cper), c1 = std::min((size_t)C, c0 + cper), nc = c1 - c0;
    const size_t stride = Nloc + halo;
    u64* rows = ar.alloc_n<u64>(Cpad * stride);
    const size_t mark = ar.off;
    u64* col_lde = ar.alloc_n<u64>(cper * N);
    u64* send = ar.alloc_n<u64>(P * cper * stride);
    const std::string t = tag;
    // Chunk q of the exchange: rows [q Nloc, (q + 1) Nloc + halo) (mod N) of this rank's columns, so that the
    // receiver's buffer IS its row block with the next-row halo: [source rank][column][Nloc + halo] = [Cpad][stride].
    // The last NTT pass writes this layout itself (ntt::RowBlocks); only transforms too small for a strided last pass
    // are repacked by copies.
    bool packed = false;
    {
      Stage st(c, ("lde " + t).c_str());
      int log_nloc = 0;
      while (((size_t)1 << log_nloc) < Nloc) log_nloc++;
      const ntt::RowBlocks rb = {send, log_nloc, (unsigned)P, stride, cper * stride, halo};
      if (nc)
        packed = ntt::lde_columns_row_blocks(c->tables, shard, n, col_lde, N, scratch_, (int)nc, L, r, ntt::FROM_VALUES_LDE, rb, s);
    }
    {
      Stage st(c, ("exchange " + t).c_str());
      if (nc && !packed)
        for (size_t q = 0; q < P; q++) {
          u64* dst = send + q * cper * stride;
          if (q + 1 < P) {
            pb_copy2d(dst, stride * 8, col_lde + q * Nloc, N * 8, stride * 8, cper, s);
          } else {  // the halo of the last block wraps around to row 0
            pb_copy2d(dst, stride * 8, col_lde + q * Nloc, N * 8, Nloc * 8, cper, s);
            pb_copy2d(dst + Nloc, stride * 8, col_lde, N * 8, halo * 8, cper, s);
          }
        }
      coll(comm->all_to_all(comm->user, send, rows, cper * stride * 8), "all_to_all");
    }
    {
      Stage st(c, ("merkle " + t).c_str());
      Digest* mine = ar.alloc_n<Digest>(Nloc);
      Digest* all = ar.alloc_n<Digest>(N);
      merkle::hash_rows_natural(rows, stride, C, Nloc, mine, s);
      coll(comm->all_gather(comm->user, mine, all, Nloc * sizeof(Digest)), "all_gather (digests)");
      pb_launch("leaves in tree order", merkle::SubtreeLeavesK{all, dig, 0, logN}, N, s, 128);
      levels_sharded(dig, mine);
    }
    ar.off = mark;  // the temporaries are dead in stream order
    return RowBlock{rows, stride};
  };

  std::vector<u64>& blob = out.blob;
  blob.clear();
  blob.push_back(PROOF_MAGIC);
  blob.push_back((u64)kind);
  blob.push_back((u64)L);
  blob.push_back(cfg.rate_bits);
  blob.push_back(cfg.cap_height);
  blob.push_back(cfg.num_challenges);
  blob.push_back(cfg.num_query_rounds);
  blob.push_back(cfg.pow_bits);
  blob.push_back(cfg.arity_bits);
  blob.push_back(cfg.final_poly_bits);
  const size_t pos_state = blob.size();
  blob.resize(blob.size() + 12);

  // ---- trace commitment (common/prover.rs:31-44) ----------------------------------------------
  u64* scratch = ar.alloc_n<u64>((sharded ? std::max((WA + P - 1) / P, (size_t)Q) : WA) * n);
  const size_t nd = merkle::tree_digests(logN, cap_h);
  Digest* dig_tr = ar.alloc_n<Digest>(nd);
  RowBlock rb_tr;  // the rows of the trace LDE this rank holds: all of them, or its block
  if (trace_is_block && !sharded) throw Pb254Error(PB254_E_BAD_ARG, "a row-block trace needs a communicator");
  const u64* tr_shard = nullptr;  // sharded: the trace values of this rank's columns
  if (sharded) {
    tr_shard = trace_is_block ? to_column_shard(d_trace, W, "trace") : d_trace + first_col(W) * n;
    rb_tr = commit_sharded(tr_shard, W, dig_tr, scratch, "trace");
  } else {
    u64* lde_tr = ar.alloc_n<u64>((size_t)W * N);
    {
      Stage st(c, "lde trace");
      ntt::lde_columns(c->tables, d_trace, n, lde_tr, N, scratch, W, L, r, ntt::FROM_VALUES_LDE, s);
    }
    {
      Stage st(c, "merkle trace");
      merkle::build_from_lde(lde_tr, N, W, logN, cap_h, dig_tr, s);
    }
    rb_tr = RowBlock{lde_tr, N};
  }
  std::vector<u64> cap(ncap * 4);
  pb_d2h(cap.data(), dig_tr + (nd - ncap), ncap * 32, s);
  pb_sync(s);
  Challenger ch;
  ch.observe_n(cap.data(), cap.size());
  const size_t pos_caps = blob.size();
  blob.insert(blob.end(), cap.begin(), cap.end());

  // ---- CTL challenges and auxiliary columns (prover.rs:46-54, starky lookup / CTL) -------------
  aux::Challenges chal;
  chal.nch = nch;
  for (int j = 0; j < nch; j++) {
    chal.beta[j] = ch.challenge();
    chal.gamma[j] = ch.challenge();
  }
  // whole matrix, or (row-block trace) this rank's row block [ceil(A / P) P][nloc]
  const size_t Apad = ((size_t)A + P - 1) / P * P;
  u64* aux_vals = ar.alloc_n<u64>(trace_is_block ? Apad * nloc : (size_t)A * n);
  {
    Stage st(c, "aux columns");
    size_t mark = ar.off;
    if (trace_is_block) {
      aux::BlockScan bs;
      bs.world = (int)P;
      bs.rank = (int)rk;
      bs.gather = [&](const void* a, void* b, size_t bytes) { coll(comm->all_gather(comm->user, a, b, bytes), "all_gather (scan)"); };
      aux::build(ar, l, d_trace, nloc, chal, aux_vals, s, &bs);
    } else {
      aux::build(ar, l, d_trace, n, chal, aux_vals, s);
    }
    pb_sync(s);
    ar.off = mark;
  }
  ch.compact(&blob[pos_state]);
  Digest* dig_ax = ar.alloc_n<Digest>(nd);
  RowBlock rb_ax;
  const u64* ax_shard = nullptr;
  if (sharded) {
    ax_shard = trace_is_block ? to_column_shard(aux_vals, A, "aux") : aux_vals + first_col(A) * n;
    rb_ax = commit_sharded(ax_shard, A, dig_ax, scratch, "aux");
  } else {
    u64* lde_ax = ar.alloc_n<u64>((size_t)A * N);
    {
      Stage st(c, "lde aux");
      ntt::lde_columns(c->tables, aux_vals, n, lde_ax, N, scratch, A, L, r, ntt::FROM_VALUES_LDE, s);
    }
    {
      Stage st(c, "merkle aux");
      merkle::build_from_lde(lde_ax, N, A, logN, cap_h, dig_ax, s);
    }
    rb_ax = RowBlock{lde_ax, N};
  }
  pb_d2h(cap.data(), dig_ax + (nd - ncap), ncap * 32, s);
  pb_sync(s);
  ch.observe_n(cap.data(), cap.size());
  blob.insert(blob.end(), cap.begin(), cap.end());
  std::vector<u64> alphas(nch);
  for (int j = 0; j < nch; j++) alphas[j] = ch.challenge();

  // ---- quotient (compute_quotient_polys) --------------------------------------------------------
  const size_t qsize = 2 * n;
  const int K = quot::num_constraints(kind, nch);
  u64* d_w = ar.alloc_n<u64>((size_t)K * nch);
  {
    std::vector<u64> w((size_t)K * nch);
    for (int j = 0; j < nch; j++) {
      u64 p = 1;
      for (int k = K - 1; k >= 0; k--) {
        w[(size_t)k * nch + j] = p;
        p = gl::mul(p, alphas[j]);
      }
    }
    pb_h2d(d_w, w.data(), w.size() * 8, s);
    pb_sync(s);
  }
  const int bpow_stride = 2 * l.L + 17;
  u64* d_bpow = ar.alloc_n<u64>((size_t)nch * bpow_stride);
  {
    std::vector<u64> bp((size_t)nch * bpow_stride);
    for (int j = 0; j < nch; j++) {
      u64 pw = 1;
      for (int k = 0; k < bpow_stride; k++) {
        bp[(size_t)j * bpow_stride + k] = pw;
        pw = gl::mul(pw, chal.beta[j]);
      }
    }
    pb_h2d(d_bpow, bp.data(), bp.size() * 8, s);
    pb_sync(s);
  }
  u64* qvals = ar.alloc_n<u64>((size_t)nch * qsize);
  u64* qcoef = ar.alloc_n<u64>((size_t)nch * qsize);
  int* d_err = ar.alloc_n<int>(1);
  pb_memset(d_err, 0, sizeof(int), s);
  u64* d_dbg_groups = nullptr;
  {
    Stage st(c, "quotient eval");
    quot::Params qp;
    qp.tr = rb_tr.ptr;
    qp.tr_stride = rb_tr.stride;
    qp.ax = rb_ax.ptr;
    qp.ax_stride = rb_ax.stride;
    // sharded: this rank evaluates the points of its own LDE rows into [nch][qloc], gathered below
    const size_t qloc = qsize / P;
    u64* q_mine = sharded ? ar.alloc_n<u64>((size_t)nch * qloc) : nullptr;
    qp.out = sharded ? q_mine : qvals;
    qp.i_base = rk * qloc;
    qp.count = qloc;
    qp.out_stride = sharded ? qloc : qsize;
    qp.wrap = sharded ? 0 : 1;
    qp.weights = d_w;
    qp.bpow = d_bpow;
    qp.bpow_stride = bpow_stride;
    qp.size = qsize;
    qp.log_size = L + 1;
    qp.step = (size_t)1 << (r - 1);
    qp.t = c->tables.t;
    qp.g = gl::root_of_unity(L);
    qp.g_inv = gl::inv(qp.g);
    qp.n_field = (u64)n % gl::P;
    u64 g_pow_n = gl::COSET_SHIFT;
    for (int i = 0; i < L; i++) g_pow_n = gl::sqr(g_pow_n);
    qp.zh[0] = gl::sub(g_pow_n, 1);
    qp.zh[1] = gl::sub(gl::neg(g_pow_n), 1);
    qp.zh_inv[0] = gl::inv(qp.zh[0]);
    qp.zh_inv[1] = gl::inv(qp.zh[1]);
    qp.ch = chal;
    qp.err = d_err;
    qp.dbg = nullptr;
    qp.dbg_point = 5;
    if (keep_debug) {
      qp.dbg = ar.alloc_n<u64>(4096);
      pb_memset(qp.dbg, 0, 4096 * 8, s);
    }
    d_dbg_groups = qp.dbg;
    if (kind == 0)
      quot::run_g1(qp, s);
    else if (kind == 1)
      quot::run_g2(qp, s);
    else
      quot::run_fq(qp, s);
    if (sharded) {
      u64* q_all = ar.alloc_n<u64>((size_t)nch * qsize);  // [rank][challenge][qloc]
      coll(comm->all_gather(comm->user, q_mine, q_all, (size_t)nch * qloc * 8), "all_gather (quotient values)");
      for (size_t p = 0; p < P; p++)
        for (int j = 0; j < nch; j++)
          pb_d2d(qvals + (size_t)j * qsize + p * qloc, q_all + (p * nch + j) * qloc, qloc * 8, s);
    }
  }
  {
    Stage st(c, "quotient intt");
    ntt::coset_intt_columns(c->tables, qvals, qsize, qcoef, qsize, scratch, nch, L + 1, s);
  }
  // chunk (2 j + c) = coefficients [c n, (c+1) n) of quotient j: contiguous with stride n
  u64* lde_q = ar.alloc_n<u64>((size_t)Q * N);
  Digest* dig_q = ar.alloc_n<Digest>(nd);
  {
    Stage st(c, "lde+merkle quotient");
    ntt::lde_columns(c->tables, qcoef, n, lde_q, N, scratch, Q, L, r, ntt::FROM_COEFFS_LDE, s);
    if (sharded) {  // leaves everywhere (Q <= 4 columns are copied, not hashed), inner levels shared out
      merkle::build_from_lde(lde_q, N, Q, logN, logN, dig_q, s);
      size_t mk = ar.off;
      levels_sharded(dig_q, ar.alloc_n<Digest>(Nloc));
      ar.off = mk;
    } else {
      merkle::build_from_lde(lde_q, N, Q, logN, cap_h, dig_q, s);
    }
  }
  int herr = 0;
  pb_d2h(&herr, d_err, sizeof(int), s);
  pb_d2h(cap.data(), dig_q + (nd - ncap), ncap * 32, s);
  pb_sync(s);
  if (herr) throw Pb254Error(PB254_E_BAD_ARG, "internal: constraint count mismatch in the quotient kernel");
  ch.observe_n(cap.data(), cap.size());
  blob.insert(blob.end(), cap.begin(), cap.end());
  (void)pos_caps;
  const E2 zeta = ch.ext_challenge();
  const u64 g = gl::root_of_unity(L);
  E2 zeta_pow_n = zeta;
  for (int i = 0; i < L; i++) zeta_pow_n = gl::emul(zeta_pow_n, zeta_pow_n);
  if (zeta_pow_n.a == 1 && zeta_pow_n.b == 0) throw Pb254Error(PB254_E_BAD_ARG, "opening point is in the subgroup");
  const E2 zeta_next = gl::emul_base(zeta, g);

  // ---- openings (StarkOpeningSet::new) ----------------------------------------------------------
  std::vector<u64> op_tr(4 * (size_t)W), op_ax(4 * (size_t)A), op_q(2 * (size_t)Q), zs_first(2 * (size_t)nch);
  {
    Stage st(c, "openings");
    size_t mark = ar.off;
    E2* wz = ar.alloc_n<E2>(n);
    u64* partial = ar.alloc_n<u64>(WA * fri::PARTS * 4);
    E2* d_op = ar.alloc_n<E2>(2 * WA);
    const E2 scale = gl::emul_base(gl::esub(zeta_pow_n, gl::e2(1, 0)), gl::inv((u64)n % gl::P));
    pb_launch("bary weights", fri::BaryWeightsK{wz, zeta, c->tables.t, L}, n, s, 128);
    if (sharded) {
      // every rank evaluates the columns of its own shard; all-gather of the 2 x cper extension values per rank
      auto open_sharded = [&](const u64* shard, int C, std::vector<u64>& op) {
        const size_t cper = ((size_t)C + P - 1) / P;
        const size_t c0 = std::min((size_t)C, rk * cper), c1 = std::min((size_t)C, c0 + cper), nc = c1 - c0;
        E2* d_mine = ar.alloc_n<E2>(2 * cper);
        E2* d_all = ar.alloc_n<E2>(P * 2 * cper);
        pb_memset(d_mine, 0, 2 * cper * sizeof(E2), s);
        if (nc) {
          pb_launch("open shard", fri::WeightedPartialK{shard, n, n, wz, partial, 1}, nc * fri::PARTS, s, 256);
          fri::finish_openings(partial, nc, scale, d_mine, d_mine + cper, s);
        }
        coll(comm->all_gather(comm->user, d_mine, d_all, 2 * cper * sizeof(E2)), "all_gather (openings)");
        std::vector<u64> h(P * 4 * cper);
        pb_d2h(h.data(), d_all, h.size() * 8, s);
        pb_sync(s);
        for (size_t col = 0; col < (size_t)C; col++) {
          const size_t q = col / cper, j = col % cper;
          for (int e = 0; e < 2; e++) {
            op[2 * col + e] = h[((q * 2 + 0) * cper + j) * 2 + e];                 // at zeta
            op[2 * ((size_t)C + col) + e] = h[((q * 2 + 1) * cper + j) * 2 + e];   // at g zeta
          }
        }
      };
      open_sharded(tr_shard, W, op_tr);
      ch.observe_n(op_tr.data(), 2 * (size_t)W);
      open_sharded(ax_shard, A, op_ax);
    } else {
      // The transcript absorbs [local | aux | quotient], [next | aux_next], [ctl_zs_first]; every batch of opened
      // values is hashed on the host while the GPU evaluates the next one (the observe ORDER is unchanged).
      E2* d_op2 = ar.alloc_n<E2>(2 * WA);
      pb_launch("open trace", fri::WeightedPartialK{d_trace, n, n, wz, partial, 1}, (size_t)W * fri::PARTS, s, 256);
      fri::finish_openings(partial, W, scale, d_op, d_op + W, s);
      pb_d2h(op_tr.data(), d_op, (size_t)W * 32, s);
      pb_sync(s);
      pb_launch("open aux", fri::WeightedPartialK{aux_vals, n, n, wz, partial, 1}, (size_t)A * fri::PARTS, s, 256);
      fri::finish_openings(partial, A, scale, d_op2, d_op2 + A, s);
      // (host hashing comes before the copy: a device-to-host copy into pageable memory blocks the host)
      ch.observe_n(op_tr.data(), 2 * (size_t)W);  // local trace values, overlapped with the auxiliary openings
      pb_d2h(op_ax.data(), d_op2, (size_t)A * 32, s);
      pb_sync(s);
    }
    pb_launch("zeta powers", fri::PowTableK{wz, zeta}, n, s, 128);
    pb_launch("open quotient", fri::WeightedPartialK{qcoef, n, n, wz, partial, 0}, (size_t)Q * fri::PARTS, s, 256);
    fri::finish_openings(partial, Q, gl::e2(1, 0), d_op, nullptr, s);
    ch.observe_n(op_ax.data(), 2 * (size_t)A);  // local auxiliary values, overlapped with the quotient openings
    pb_d2h(op_q.data(), d_op, (size_t)Q * 16, s);
    if (trace_is_block) {  // row 0 of the CTL-Z columns lives on rank 0: everyone contributes its local row 0
      u64* z_mine = ar.alloc_n<u64>(2 * nch);
      u64* z_all = ar.alloc_n<u64>(P * 2 * nch);
      for (int k = 0; k < 2 * nch; k++) pb_d2d(z_mine + k, aux_vals + (size_t)(nlk + k) * nloc, 8, s);
      coll(comm->all_gather(comm->user, z_mine, z_all, (size_t)2 * nch * 8), "all_gather (ctl_zs_first)");
      pb_d2h(zs_first.data(), z_all, (size_t)2 * nch * 8, s);
    } else {
      for (int k = 0; k < 2 * nch; k++) pb_d2h(&zs_first[k], aux_vals + (size_t)(nlk + k) * n, 8, s);
    }
    pb_sync(s);
    ar.off = mark;
  }
  // proof order: local, next, aux, aux_next, ctl_zs_first, quotient
  blob.insert(blob.end(), op_tr.begin(), op_tr.end());
  blob.insert(blob.end(), op_ax.begin(), op_ax.end());
  blob.insert(blob.end(), zs_first.begin(), zs_first.end());
  blob.insert(blob.end(), op_q.begin(), op_q.end());
  // observe_openings, continued: quotient, then [next | aux_next], [ctl_zs_first]
  ch.observe_n(op_q.data(), 2 * (size_t)Q);
  ch.observe_n(op_tr.data() + 2 * W, 2 * (size_t)W);
  ch.observe_n(op_ax.data() + 2 * A, 2 * (size_t)A);
  for (int k = 0; k < 2 * nch; k++) {
    ch.observe(zs_first[k]);
    ch.observe(0);
  }

  // ---- FRI (PolynomialBatch::prove_openings) ------------------------------------------------------
  const E2 fri_alpha = ch.ext_challenge();
  const int NP = W + A + Q;
  std::vector<E2> apow(NP + 1);
  apow[0] = gl::e2(1, 0);
  for (int i = 1; i <= NP; i++) apow[i] = gl::emul(apow[i - 1], fri_alpha);
  auto ext_at = [](const std::vector<u64>& v, size_t i) { return gl::e2(v[2 * i], v[2 * i + 1]); };
  E2 O0 = gl::e2(0, 0), O1 = gl::e2(0, 0), O2 = gl::e2(0, 0);
  for (int i = 0; i < W; i++) {
    O0 = gl::eadd(O0, gl::emul(apow[i], ext_at(op_tr, i)));
    O1 = gl::eadd(O1, gl::emul(apow[i], ext_at(op_tr, W + i)));
  }
  for (int i = 0; i < A; i++) {
    O0 = gl::eadd(O0, gl::emul(apow[W + i], ext_at(op_ax, i)));
    O1 = gl::eadd(O1, gl::emul(apow[W + i], ext_at(op_ax, A + i)));
  }
  for (int i = 0; i < Q; i++) O0 = gl::eadd(O0, gl::emul(apow[W + A + i], ext_at(op_q, i)));
  for (int k = 0; k < 2 * nch; k++) O2 = gl::eadd(O2, gl::emul_base(apow[k], zs_first[k]));
  E2* d_apow = ar.alloc_n<E2>(NP + 1);
  pb_h2d(d_apow, apow.data(), (size_t)(NP + 1) * 16, s);
  E2* V = ar.alloc_n<E2>(N);
  {
    Stage st(c, "fri combine");
    fri::CombineK k;
    k.tr = rb_tr.ptr;
    k.ax = rb_ax.ptr;
    k.qt = lde_q + rk * Nloc;
    k.tr_stride = rb_tr.stride;
    k.ax_stride = rb_ax.stride;
    k.qt_stride = N;
    k.i_base = rk * Nloc;
    k.natural_out = sharded ? 1 : 0;
    k.N = N;
    k.W = W;
    k.A = A;
    k.Q = Q;
    k.nlk = nlk;
    k.nz = 2 * nch;
    k.apow = d_apow;
    k.O0 = O0;
    k.O1 = O1;
    k.O2 = O2;
    k.zeta = zeta;
    k.zeta_next = zeta_next;
    k.sh1 = apow[W + A];
    k.sh2 = apow[2 * nch];
    k.t = c->tables.t;
    k.log_N = logN;
    k.out = V;
    if (sharded) {
      E2* v_mine = ar.alloc_n<E2>(Nloc);
      E2* v_nat = ar.alloc_n<E2>(N);
      k.out = v_mine;
      pb_launch("fri combine", k, Nloc, s, 128);
      coll(comm->all_gather(comm->user, v_mine, v_nat, Nloc * sizeof(E2)), "all_gather (combined polynomial)");
      pb_launch("bit reverse", fri::BitReverseE2K{v_nat, V, logN}, N, s, 128);
    } else {
      pb_launch("fri combine", k, N, s, 128);
    }
    pb_sync(s);  // apow (host vector) must outlive the H2D copy
  }
  struct Layer {
    E2* vals;
    Digest* dig;
    int log_len, arity_bits, log_leaves;
  };
  std::vector<Layer> layers;
  std::vector<E2> fri_betas;
  std::vector<u64> final_poly;
  {
    Stage st(c, "fri commit phase");
    int log_len = logN;
    u64 shift = gl::COSET_SHIFT;
    for (unsigned ab : arities) {
      Layer ly;
      ly.vals = V;
      ly.log_len = log_len;
      ly.arity_bits = (int)ab;
      ly.log_leaves = log_len - (int)ab;
      if (ly.log_leaves < cap_h) throw Pb254Error(PB254_E_BAD_ARG, "FRI layer smaller than the Merkle cap");
      size_t ndl = merkle::tree_digests(ly.log_leaves, cap_h);
      ly.dig = ar.alloc_n<Digest>(ndl);
      merkle::build_from_rows((const u64*)V, 2 << ab, ly.log_leaves, cap_h, ly.dig, s);
      pb_d2h(cap.data(), ly.dig + (ndl - ncap), ncap * 32, s);
      pb_sync(s);
      ch.observe_n(cap.data(), cap.size());
      blob.insert(blob.end(), cap.begin(), cap.end());
      E2 beta = ch.ext_challenge();
      fri_betas.push_back(beta);
      E2* Vn = ar.alloc_n<E2>((size_t)1 << ly.log_leaves);
      pb_launch("fri fold", fri::FoldK{V, Vn, beta, gl::inv(shift), c->tables.t, log_len, (int)ab},
                (size_t)1 << ly.log_leaves, s, 64);
      layers.push_back(ly);
      V = Vn;
      log_len = ly.log_leaves;
      shift = gl::pow(shift, (u64)1 << ab);
    }
    // final polynomial: coset iNTT of the last layer on the host (<= a few hundred points)
    size_t m = (size_t)1 << log_len;
    std::vector<u64> vb(2 * m);
    pb_d2h(vb.data(), V, m * 16, s);
    pb_sync(s);
    std::vector<E2> nat(m);
    for (size_t i = 0; i < m; i++) {
      size_t j = gl::brev32((u32)i, log_len);
      nat[j] = gl::e2(vb[2 * i], vb[2 * i + 1]);
    }
    const u64 winv = gl::inv(gl::root_of_unity(log_len)), minv = gl::inv((u64)m), sinv = gl::inv(shift);
    std::vector<E2> coef(m);
    u64 wi = 1, si = minv;  // w^-i and s^-i / m
    for (size_t i = 0; i < m; i++) {
      E2 acc = gl::e2(0, 0);
      u64 x = 1;  // w^(-i j)
      for (size_t j = 0; j < m; j++) {
        acc = gl::eadd(acc, gl::emul_base(nat[j], x));
        x = gl::mul(x, wi);
      }
      coef[i] = gl::emul_base(acc, si);
      wi = gl::mul(wi, winv);
      si = gl::mul(si, sinv);
    }
    size_t keep = m >> r;
    for (size_t i = keep; i < m; i++)
      if (coef[i].a || coef[i].b) throw Pb254Error(PB254_E_BAD_ARG, "internal: FRI final polynomial has too high degree");
    for (size_t i = 0; i < keep; i++) {
      ch.observe(coef[i].a);
      ch.observe(coef[i].b);
    }
    final_poly.resize(2 * keep);
    for (size_t i = 0; i < keep; i++) {
      final_poly[2 * i] = coef[i].a;
      final_poly[2 * i + 1] = coef[i].b;
    }
  }

  // ---- proof of work: minimal witness -----------------------------------------------------------
  u64 pow_witness = 0;
  {
    Stage st(c, "pow");
    fri::PowK pk;
    memcpy(pk.state, ch.state, sizeof pk.state);
    pk.pos = (int)ch.in.size();
    for (size_t i = 0; i < ch.in.size(); i++) pk.state[i] = ch.in[i];
    pk.pow_bits = (int)cfg.pow_bits;
    u64* d_res = ar.alloc_n<u64>(1);
    pk.result = d_res;
    // candidates are tried in increasing order, chunk by chunk (the minimum of the first successful chunk is the
    // minimal witness); a first chunk of 2^(pow_bits + 1) succeeds with probability 1 - e^-2
    size_t chunk = (size_t)2 << (cfg.pow_bits < 19 ? cfg.pow_bits : 19);
    u64 found = ~(u64)0;
    for (u64 base = 0; found == ~(u64)0; base += chunk, chunk = (size_t)1 << 20) {
      if (base >= ((u64)1 << 44)) throw Pb254Error(PB254_E_BAD_ARG, "proof of work search failed");
      pb_memset(d_res, 0xff, 8, s);
      pk.base = base;
      pb_launch("pow grind", pk, chunk, s, 128);
      pb_d2h(&found, d_res, 8, s);
      pb_sync(s);
    }
    pow_witness = found;
    ch.observe(pow_witness);
    u64 resp = ch.challenge();
    if (cfg.pow_bits && (resp >> (64 - cfg.pow_bits)) != 0) throw Pb254Error(PB254_E_BAD_ARG, "internal: pow check failed");
  }

  // ---- query rounds -------------------------------------------------------------------------------
  {
    Stage st(c, "queries");
    const size_t nq = cfg.num_query_rounds;
    std::vector<u64> idx(nq);
    for (auto& x : idx) x = ch.challenge() % (u64)N;
    fri::GatherK gk;
    int ns = 0, off = 0;
    auto add = [&](int type, int words, int shift, int log_n, const void* ptr, size_t stride, bool block = false) {
      if (ns >= fri::MAX_SECTIONS) throw Pb254Error(PB254_E_BAD_ARG, "too many proof sections");
      gk.sec[ns] = fri::Section{type, off, words, shift, log_n, (const u64*)ptr, stride};
      if (block) {  // only the rows of this rank's block are here
        gk.sec[ns].row0 = rk * Nloc;
        gk.sec[ns].rows = Nloc;
      }
      off += words;
      ns++;
    };
    const int nsib = 4 * (logN - cap_h);
    add(0, W, 0, logN, rb_tr.ptr, rb_tr.stride, sharded);
    add(1, nsib, 0, logN, dig_tr, 0);
    add(0, A, 0, logN, rb_ax.ptr, rb_ax.stride, sharded);
    add(1, nsib, 0, logN, dig_ax, 0);
    add(0, Q, 0, logN, lde_q, N);
    add(1, nsib, 0, logN, dig_q, 0);
    int shift = 0;
    for (auto& ly : layers) {
      shift += ly.arity_bits;
      add(2, 2 << ly.arity_bits, shift, ly.log_leaves, ly.vals, 0);
      add(1, 4 * (ly.log_leaves - cap_h), shift, ly.log_leaves, ly.dig, 0);
    }
    gk.nsec = ns;
    gk.rec_words = off;
    u64* d_idx = ar.alloc_n<u64>(nq);
    u64* d_out = ar.alloc_n<u64>(nq * (size_t)off);
    pb_h2d(d_idx, idx.data(), nq * 8, s);
    gk.indices = d_idx;
    gk.out = d_out;
    gk.zero_whole = sharded && rk != 0;
    pb_launch("query gather", gk, nq * (size_t)off, s, 128);
    if (sharded) {  // every word of a record is non-zero on at most one rank: gather the records and add them up
      u64* d_all = ar.alloc_n<u64>(P * nq * (size_t)off);
      coll(comm->all_gather(comm->user, d_out, d_all, nq * (size_t)off * 8), "all_gather (query records)");
      pb_launch("merge query records", SumRecordsK{d_all, d_out, nq * (size_t)off, (int)P}, nq * (size_t)off, s, 128);
    }
    size_t pos = blob.size();
    blob.resize(pos + nq * (size_t)off);
    pb_d2h(&blob[pos], d_out, nq * (size_t)off * 8, s);
    pb_sync(s);
    out.dbg_indices = idx;
  }
  blob.insert(blob.end(), final_poly.begin(), final_poly.end());
  blob.push_back(pow_witness);

  if (keep_debug) {
    out.dbg_aux.resize((size_t)A * n);
    pb_d2h(out.dbg_aux.data(), aux_vals, (size_t)A * n * 8, s);
    out.dbg_chunks.resize((size_t)Q * n);
    pb_d2h(out.dbg_chunks.data(), qcoef, (size_t)Q * n * 8, s);
    out.dbg_groups.resize(4096);
    pb_d2h(out.dbg_groups.data(), d_dbg_groups, 4096 * 8, s);
    pb_sync(s);
    auto& d = out.dbg_challenges;
    d.clear();
    for (int j = 0; j < nch; j++) d.push_back(chal.beta[j]);
    for (int j = 0; j < nch; j++) d.push_back(chal.gamma[j]);
    for (int j = 0; j < nch; j++) d.push_back(alphas[j]);
    d.push_back(zeta.a);
    d.push_back(zeta.b);
    d.push_back(fri_alpha.a);
    d.push_back(fri_alpha.b);
    for (auto& b : fri_betas) {
      d.push_back(b.a);
      d.push_back(b.b);
    }
  }
}

}  // namespace prover
