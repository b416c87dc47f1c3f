// K15 `verify_device`: the two heavy parts of verify::verify_walk on the context's GPU, for a batch of proofs of one
// kind under one StarkConfig (pb254_verify_many_device; pb254_verify_device is the batch of one).
//   1. native CTL  NativeCtlK, one thread per instance of every proof of a round: canonical loads, the native output
//                  with the shared ladder (verify::native_output), then per challenge j of its proof the input and
//                  output tuple combinations in the host's Horner order (last tuple element first, then + gamma), a
//                  zero flag per (proof, c, j) or the inverse. Each proof's lowest failing instance and its status go
//                  into one word per proof with tg::set_lowest. SumInvK / SumPartK add the inverses per (proof, c, j);
//                  Goldilocks addition is exact, so any order gives the host sum.
//   2. Merkle      MerkleCheckK, one thread per (proof, query, tree): verify::merkle_path_ok with the device
//                  permutation. The walk has rejected every blob word >= p before this runs, as the lazy permutation
//                  requires.
// A segment table per round says where each proof's instances, sum chunks and (query, tree) pairs start; proofs of
// different degree_bits have different tree depths and numbers of FRI layers, so each proof has its own trees.
//
// Host side: proofs go in rounds of at most ROUND. Each proof of a round runs verify_walk on its own host thread with a
// DeviceChecks provider; the round's coordinator (the calling thread) waits until every walk has called start() or
// ended, uploads the round once, launches each kernel once over all its proofs, copies the results back and wakes the
// walks. The walks evaluate their quotient identities meanwhile and then read their own results in their own order, so
// every outcome equals pb254_verify's for that proof alone.
#pragma once
#include "verify.cuh"
#include <condition_variable>
#include <memory>
#include <mutex>
#include <system_error>
#include <thread>

namespace verify_dev {

// where the leaf and the path of tree t sit in a query record, and its cap in the proof's blob (words)
struct Tree {
  u32 leaf, leaf_len, path, depth, shift;  // the leaf index is the query index >> shift
  u64 cap;
};
// one proof of a round: its blob in the round's blob buffer, its query records and its trees
struct Seg {
  u64 blob, queries, rec;  // first word of the blob, of the first query record, and the record length (words)
  u32 t0, T;               // trees[t0 .. t0 + T)
};
static_assert(sizeof(Tree) % 8 == 0 && sizeof(Seg) % 8 == 0, "Tree and Seg are uploaded as u64 words");
static constexpr int STATUS_BITS = 3;  // bad = (k << STATUS_BITS) | verify::NATIVE_*
static constexpr unsigned NO_BAD = 0xffffffffu;
static constexpr int SUM_CHUNK = 256;
static constexpr size_t ROUND = 64;             // proofs per round: host threads and one launch per stage
static constexpr size_t MAX_PROOFS = 1u << 12;  // per call

// a = a * beta^4 + (the four 16-bit limbs of w, most significant first)
PB_HD u64 horner_word(u64 a, u64 w, u64 beta) {
#pragma unroll
  for (int q = 3; q >= 0; q--) a = gl::add(gl::mul(a, beta), (w >> (16 * q)) & 0xffff);
  return a;
}

// the proof b with s[b] <= g < s[b + 1], for the non-decreasing segment starts s[0 .. nb] and g < s[nb]
PB_HD int seg_of(const u64* s, int nb, u64 g) {
  int lo = 0, hi = nb - 1;
  while (lo < hi) {
    const int mid = (lo + hi + 1) >> 1;
    if (s[mid] <= g)
      lo = mid;
    else
      hi = mid - 1;
  }
  return lo;
}

template <int KIND>
struct NativeCtlK {
  static constexpr int IN = KIND == 0 ? 20 : KIND == 1 ? 36 : 8, OUT = KIND == 0 ? 8 : KIND == 1 ? 16 : 4;
  const u64* inputs;  // [K][IN]: the batches of the round's proofs, back to back
  const u64* ts;      // [K]
  const u64* k0;      // [nb + 1]: proof b's instances are k0[b] .. k0[b + 1]
  const u64* chal;    // [nb][2 nch]: beta[nch], gamma[nch] of each proof
  u64* inv;           // [2 nch][K]: 1 / combination, 0 where it is zero or the instance failed
  int* zero;          // [nb][2 nch]
  unsigned* bad;      // [nb]: each proof's lowest (k << STATUS_BITS) | status
  size_t K;
  int nb, nch;
  PB_HD void operator()(size_t g) const {
    const int pb = seg_of(k0, nb, g);
    const size_t k = g - k0[pb];
    const u64* w = inputs + g * IN;
    u64 out[OUT];
    const int st = verify::native_output<KIND>(w, out);
    if (st) tg::set_lowest(bad + pb, (unsigned)(k << STATUS_BITS) | (unsigned)st);
    const u64 t = ts[g] % gl::P;
    const u64* ch = chal + (size_t)pb * 2 * nch;
#pragma unroll 1
    for (int j = 0; j < nch; j++) {
      const u64 beta = ch[j], gamma = ch[nch + j];
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
        if (!st && v == 0) zero[(size_t)pb * 2 * nch + cj] = 1;
        inv[cj * K + g] = v ? gl::inv(v) : 0;
      }
    }
  }
};

// part[cj][p] = sum of inv[cj][..] over the SUM_CHUNK instances of chunk p; proof b's chunks are p0[b] .. p0[b + 1]
struct SumInvK {
  const u64* inv;
  const u64 *k0, *p0;
  u64* part;
  size_t K, P;
  int nb;
  PB_HD void operator()(size_t gid) const {
    const size_t cj = gid / P, p = gid % P;
    const int b = seg_of(p0, nb, p);
    const size_t begin = k0[b] + (p - p0[b]) * SUM_CHUNK, end = begin + SUM_CHUNK < k0[b + 1] ? begin + SUM_CHUNK : k0[b + 1];
    u64 s = 0;
    for (size_t k = begin; k < end; k++) s = gl::add(s, inv[cj * K + k]);
    part[gid] = s;
  }
};
// sum[b][cj] = the parts of proof b under (c, j)
struct SumPartK {
  const u64 *part, *p0;
  u64* sum;  // [nb][2 nch]
  size_t P;
  int ncj;
  PB_HD void operator()(size_t gid) const {
    const size_t b = gid / ncj, cj = gid % ncj;
    u64 s = 0;
    for (size_t p = p0[b]; p < p0[b + 1]; p++) s = gl::add(s, part[cj * P + p]);
    sum[gid] = s;
  }
};

struct MerkleCheckK {
  const u64* blob;    // the round's blobs
  const Seg* segs;    // [nb]
  const u64* m0;      // [nb + 1]: proof b's (query, tree) pairs are m0[b] .. m0[b + 1], (q, t) at m0[b] + q T + t
  const Tree* trees;
  const u64* idx;     // [nb][nq]
  size_t nq;
  int nb;
  int* ok;            // [m0[nb]]
  PB_HD void operator()(size_t gid) const {
    const int b = seg_of(m0, nb, gid);
    const Seg sg = segs[b];
    const size_t local = gid - m0[b], q = local / sg.T;
    const Tree tr = trees[sg.t0 + local % sg.T];
    const u64* bp = blob + sg.blob;
    const u64* rp = bp + sg.queries + q * sg.rec;
    ok[gid] = verify::merkle_path_ok(rp + tr.leaf, tr.leaf_len, (size_t)(idx[(size_t)b * nq + q] >> tr.shift), rp + tr.path,
                                     (int)tr.depth, bp + tr.cap);
  }
};

// What one walk's start() copies from its Job: the Job points at locals of the walk, which may return (at the quotient
// identity) before the coordinator has read them. The blob and the batch are the caller's and outlive the call.
struct Item {
  bool started = false;
  const u64 *blob = nullptr, *inputs = nullptr, *ts = nullptr;
  size_t words = 0, K = 0;
  u64 queries = 0, rec = 0;
  std::vector<u64> chal, idx;  // beta[nch], gamma[nch]; the query indices
  std::vector<Tree> trees;     // of one query record (proofview.cuh)
};

static inline Item item_of(const verify::Job& j) {
  const pb254_proof_layout& lay = *j.lay;
  Item it;
  it.started = true;
  it.blob = j.blob;
  it.words = j.words;
  it.inputs = j.inputs;
  it.ts = j.timestamps;
  it.K = j.K;
  it.queries = lay.query_round_proofs;
  it.rec = lay.query_words;
  it.idx = *j.idx;
  it.chal.resize(2 * (size_t)j.nch);
  for (int i = 0; i < j.nch; i++) {
    it.chal[i] = j.chal->beta[i];
    it.chal[j.nch + i] = j.chal->gamma[i];
  }
  const u32 d0 = (u32)(j.logN - j.cap_h);
  it.trees.push_back(Tree{lay.q_trace_leaf, lay.trace_width, lay.q_trace_path, d0, 0, lay.trace_cap});
  it.trees.push_back(Tree{lay.q_aux_leaf, lay.aux_width, lay.q_aux_path, d0, 0, lay.auxiliary_polys_cap});
  it.trees.push_back(Tree{lay.q_quotient_leaf, lay.quotient_width, lay.q_quotient_path, d0, 0, lay.quotient_polys_cap});
  u32 shift = 0;
  for (size_t i = 0; i < j.arities->size(); i++) {
    shift += (*j.arities)[i];
    it.trees.push_back(Tree{lay.q_step_evals[i], lay.q_step_evals_words[i], lay.q_step_path[i],
                            lay.q_step_path_words[i] / 4, shift, lay.commit_phase_merkle_caps + i * lay.cap_words});
  }
  return it;
}

// One round: the walks' side (arrive, wait, the results) and the coordinator's (run).
struct Round {
  pb254_ctx* c;
  int kind, ncj;
  size_t nq;
  std::vector<Item> items;
  // results, valid once ready: per proof its bad word, its zero flags and sums per (c, j), its Merkle pairs
  std::vector<u64> m0, sum;
  std::vector<u32> flags;  // bad[nb] | zero[nb][ncj] | ok[m0[nb]]
  std::mutex mu;
  std::condition_variable cv;
  size_t pending;  // walks that have neither started nor ended
  bool ready = false;
  int err = 0;  // the coordinator's PB254_E_CUDA / PB254_E_OOM, passed to every waiting walk
  std::string err_msg;

  Round(pb254_ctx* ctx, int kind_, const pb254_config& cfg, size_t n)
      : c(ctx), kind(kind_), ncj(2 * (int)cfg.num_challenges), nq(cfg.num_query_rounds), items(n), pending(n) {}

  void arrive(size_t b, Item* it) {
    std::lock_guard<std::mutex> lk(mu);
    if (it) items[b] = std::move(*it);
    if (--pending == 0) cv.notify_all();
  }
  void wait() {
    std::unique_lock<std::mutex> lk(mu);
    cv.wait(lk, [&] { return ready; });
    if (err) throw Pb254Error(err, err_msg);
  }

  // the coordinator, on the calling thread
  void run() {
    {
      std::unique_lock<std::mutex> lk(mu);
      cv.wait(lk, [&] { return pending == 0; });
    }
    try {
      launch();
    } catch (const Pb254Error& e) {
      err = e.code;
      err_msg = e.what();
    } catch (const std::bad_alloc&) {
      err = PB254_E_OOM;
      err_msg = "verify: host memory exhausted";
    }
    if (err) {
#if !PB_HOSTSIM
      (void)cudaStreamSynchronize(c->stream);  // nothing of the round may still run once the walks are woken
#endif
    }
    {
      std::lock_guard<std::mutex> lk(mu);
      ready = true;
    }
    cv.notify_all();
  }

  void launch() {
    const int nb = (int)items.size();
    const int IN = tg::layout_for(kind).in_words;
    const pbStream s = c->stream;
    // the segment table over every proof of the round; a proof that never started has empty segments
    std::vector<u64> starts(3 * (size_t)(nb + 1), 0);  // k0 | p0 | m0
    u64 *k0 = starts.data(), *p0 = k0 + nb + 1, *mm = p0 + nb + 1;
    std::vector<Seg> segs(nb);
    size_t W = 0, NT = 0;
    bool any = false;
    for (int b = 0; b < nb; b++) {
      const Item& it = items[b];
      const size_t T = it.started ? it.trees.size() : 0;
      segs[b] = Seg{W, it.queries, it.rec, (u32)NT, (u32)T};
      k0[b + 1] = k0[b] + it.K;
      p0[b + 1] = p0[b] + (it.K + SUM_CHUNK - 1) / SUM_CHUNK;
      mm[b + 1] = mm[b] + nq * T;
      W += it.words;
      NT += T;
      any |= it.started;
    }
    m0.assign(mm, mm + nb + 1);
    if (!any) return;  // every walk ended before the device part: nothing to run
    const size_t K = k0[nb], P = p0[nb], M = mm[nb], ncjs = (size_t)ncj;
    const size_t TW = sizeof(Tree) / 8, SW = sizeof(Seg) / 8;
    // one upload: blobs | inputs | timestamps | challenges | query indices | trees | segments | segment starts
    const size_t o_in = W, o_ts = o_in + K * IN, o_ch = o_ts + K, o_idx = o_ch + nb * ncjs, o_tr = o_idx + nb * nq,
                 o_seg = o_tr + NT * TW, o_st = o_seg + nb * SW, S = o_st + starts.size();
    std::unique_ptr<u64[]> stage(new u64[S]);
    u64* h = stage.get();
    NT = 0;
    for (int b = 0; b < nb; b++) {
      const Item& it = items[b];
      if (!it.started) {
        std::fill(h + o_ch + b * ncjs, h + o_ch + (b + 1) * ncjs, 0);
        std::fill(h + o_idx + b * nq, h + o_idx + (b + 1) * nq, 0);
        continue;
      }
      memcpy(h + segs[b].blob, it.blob, it.words * 8);
      memcpy(h + o_in + k0[b] * IN, it.inputs, it.K * IN * 8);
      memcpy(h + o_ts + k0[b], it.ts, it.K * 8);
      memcpy(h + o_ch + b * ncjs, it.chal.data(), ncjs * 8);
      memcpy(h + o_idx + b * nq, it.idx.data(), nq * 8);
      memcpy(h + o_tr + NT * TW, it.trees.data(), it.trees.size() * sizeof(Tree));
      NT += it.trees.size();
    }
    memcpy(h + o_seg, segs.data(), nb * sizeof(Seg));
    memcpy(h + o_st, starts.data(), starts.size() * 8);

    const size_t NF = nb + nb * ncjs + M;
    c->arena.reserve((S + ncjs * K + ncjs * P + nb * ncjs) * 8 + NF * 4 + 8 * 256);
    c->arena.reset();
    u64* d = c->arena.alloc_n<u64>(S);
    u64* d_inv = c->arena.alloc_n<u64>(ncjs * K + 1);
    u64* d_part = c->arena.alloc_n<u64>(ncjs * P + 1);
    u64* d_sum = c->arena.alloc_n<u64>(nb * ncjs);
    u32* d_flags = c->arena.alloc_n<u32>(NF);
    unsigned* d_bad = d_flags;
    int* d_zero = (int*)d_flags + nb;
    int* d_ok = d_zero + nb * ncjs;
    pb_h2d(d, h, S * 8, s);
    pb_memset(d_bad, 0xff, nb * sizeof(unsigned), s);
    pb_memset(d_zero, 0, nb * ncjs * sizeof(int), s);
    const u64 *d_k0 = d + o_st, *d_p0 = d_k0 + nb + 1, *d_m0 = d_p0 + nb + 1;
    const int nch = ncj / 2;

    int t = c->times.begin("verify native ctl", s);
    if (kind == 0)
      pb_launch("verify native ctl", NativeCtlK<0>{d + o_in, d + o_ts, d_k0, d + o_ch, d_inv, d_zero, d_bad, K, nb, nch}, K,
                s, 32);
    else if (kind == 1)
      pb_launch("verify native ctl", NativeCtlK<1>{d + o_in, d + o_ts, d_k0, d + o_ch, d_inv, d_zero, d_bad, K, nb, nch}, K,
                s, 32);
    else
      pb_launch("verify native ctl", NativeCtlK<2>{d + o_in, d + o_ts, d_k0, d + o_ch, d_inv, d_zero, d_bad, K, nb, nch}, K,
                s, 32);
    pb_launch("verify ctl sums", SumInvK{d_inv, d_k0, d_p0, d_part, K, P, nb}, ncjs * P, s, 128);
    pb_launch("verify ctl total", SumPartK{d_part, d_p0, d_sum, P, ncj}, nb * ncjs, s, 32);
    c->times.end(t, s);
    t = c->times.begin("verify merkle", s);
    pb_launch("verify merkle", MerkleCheckK{d, (const Seg*)(d + o_seg), d_m0, (const Tree*)(d + o_tr), d + o_idx, nq, nb, d_ok},
              M, s, 32);
    c->times.end(t, s);

    sum.resize(nb * ncjs);
    flags.resize(NF);
    pb_d2h(sum.data(), d_sum, sum.size() * 8, s);
    pb_d2h(flags.data(), d_flags, NF * 4, s);
    pb_sync(s);
  }
};

// verify::Checks for proof b of a round: start() hands its Item to the coordinator, ctl() and merkle_ok() wait for the
// round's results. A walk that ends without start() still arrives, from the destructor, so the coordinator never waits
// on it.
struct DeviceChecks : verify::Checks {
  Round& r;
  size_t b;
  bool arrived = false;
  DeviceChecks(Round& round, size_t index) : r(round), b(index) {}
  ~DeviceChecks() override {
    if (!arrived) r.arrive(b, nullptr);
  }
  void start(const verify::Job& j) override {
    Item it = item_of(j);
    arrived = true;
    r.arrive(b, &it);
  }
  void ctl(verify::CtlResults& o) override {
    r.wait();
    const unsigned bad = r.flags[b];
    if (bad != NO_BAD) {
      const Pb254Error e = verify::native_error((int)(bad & ((1u << STATUS_BITS) - 1)));
      o.code = e.code;
      o.msg = e.what();
      return;
    }
    const size_t nb = r.items.size(), ncj = (size_t)r.ncj;
    o.zero.assign(r.flags.begin() + nb + b * ncj, r.flags.begin() + nb + (b + 1) * ncj);
    o.sum.assign(r.sum.begin() + b * ncj, r.sum.begin() + (b + 1) * ncj);
  }
  bool merkle_ok(size_t q, int tree, const u64*, size_t, size_t, const u64*, int, const u64*) override {
    r.wait();
    const size_t nb = r.items.size();
    return r.flags[nb + nb * (size_t)r.ncj + r.m0[b] + q * r.items[b].trees.size() + tree] != 0;
  }
};

// One proof's outcome, as pb254_verify reports it: 0 = accepted, else its code and pb254_last_error().
struct Outcome {
  int code = 0;
  std::string msg;
};

// pb254_verify_many_device on a context already in scope: proof b's rows are starts[b] .. starts[b + 1] of
// inputs / ts. Writes out[b] for every proof, or throws the PB254_E_CUDA / PB254_E_OOM error that failed a round.
static inline void verify_many(pb254_ctx* c, int kind, const pb254_config& cfg, const u64* const* blobs,
                               const size_t* words, size_t n, const u64* inputs, const u64* ts, const u64* starts,
                               Outcome* out) {
  const size_t IN = (size_t)tg::layout_for(kind).in_words;
  for (size_t first = 0; first < n; first += ROUND) {
    const size_t nb = std::min(ROUND, n - first);
    Round r(c, kind, cfg, nb);
    std::vector<std::thread> walks;
    walks.reserve(nb);
    bool spawn_failed = false;
    for (size_t i = 0; i < nb; i++) {
      const size_t b = first + i;
      try {
        walks.emplace_back([&, i, b] {
          DeviceChecks checks(r, i);
          try {
            verify::verify_walk(kind, cfg, blobs[b], words[b], inputs + starts[b] * IN, ts + starts[b],
                                (size_t)(starts[b + 1] - starts[b]), checks);
          } catch (const Pb254Error& e) {
            out[b] = Outcome{e.code, e.what()};
          } catch (const std::exception& e) {
            out[b] = Outcome{PB254_E_BAD_ARG, e.what()};
          }
        });
      } catch (const std::system_error&) {
        spawn_failed = true;
        r.arrive(i, nullptr);
      }
    }
    r.run();
    for (auto& w : walks) w.join();
    if (spawn_failed) throw Pb254Error(PB254_E_OOM, "verify: could not start a host thread");
    if (r.err) throw Pb254Error(r.err, r.err_msg);
  }
}

}  // namespace verify_dev
