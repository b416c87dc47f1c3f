// Unity translation unit of libpb254.so: kernels + host orchestration + C ABI (include/pb254.h).
// Built by plonky2_bn254_b200/build.py with
//   nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
// (or, test-only, g++ -x c++ -DPB254_HOSTSIM for the host-simulation library under tests/hostsim/).
#include "../../include/pb254.h"
#include "compat.cuh"
std::atomic<unsigned long long> g_pb_launches{0};
#include "context.cuh"
#include "ntt.cuh"
#include <memory>
#include <thread>
#include "merkle.cuh"
#include "tracegen.h"
#include "chains.cuh"
#include "hash_to_g2.cuh"
#include "prover.cuh"
#include "verify.cuh"
#include "verify_dev.cuh"

struct pb254_proof {
  prover::ProofData data;
  std::vector<u64> results;  // n_inputs x L limbs (pb254_prove / pb254_prove_dev only)
};

namespace {
thread_local std::string g_last_error;

template <class F>
int guarded(F&& f) {
  try {
    f();
    return PB254_OK;
  } catch (const Pb254Error& e) {
    g_last_error = e.what();
    return e.code;
  } catch (const std::exception& e) {
    g_last_error = e.what();
    return PB254_E_BAD_ARG;
  }
}

// Every call on a context runs its work in this scope, after its argument checks: on the context's device, with an
// empty arena of at least `arena_bytes` and an empty stage list. A call that succeeds drains the stream and reads the
// stage times. One that fails returns without waiting: a failed sharded proof may have left a collective in the stream
// that the other ranks never enqueue.
template <class F>
void on_context(pb254_ctx* c, size_t arena_bytes, F&& body) {
  PbDeviceGuard device_guard(c->device);
  c->arena.reserve(arena_bytes);
  c->arena.reset();
  c->times.clear();
  body();
  pb_sync(c->stream);
  c->times.resolve();
}

int ilog2_strict(size_t n) {
  int k = 0;
  while (((size_t)1 << k) < n) k++;
  if (((size_t)1 << k) != n) throw Pb254Error(PB254_E_BAD_ARG, "size is not a power of two");
  return k;
}

// One argument check for every extern "C" entry: never dereference before these pass (PB254_E_BAD_ARG).
void need(bool ok, const char* what) {
  if (!ok) throw Pb254Error(PB254_E_BAD_ARG, what);
}
void need_ctx(const pb254_ctx* c) { need(c != nullptr, "null context"); }
bool valid_kind(int kind) { return kind >= 0 && kind <= 2; }
void need_kind(int kind) { need(valid_kind(kind), "unknown STARK kind (0 = G1, 1 = G2, 2 = Fq)"); }
// trace heights: a power of two, at least 2^16 (the range-check table needs 65536 rows) and at most 2^26
int need_trace_rows(size_t n_rows) {
  int k = 0;
  while (k < 27 && ((size_t)1 << k) < n_rows) k++;
  need(((size_t)1 << k) == n_rows && k >= 16 && k <= 26, "trace height must be a power of two in 2^16 .. 2^26");
  return k;
}
pb254_config config_or_default(const pb254_config* cfg_in, int log_rows) {
  pb254_config cfg;
  if (cfg_in)
    cfg = *cfg_in;
  else
    pb254_config_standard_fast(&cfg);
  prover::validate_config(cfg);
  if (log_rows >= 0) need(cfg.cap_height <= (unsigned)log_rows + cfg.rate_bits, "cap_height larger than log2 of the LDE size");
  return cfg;
}

void throw_trace_error(int herr) {
  if (herr == tg::ERR_NOT_ON_CURVE)
    throw Pb254Error(PB254_E_NOT_ON_CURVE, "an input point is not on the curve (G1: y^2 = x^3 + 3, G2: y^2 = x^3 + 3/(9+u))");
  if (herr == tg::ERR_NOT_CANONICAL) throw Pb254Error(PB254_E_NOT_CANONICAL, "input coordinate >= p");
  if (herr == tg::ERR_INFINITY)
    throw Pb254Error(PB254_E_INFINITY, "an intermediate sum is the point at infinity (a = -b), unsupported by design");
  if (herr) throw Pb254Error(PB254_E_BAD_ARG, "trace generation: witness consistency check failed");
}

// results[k][i] = limb i of the `sum` / `product` register at the last row of instance k: s * x + offset (x^s)
struct GatherResultsK {
  const u64* trace;
  u64* out;
  size_t n_rows;
  int reg1, L;
  PB_HD void operator()(size_t gid) const {
    size_t k = gid / L;
    int i = (int)(gid % L);
    out[gid] = trace[(size_t)(reg1 + i) * n_rows + k * tg::PERIOD + (tg::PERIOD - 1)];
  }
};

// The chains of pb254_scalar_mul_chains on device buffers (terms, starts and offsets uploaded, d_rows and d_sums
// allocated; d_sums may be null), with scratch from the arena. Decodes the errors (the host chain_starts name the
// failing chain and term) and copies the rows and sums to whichever of inputs_out / sums_out is non-null.
template <class F>
void run_chains(pb254_ctx* c, const u64* d_terms, const u64* d_starts, const u64* d_offsets, size_t n_terms,
                const u64* chain_starts, size_t n_chains, u64* d_rows, u64* d_sums, u64* inputs_out, u64* sums_out) {
  const size_t FW = tg::FieldIO<F>::WORDS, RW = 4 + 4 * FW, n = n_terms + n_chains;
  const pbStream s = c->stream;
  chains::Bufs<F> B;
  B.terms = d_terms;
  B.starts = d_starts;
  B.offsets = d_offsets;
  B.D = c->arena.alloc_n<bn::Jac<F>>(256 * n_terms);
  B.E = c->arena.alloc_n<bn::Jac<F>>(n);
  B.head = c->arena.alloc_n<int>(n);
  B.A = c->arena.alloc_n<bn::Aff<F>>(n);
  B.err = c->arena.alloc_n<int>(1);
  B.first_inf = c->arena.alloc_n<unsigned>(1);
  B.n_terms = n_terms;
  B.n_chains = n_chains;
  pb_memset(B.err, 0, sizeof(int), s);
  pb_memset(B.first_inf, 0xff, sizeof(unsigned), s);
  chains::run<F>(c, B, d_rows, d_sums);
  int herr = 0;
  unsigned first_inf = chains::NO_INF;
  pb_d2h(&herr, B.err, sizeof(int), s);
  pb_d2h(&first_inf, B.first_inf, sizeof(unsigned), s);
  pb_sync(s);
  if (herr == tg::ERR_NOT_CANONICAL || herr == tg::ERR_NOT_ON_CURVE) throw_trace_error(herr);
  if (first_inf != chains::NO_INF) {
    // element e = i + ch + 1 holds the accumulator after term i of chain ch
    size_t ch = 0;
    while (ch + 1 < n_chains && chain_starts[ch + 1] + ch + 1 <= first_inf) ch++;
    const size_t i = first_inf - ch - 1;
    throw Pb254Error(PB254_E_INFINITY, "chain " + std::to_string(ch) + ", term " + std::to_string(i) + " (index " +
                                           std::to_string(i - chain_starts[ch]) +
                                           " in the chain): the accumulator s*x + offset is the point at infinity, "
                                           "unsupported by design");
  }
  throw_trace_error(herr);
  if (n_terms && inputs_out) pb_d2h(inputs_out, d_rows, n_terms * RW * 8, s);
  if (sums_out) pb_d2h(sums_out, d_sums, n_chains * 2 * FW * 8, s);
}

template <class F>
void scalar_mul_chains_impl(pb254_ctx* c, const u64* terms, size_t n_terms, const u64* chain_starts, size_t n_chains,
                            const u64* offsets, u64* inputs_out, u64* sums_out) {
  const size_t FW = tg::FieldIO<F>::WORDS, TW = 4 + 2 * FW, RW = TW + 2 * FW;
  const size_t bytes = chains::scratch_bytes<F>(n_terms, n_chains) +
                       (n_terms * (TW + RW) + (n_chains + 1) + 2 * n_chains * 2 * FW) * 8 + 65536;
  on_context(c, bytes, [&] {
    const pbStream s = c->stream;
    u64* d_terms = c->arena.alloc_n<u64>(n_terms * TW);
    u64* d_starts = c->arena.alloc_n<u64>(n_chains + 1);
    u64* d_offsets = c->arena.alloc_n<u64>(n_chains * 2 * FW);
    u64* d_rows = c->arena.alloc_n<u64>(n_terms * RW);
    u64* d_sums = sums_out ? c->arena.alloc_n<u64>(n_chains * 2 * FW) : nullptr;
    if (n_terms) pb_h2d(d_terms, terms, n_terms * TW * 8, s);
    pb_h2d(d_starts, chain_starts, (n_chains + 1) * 8, s);
    pb_h2d(d_offsets, offsets, n_chains * 2 * FW * 8, s);
    run_chains<F>(c, d_terms, d_starts, d_offsets, n_terms, chain_starts, n_chains, d_rows, d_sums, inputs_out,
                  sums_out);
  });
}

// the lowest failing message (or u) of each h2g2::BAD_* slot, checked in stage order
void throw_h2g2_error(const unsigned bad[h2g2::N_BAD]) {
  static const struct {
    int code;
    const char* what;
  } kinds[h2g2::N_BAD] = {
      {PB254_E_NOT_CANONICAL, "a message element >= the Goldilocks prime or a u coordinate >= p"},
      {PB254_E_BAD_ARG, "exceptional u of the SvdW map (tv1 * tv2 = 0)"},
      {PB254_E_BAD_ARG, "the offset scalar k is 0 mod r"},
      {PB254_E_INFINITY, "cofactor * x is the point at infinity"},
  };
  for (int k = 0; k < h2g2::N_BAD; k++)
    if (bad[k] != chains::NO_INF)
      throw Pb254Error(kinds[k].code, "index " + std::to_string(bad[k]) + ": " + kinds[k].what);
}
void check_h2g2(pb254_ctx* c, const unsigned* d_bad) {
  unsigned bad[h2g2::N_BAD];
  pb_d2h(bad, d_bad, sizeof(bad), c->stream);
  pb_sync(c->stream);
  throw_h2g2_error(bad);
}

void map_to_g2_impl(pb254_ctx* c, const u64* us, size_t n, u64* points_out) {
  on_context(c, n * (8 * 8 + sizeof(h2g2::Fq2) + sizeof(h2g2::Aff) + 16 * 8) + 65536, [&] {
    const pbStream s = c->stream;
    u64* d_us = c->arena.alloc_n<u64>(n * 8);
    h2g2::Fq2* d_u = c->arena.alloc_n<h2g2::Fq2>(n);
    h2g2::Aff* d_pts = c->arena.alloc_n<h2g2::Aff>(n);
    u64* d_out = c->arena.alloc_n<u64>(n * 16);
    unsigned* d_bad = c->arena.alloc_n<unsigned>(h2g2::N_BAD);
    pb_h2d(d_us, us, n * 64, s);
    pb_memset(d_bad, 0xff, h2g2::N_BAD * sizeof(unsigned), s);
    const int t0 = c->times.begin("h2g2 map", s);
    pb_launch("h2g2 load u", h2g2::LoadUK{d_us, d_u, d_bad}, n, s, 128);
    pb_launch("h2g2 map", h2g2::MapK{d_u, d_pts, d_bad}, n, s, 128);
    pb_launch("h2g2 points", h2g2::PutK{d_pts, d_out, 16}, n, s, 128);
    c->times.end(t0, s);
    check_h2g2(c, d_bad);
    pb_d2h(points_out, d_out, n * 128, s);
  });
}

void hash_to_g2_impl(pb254_ctx* c, const u64* messages, size_t n, size_t msg_len, u64 seed, u64* inputs_out,
                     u64* hashes_out) {
  using namespace h2g2;
  typedef bn::F2 F;
  const size_t TW = 20, RW = 36, PW = 16;
  const size_t bytes = chains::scratch_bytes<F>(n, n) + n * msg_len * 8 +
                       n * (sizeof(Fq2) + 2 * sizeof(Aff) + 2 * sizeof(Jac) + (TW + 4 + PW + 1 + RW + 2 * PW) * 8) +
                       65536;
  on_context(c, bytes, [&] {
    const pbStream s = c->stream;
    if (!c->g2_pow2) {
      c->g2_pow2 = pb_dev_alloc(TABLE_POINTS * sizeof(Jac));
      pb_launch("h2g2 table", TableK{(Jac*)c->g2_pow2}, 1, s, 32);
    }
    u64* d_msgs = c->arena.alloc_n<u64>(n * msg_len + 1);
    Fq2* d_u = c->arena.alloc_n<Fq2>(n);
    Aff* d_pts = c->arena.alloc_n<Aff>(n);
    u64* d_terms = c->arena.alloc_n<u64>(n * TW);
    u64* d_k = c->arena.alloc_n<u64>(n * 4);
    Jac* d_jac = c->arena.alloc_n<Jac>(n);
    u64* d_offsets = c->arena.alloc_n<u64>(n * PW);
    u64* d_starts = c->arena.alloc_n<u64>(n + 1);
    u64* d_rows = c->arena.alloc_n<u64>(n * RW);
    u64* d_sums = c->arena.alloc_n<u64>(n * PW);
    u64* d_hashes = c->arena.alloc_n<u64>(n * PW);
    unsigned* d_bad = c->arena.alloc_n<unsigned>(N_BAD);
    int* d_err = c->arena.alloc_n<int>(1);  // the affine passes' flag: their points are never at infinity (d_bad)
    std::vector<u64> starts(n + 1);
    for (size_t i = 0; i <= n; i++) starts[i] = i;
    if (msg_len) pb_h2d(d_msgs, messages, n * msg_len * 8, s);
    pb_h2d(d_starts, starts.data(), (n + 1) * 8, s);
    pb_memset(d_bad, 0xff, N_BAD * sizeof(unsigned), s);
    pb_memset(d_err, 0, sizeof(int), s);

    int t = c->times.begin("h2g2 hash", s);
    pb_launch("h2g2 hash", HashK{d_msgs, msg_len, d_u, d_bad}, n, s, 128);
    c->times.end(t, s);
    t = c->times.begin("h2g2 map", s);
    pb_launch("h2g2 map", MapK{d_u, d_pts, d_bad}, n, s, 128);
    pb_launch("h2g2 terms", CofactorK{d_terms}, n, s, 128);
    pb_launch("h2g2 points", PutK{d_pts, d_terms + 4, TW}, n, s, 128);
    c->times.end(t, s);
    t = c->times.begin("h2g2 offsets", s);
    pb_launch("h2g2 draw", DrawK{seed, d_k, d_bad}, n, s, 128);
    fixed_base((const Jac*)c->g2_pow2, d_k, n, d_jac, s);
    chains::to_affine<F>(d_jac, d_pts, n, d_err, s);
    pb_launch("h2g2 offsets out", PutK{d_pts, d_offsets, PW}, n, s, 128);
    c->times.end(t, s);
    check_h2g2(c, d_bad);

    run_chains<F>(c, d_terms, d_starts, d_offsets, n, starts.data(), n, d_rows, d_sums, inputs_out, nullptr);

    t = c->times.begin("h2g2 outputs", s);
    pb_launch("h2g2 sub offset", SubOffsetK{d_sums, d_offsets, d_jac, d_bad}, n, s, 128);
    chains::to_affine<F>(d_jac, d_pts, n, d_err, s);
    pb_launch("h2g2 hashes out", PutK{d_pts, d_hashes, PW}, n, s, 128);
    c->times.end(t, s);
    check_h2g2(c, d_bad);
    pb_d2h(hashes_out, d_hashes, n * PW * 8, s);
  });
}

struct PermuteK {
  const u64* in;
  u64* out;
  PB_HD void operator()(size_t i) const {
    u64 s[12];
    for (int k = 0; k < 12; k++) s[k] = in[i * 12 + k];
    poseidon::permute(s);
    for (int k = 0; k < 12; k++) out[i * 12 + k] = s[k];
  }
};

// One proof on context c (pb254_prove, _dev, _sharded and _trace). The arena holds the trace words, then either the
// scratch of `fill` or the prover's workspace. fill(d_trace, results) writes the trace, and the native results where
// the caller has them, with arena space after the trace that the prover reuses.
template <class Fill>
void prove_filled(pb254_ctx* c, int kind, size_t n_rows, const pb254_config& cfg, bool keep_debug,
                  const pb254_comm* comm, bool trace_is_block, size_t trace_words, size_t fill_bytes, Fill&& fill,
                  pb254_proof** out) {
  const size_t workspace = comm ? prover::workspace_bytes_sharded(kind, n_rows, cfg, comm->world)
                                : prover::workspace_bytes(kind, n_rows, cfg);
  size_t bytes = trace_words * 8 + std::max(fill_bytes, workspace) + 65536;
#if !PB_HOSTSIM
  if (trace_is_block) {  // the estimate is an upper bound: never ask for more than the device has left (the
                         // collectives of the caller need room too); a proof that really does not fit fails in
                         // Arena::alloc with PB254_E_OOM
    const size_t avail = pb_free_bytes(c->device) + c->arena.cap, margin = (size_t)4 << 30;
    if (avail > margin && bytes > avail - margin) bytes = avail - margin;
  }
#endif
  std::unique_ptr<pb254_proof> pf(new pb254_proof());
  on_context(c, bytes, [&] {
    u64* d_trace = c->arena.alloc_n<u64>(trace_words);
    const size_t mark = c->arena.off;
    fill(d_trace, pf->results);
    c->arena.off = mark;
    prover::prove_device(c, kind, d_trace, n_rows, cfg, pf->data, keep_debug, comm, trace_is_block);
  });
  *out = pf.release();
}

// Whether every rank of a sharded proof can generate only ITS instances: the trace splits into per-rank row blocks of
// whole instances that each hold the 2^16-row range-check table or none of it (every BASELINE size does). Otherwise
// (small traces) every rank generates the whole trace.
bool generate_by_instance(size_t n_rows, size_t world) {
  return n_rows % world == 0 && (n_rows / world) % tg::PERIOD == 0 && n_rows / world >= 65536;
}

// generate_trace + prove in one call: what run_once does between src/generators/g1/stark_proof.rs:154 and :163. The
// trace never leaves the device. comm: one proof across its ranks (include/pb254.h); NULL or world 1 is one GPU.
int prove_inputs(pb254_ctx* c, int kind, const u64* inputs, const u64* timestamps, size_t n_inputs, size_t min_rows,
                 const pb254_config* cfg_in, int keep_debug, pb254_proof** out, bool inputs_on_device,
                 const pb254_comm* comm = nullptr) {
  return guarded([&] {
    need(out != nullptr, "null out pointer");
    need_ctx(c);
    need_kind(kind);
    need(inputs && timestamps && n_inputs > 0, "null or empty input");
    need(!comm || (comm->world && (comm->world & (comm->world - 1)) == 0 && comm->rank < comm->world &&
                   comm->all_to_all && comm->all_gather),
         "comm: world must be a power of two, rank < world, callbacks non-null");
    if (comm && comm->world == 1) comm = nullptr;
    const tg::Layout l = tg::layout_for(kind);
    const size_t n_rows = pb254_trace_rows(n_inputs, min_rows);
    const pb254_config cfg = config_or_default(cfg_in, need_trace_rows(n_rows));
    if (comm && generate_by_instance(n_rows, comm->world)) {
      // this rank's row block [rank n / P, (rank + 1) n / P) of the trace, [ceil(W / P) P columns][n / P]
      const size_t P = comm->world, rk = comm->rank, nloc = n_rows / P;
      const size_t per = nloc / tg::PERIOD;  // instances per rank
      const size_t i0 = std::min(n_inputs, rk * per), i1 = std::min(n_inputs, (rk + 1) * per), kloc = i1 - i0;
      const size_t Wpad = ((size_t)l.width + P - 1) / P * P;
      const size_t tg_bytes =
          tg::scratch_bytes(kind, kloc ? kloc : 1) + (kloc + 1) * (l.in_words + 1) * 8 + (P + 1) * 65536 * 8 + 65536;
      // no native results in this mode: they are spread over the ranks
      prove_filled(c, kind, n_rows, cfg, keep_debug != 0, comm, true, Wpad * nloc, tg_bytes,
                   [&](u64* d_rows, std::vector<u64>&) {
        prover::Stage st(c, "tracegen");
        u64* d_in = c->arena.alloc_n<u64>(kloc * l.in_words + 1);
        u64* d_ts = c->arena.alloc_n<u64>(kloc + 1);
        if (kloc) {
          pb_h2d(d_in, inputs + i0 * l.in_words, kloc * l.in_words * 8, c->stream);
          pb_h2d(d_ts, timestamps + i0, kloc * 8, c->stream);
        }
        int* d_err = c->arena.alloc_n<int>(1);
        pb_memset(d_err, 0, sizeof(int), c->stream);
        tg::generate(c->arena, kind, d_in, d_ts, kloc, nloc, d_rows, d_err, c->stream, rk * nloc);
        // range-check frequencies: every block counted its own cells into the first 2^16 rows of its frequency
        // column; the table rows are rows 0 .. 65535 of the whole trace, i.e. of rank 0's block
        u64* freq = d_rows + (size_t)l.freq * nloc;
        u64* all = c->arena.alloc_n<u64>(P * 65536);
        if (comm->all_gather(comm->user, freq, all, 65536 * 8)) throw Pb254Error(PB254_E_CUDA, "collective failed: all_gather");
        if (rk == 0)
          pb_launch("sum histograms", prover::SumRecordsK{all, freq, 65536, (int)P}, 65536, c->stream, 128);
        else
          pb_memset(freq, 0, 65536 * 8, c->stream);
        // an input error on one rank must fail the call on every rank (the others would wait in the next collective)
        u64* e_mine = c->arena.alloc_n<u64>(1);
        u64* e_all = c->arena.alloc_n<u64>(P);
        pb_memset(e_mine, 0, 8, c->stream);
        pb_d2d(e_mine, d_err, sizeof(int), c->stream);
        if (comm->all_gather(comm->user, e_mine, e_all, 8)) throw Pb254Error(PB254_E_CUDA, "collective failed: all_gather");
        std::vector<u64> herr(P);
        pb_d2h(herr.data(), e_all, P * 8, c->stream);
        pb_sync(c->stream);
        for (size_t p = 0; p < P; p++) throw_trace_error((int)(herr[p] & 0xffffffffu));
      }, out);
    } else {
      const size_t tg_bytes = tg::scratch_bytes(kind, n_inputs) + n_inputs * (l.in_words + 1) * 8 + 65536;
      prove_filled(c, kind, n_rows, cfg, keep_debug != 0, comm, false, (size_t)l.width * n_rows, tg_bytes,
                   [&](u64* d_trace, std::vector<u64>& results) {
        prover::Stage st(c, "tracegen");
        const u64 *d_in = inputs, *d_ts = timestamps;
        if (!inputs_on_device) {
          u64* hin = c->arena.alloc_n<u64>(n_inputs * l.in_words + 1);
          u64* hts = c->arena.alloc_n<u64>(n_inputs + 1);
          pb_h2d(hin, inputs, n_inputs * l.in_words * 8, c->stream);
          pb_h2d(hts, timestamps, n_inputs * 8, c->stream);
          d_in = hin;
          d_ts = hts;
        }
        int* d_err = c->arena.alloc_n<int>(1);
        pb_memset(d_err, 0, sizeof(int), c->stream);
        tg::generate(c->arena, kind, d_in, d_ts, n_inputs, n_rows, d_trace, d_err, c->stream);
        int herr = 0;
        pb_d2h(&herr, d_err, sizeof(int), c->stream);
        u64* d_res = c->arena.alloc_n<u64>(n_inputs * l.L);
        pb_launch("gather results", GatherResultsK{d_trace, d_res, n_rows, l.reg1, l.L}, n_inputs * l.L, c->stream,
                  128);
        results.resize(n_inputs * l.L);
        pb_d2h(results.data(), d_res, results.size() * 8, c->stream);
        pb_sync(c->stream);
        throw_trace_error(herr);
      }, out);
    }
  });
}

// the keep_debug artefacts of include/pb254.h; slot 4 and any other slot are empty
const std::vector<u64>* debug_slot(const pb254_proof* p, int which) {
  const prover::ProofData& d = p->data;
  const std::vector<u64>* slots[] = {&d.dbg_aux, &d.dbg_chunks, &d.dbg_challenges, &d.dbg_indices, nullptr,
                                     &d.dbg_groups};
  return which >= 0 && which < 6 ? slots[which] : nullptr;
}
}  // namespace

extern "C" {

void pb254_config_standard_fast(pb254_config* c) {
  c->rate_bits = 1;
  c->cap_height = 4;
  c->num_challenges = 2;
  c->num_query_rounds = 84;
  c->pow_bits = 16;
  c->arity_bits = 4;
  c->final_poly_bits = 5;
}

const char* pb254_last_error(void) { return g_last_error.c_str(); }
uint64_t pb254_launch_count(void) { return g_pb_launches.load(); }

int pb254_ctx_create(int device, void* stream, pb254_ctx** out) {
  return guarded([&] {
    need(out != nullptr, "null out pointer");
    std::unique_ptr<pb254_ctx> c(new pb254_ctx());
    c->device = device;
    // the first call on the new context: no arena yet, and tables.init has drained the stream already
    on_context(c.get(), 0, [&] {
#if PB_HOSTSIM
      c->stream = stream;
#else
      if (stream) {
        c->stream = (cudaStream_t)stream;
      } else {
        PB_CUDA(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
        c->own_stream = true;
      }
#endif
      c->tables.init(c->stream);
    });
    *out = c.release();
  });
}

void pb254_ctx_destroy(pb254_ctx* c) {
  if (!c) return;
  c->tables.destroy();
  c->arena.destroy();
  if (c->g2_pow2) pb_dev_free(c->g2_pow2);
#if !PB_HOSTSIM
  if (c->own_stream) cudaStreamDestroy(c->stream);
#endif
  delete c;
}

/* stage timings of the last call on this context (device time, ms) */
int pb254_timing_count(pb254_ctx* c) { return c ? (int)c->times.recs.size() : 0; }
const char* pb254_timing_name(pb254_ctx* c, int i) {
  return c && i >= 0 && i < (int)c->times.recs.size() ? c->times.recs[i].name.c_str() : "";
}
double pb254_timing_ms(pb254_ctx* c, int i) {
  return c && i >= 0 && i < (int)c->times.recs.size() ? c->times.recs[i].ms : 0.0;
}

int pb254_trace_width(int kind) { return valid_kind(kind) ? tg::layout_for(kind).width : -1; }
int pb254_input_words(int kind) { return valid_kind(kind) ? tg::layout_for(kind).in_words : -1; }
int pb254_num_aux(int kind, uint32_t nch) {
  return valid_kind(kind) ? aux::num_aux(tg::layout_for(kind), (int)nch) : -1;
}
size_t pb254_trace_rows(size_t n_inputs, size_t min_rows) {
  size_t n = n_inputs * 512 > min_rows ? n_inputs * 512 : min_rows, r = 1;
  while (r < n) r <<= 1;
  return r;
}

int pb254_poseidon_permute(pb254_ctx* c, const uint64_t* in, size_t n, uint64_t* out) {
  return guarded([&] {
    need_ctx(c);
    on_context(c, 2 * n * 96 + 1024, [&] {
      u64* din = c->arena.alloc_n<u64>(n * 12);
      u64* dout = c->arena.alloc_n<u64>(n * 12);
      pb_h2d(din, in, n * 96, c->stream);
      pb_launch("poseidon permute", PermuteK{din, dout}, n, c->stream, 128);
      pb_d2h(out, dout, n * 96, c->stream);
    });
  });
}

int pb254_lde_batch(pb254_ctx* c, const uint64_t* values, size_t cols, size_t n, uint32_t rate_bits, int from_coeffs,
                    uint64_t* lde_out) {
  return guarded([&] {
    need_ctx(c);
    int L = ilog2_strict(n);
    size_t N = n << rate_bits;
    on_context(c, (2 * cols * n + cols * N) * 8 + 4096, [&] {
      u64* dv = c->arena.alloc_n<u64>(cols * n);
      u64* scratch = c->arena.alloc_n<u64>(cols * n);
      u64* lde = c->arena.alloc_n<u64>(cols * N);
      pb_h2d(dv, values, cols * n * 8, c->stream);
      ntt::lde_columns(c->tables, dv, n, lde, N, scratch, (int)cols, L, (int)rate_bits,
                       from_coeffs ? ntt::FROM_COEFFS_LDE : ntt::FROM_VALUES_LDE, c->stream);
      pb_d2h(lde_out, lde, cols * N * 8, c->stream);
    });
  });
}

int pb254_commit(pb254_ctx* c, const uint64_t* values, size_t cols, size_t n, uint32_t rate_bits, uint32_t cap_height,
                 int from_coeffs, uint64_t* cap_out, uint64_t* digests_out) {
  return guarded([&] {
    need_ctx(c);
    int L = ilog2_strict(n);
    size_t N = n << rate_bits;
    int log_N = L + (int)rate_bits;
    size_t nd = merkle::tree_digests(log_N, (int)cap_height);
    on_context(c, (2 * cols * n + cols * N) * 8 + nd * 32 + 4096, [&] {
      u64* dv = c->arena.alloc_n<u64>(cols * n);
      u64* scratch = c->arena.alloc_n<u64>(cols * n);
      u64* lde = c->arena.alloc_n<u64>(cols * N);
      merkle::Digest* dig = c->arena.alloc_n<merkle::Digest>(nd);
      pb_h2d(dv, values, cols * n * 8, c->stream);
      int t0 = c->times.begin("lde", c->stream);
      ntt::lde_columns(c->tables, dv, n, lde, N, scratch, (int)cols, L, (int)rate_bits,
                       from_coeffs ? ntt::FROM_COEFFS_LDE : ntt::FROM_VALUES_LDE, c->stream);
      c->times.end(t0, c->stream);
      int t1 = c->times.begin("merkle", c->stream);
      merkle::build_from_lde(lde, N, (int)cols, log_N, (int)cap_height, dig, c->stream);
      c->times.end(t1, c->stream);
      size_t ncap = (size_t)1 << cap_height;
      pb_d2h(cap_out, dig + (nd - ncap), ncap * 32, c->stream);
      if (digests_out) pb_d2h(digests_out, dig, nd * 32, c->stream);
    });
  });
}

int pb254_generate_trace(pb254_ctx* c, int kind, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs,
                         size_t min_rows, uint64_t* cols_out) {
  return guarded([&] {
    need_ctx(c);
    need_kind(kind);
    need(inputs && timestamps && cols_out && n_inputs > 0, "null or empty argument");
    tg::Layout l = tg::layout_for(kind);
    size_t n_rows = pb254_trace_rows(n_inputs, min_rows);
    need_trace_rows(n_rows);
    size_t tbytes = (size_t)l.width * n_rows * 8;
    int herr = 0;
    on_context(c, tbytes + tg::scratch_bytes(kind, n_inputs) + n_inputs * (l.in_words + 1) * 8 + 65536, [&] {
      u64* d_trace = c->arena.alloc_n<u64>((size_t)l.width * n_rows);
      u64* d_in = c->arena.alloc_n<u64>(n_inputs * l.in_words + 1);
      u64* d_ts = c->arena.alloc_n<u64>(n_inputs + 1);
      int* d_err = c->arena.alloc_n<int>(1);
      pb_h2d(d_in, inputs, n_inputs * l.in_words * 8, c->stream);
      pb_h2d(d_ts, timestamps, n_inputs * 8, c->stream);
      pb_memset(d_err, 0, sizeof(int), c->stream);
      int t0 = c->times.begin("tracegen", c->stream);
      tg::generate(c->arena, kind, d_in, d_ts, n_inputs, n_rows, d_trace, d_err, c->stream);
      c->times.end(t0, c->stream);
      pb_d2h(&herr, d_err, sizeof(int), c->stream);
      pb_d2h(cols_out, d_trace, tbytes, c->stream);
    });
    throw_trace_error(herr);
  });
}

int pb254_scalar_mul_chains(pb254_ctx* c, int kind, const uint64_t* terms, size_t n_terms,
                            const uint64_t* chain_starts, size_t n_chains, const uint64_t* offsets,
                            uint64_t* inputs_out, uint64_t* sums_out) {
  return guarded([&] {
    need_ctx(c);
    need(kind == PB254_KIND_G1 || kind == PB254_KIND_G2, "kind must be PB254_KIND_G1 or PB254_KIND_G2");
    need(chain_starts != nullptr, "null chain_starts");
    need(n_terms <= chains::MAX_TERMS && n_chains <= chains::MAX_CHAINS, "more than 2^17 terms or chains");
    need(n_terms == 0 || (terms && inputs_out), "null terms or inputs_out");
    need(n_chains == 0 || offsets, "null offsets");
    need(chain_starts[0] == 0 && chain_starts[n_chains] == n_terms,
         "chain_starts must begin at 0 and end at n_terms");
    for (size_t k = 0; k < n_chains; k++) need(chain_starts[k] <= chain_starts[k + 1], "chain_starts must not decrease");
    if (n_chains == 0) return;
    if (kind == PB254_KIND_G1)
      scalar_mul_chains_impl<bn::F1>(c, terms, n_terms, chain_starts, n_chains, offsets, inputs_out, sums_out);
    else
      scalar_mul_chains_impl<bn::F2>(c, terms, n_terms, chain_starts, n_chains, offsets, inputs_out, sums_out);
  });
}

int pb254_map_to_g2(pb254_ctx* c, const uint64_t* us, size_t n, uint64_t* points_out) {
  return guarded([&] {
    need_ctx(c);
    need(n <= h2g2::MAX_N, "more than 2^17 values");
    if (n == 0) return;
    need(us && points_out, "null us or points_out");
    map_to_g2_impl(c, us, n, points_out);
  });
}

int pb254_hash_to_g2(pb254_ctx* c, const uint64_t* messages, size_t n, size_t msg_len, uint64_t seed,
                     uint64_t* inputs_out, uint64_t* hashes_out) {
  return guarded([&] {
    need_ctx(c);
    need(n <= h2g2::MAX_N, "more than 2^17 messages");
    need(msg_len <= h2g2::MAX_MSG_ELEMS && n * msg_len <= h2g2::MAX_MSG_ELEMS, "more than 2^24 message elements");
    if (n == 0) return;
    need((messages || msg_len == 0) && inputs_out && hashes_out, "null messages, inputs_out or hashes_out");
    hash_to_g2_impl(c, messages, n, msg_len, seed, inputs_out, hashes_out);
  });
}

int pb254_prove_sharded(pb254_ctx* c, int kind, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs,
                        size_t min_rows, const pb254_config* cfg_in, const pb254_comm* comm, pb254_proof** out) {
  return prove_inputs(c, kind, inputs, timestamps, n_inputs, min_rows, cfg_in, 0, out, false, comm);
}

int pb254_prove(pb254_ctx* c, int kind, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs,
                size_t min_rows, const pb254_config* cfg, int keep_debug, pb254_proof** out) {
  return prove_inputs(c, kind, inputs, timestamps, n_inputs, min_rows, cfg, keep_debug, out, false);
}

int pb254_prove_many(pb254_ctx* const* ctxs, size_t n_ctx, int kind, const uint64_t* inputs, const uint64_t* timestamps,
                     size_t n_inputs, size_t n_batches, size_t min_rows, const pb254_config* cfg, pb254_proof** proofs_out) {
  int rc = guarded([&] {
    need(ctxs && n_ctx > 0 && n_ctx <= 16 && proofs_out, "null contexts / outputs or more than 16 contexts");
    need_kind(kind);
    need(inputs && timestamps && n_inputs > 0, "null or empty input");
    for (size_t t = 0; t < n_ctx; t++) {
      need_ctx(ctxs[t]);
      for (size_t u = 0; u < t; u++) need(ctxs[u] != ctxs[t], "the same context twice");
    }
  });
  if (rc) return rc;
  const size_t in_words = (size_t)tg::layout_for(kind).in_words;
  for (size_t b = 0; b < n_batches; b++) proofs_out[b] = nullptr;
  std::vector<int> codes(n_ctx, 0);
  std::vector<std::string> messages(n_ctx);
  std::vector<std::thread> workers;
  for (size_t t = 0; t < n_ctx; t++)
    workers.emplace_back([&, t] {
      for (size_t b = t; b < n_batches && !codes[t]; b += n_ctx) {
        codes[t] = pb254_prove(ctxs[t], kind, inputs + b * n_inputs * in_words, timestamps + b * n_inputs, n_inputs,
                               min_rows, cfg, 0, &proofs_out[b]);
        if (codes[t]) messages[t] = pb254_last_error();  // thread-local in this worker
      }
    });
  for (auto& w : workers) w.join();
  for (size_t t = 0; t < n_ctx; t++)
    if (codes[t]) {
      for (size_t b = 0; b < n_batches; b++) {
        if (proofs_out[b]) pb254_proof_free(proofs_out[b]);
        proofs_out[b] = nullptr;
      }
      g_last_error = messages[t];
      return codes[t];
    }
  return PB254_OK;
}

// Same with `inputs` / `timestamps` already resident in device memory of the context's GPU.
int pb254_prove_dev(pb254_ctx* c, int kind, const uint64_t* d_inputs, const uint64_t* d_timestamps, size_t n_inputs,
                    size_t min_rows, const pb254_config* cfg, int keep_debug, pb254_proof** out) {
  return prove_inputs(c, kind, d_inputs, d_timestamps, n_inputs, min_rows, cfg, keep_debug, out, true);
}

// prove(stark, config, trace, ...) on a host trace (column-major width x n_rows), the literal
// signature of src/starks/common/prover.rs:18-30.
int pb254_prove_trace(pb254_ctx* c, int kind, const uint64_t* trace_cols, size_t n_rows, const pb254_config* cfg_in,
                      int keep_debug, pb254_proof** out) {
  return guarded([&] {
    need(out != nullptr, "null out pointer");
    need_ctx(c);
    need_kind(kind);
    need(trace_cols != nullptr, "null trace");
    const pb254_config cfg = config_or_default(cfg_in, need_trace_rows(n_rows));
    const tg::Layout l = tg::layout_for(kind);
    const size_t twords = (size_t)l.width * n_rows;
    prove_filled(c, kind, n_rows, cfg, keep_debug != 0, nullptr, false, twords, 0,
                 [&](u64* d_trace, std::vector<u64>&) {
      pb_h2d(d_trace, trace_cols, twords * 8, c->stream);
      // A host-supplied trace has not been through generate_range_checks: every looked-up cell and the table column
      // must be < 2^16 (the reference asserts this while filling the frequency column, g1/scalar_mul_stark.rs:71-87).
      int* d_err = c->arena.alloc_n<int>(1);
      pb_memset(d_err, 0, sizeof(int), c->stream);
      pb_launch("range pre-check", aux::RangePrecheckK{d_trace, n_rows, l.rc_lo, l.rc_hi, l.range_counter, d_err},
                n_rows, c->stream, 128);
      int herr = 0;
      pb_d2h(&herr, d_err, sizeof(int), c->stream);
      pb_sync(c->stream);
      if (herr) throw Pb254Error(PB254_E_BAD_ARG, "trace: a range-checked cell or the range counter is >= 2^16");
    }, out);
  });
}

// ---- device-pointer building blocks of the oversized-trace mode (column-sharded LDE -> all-to-all ->
// row-sharded leaf hashing -> digest all-gather -> per-rank subtree), orchestrated by plonky2_bn254_b200/dist.py
int pb254_lde_dev(pb254_ctx* c, const uint64_t* d_values, size_t cols, size_t n, uint32_t rate_bits, int from_coeffs,
                  uint64_t* d_lde_out) {
  return guarded([&] {
    need_ctx(c);
    int L = ilog2_strict(n);
    on_context(c, cols * n * 8 + 4096, [&] {
      u64* scratch = c->arena.alloc_n<u64>(cols * n);
      int t0 = c->times.begin("lde", c->stream);
      ntt::lde_columns(c->tables, d_values, n, d_lde_out, n << rate_bits, scratch, (int)cols, L, (int)rate_bits,
                       from_coeffs ? ntt::FROM_COEFFS_LDE : ntt::FROM_VALUES_LDE, c->stream);
      c->times.end(t0, c->stream);
    });
  });
}

int pb254_leaf_hash_rows_dev(pb254_ctx* c, const uint64_t* d_matrix, size_t stride, size_t cols, size_t rows,
                             uint64_t* d_digests_out) {
  return guarded([&] {
    need_ctx(c);
    on_context(c, 0, [&] {
      int t0 = c->times.begin("leaf hash rows", c->stream);
      merkle::hash_rows_natural(d_matrix, stride, (int)cols, rows, (merkle::Digest*)d_digests_out, c->stream);
      c->times.end(t0, c->stream);
    });
  });
}

// Roots at height `log_sub - log_roots` of the subtree whose leaves are tree positions [first, first + 2^log_sub):
// leaf(q) = d_all_digests[bit_reverse(q, log_total)] (digests of all rows in natural row order).
int pb254_merkle_subtree_dev(pb254_ctx* c, const uint64_t* d_all_digests, uint32_t log_total, size_t first,
                             uint32_t log_sub, uint32_t log_roots, uint64_t* d_roots_out) {
  return guarded([&] {
    need_ctx(c);
    if (log_roots > log_sub || log_sub > log_total) throw Pb254Error(PB254_E_BAD_ARG, "subtree shape");
    size_t nd = merkle::tree_digests((int)log_sub, (int)log_roots);
    on_context(c, nd * 32 + 4096, [&] {
      merkle::Digest* dig = c->arena.alloc_n<merkle::Digest>(nd);
      int t0 = c->times.begin("subtree", c->stream);
      pb_launch("subtree leaves", merkle::SubtreeLeavesK{(const merkle::Digest*)d_all_digests, dig, first, (int)log_total},
                (size_t)1 << log_sub, c->stream, 128);
      merkle::build_levels(dig, (int)log_sub, (int)log_roots, c->stream);
      size_t nr = (size_t)1 << log_roots;
      pb_d2d(d_roots_out, dig + (nd - nr), nr * 32, c->stream);
      c->times.end(t0, c->stream);
    });
  });
}

// verify(stark, config, ctls, proof, [], extra_looking_values) of src/starks/common/verifier.rs:32-98, with the
// extra looking values recomputed natively from the batch as run_once does (g1/scalar_mul_ctl.rs:57-80).
int pb254_verify(int kind, const pb254_config* cfg_in, const uint64_t* proof_words, size_t n_words,
                 const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs) {
  return guarded([&] {
    need_kind(kind);
    need(proof_words && inputs && timestamps, "null argument");
    const pb254_config cfg = config_or_default(cfg_in, -1);
    verify::verify_proof(kind, cfg, proof_words, n_words, inputs, timestamps, n_inputs);
  });
}

// pb254_verify with the native CTL values and the Merkle openings on the context's GPU (verify_dev.cuh): the same walk,
// so the same code and message for every input; PB254_E_CUDA / PB254_E_OOM are the only additional outcomes.
int pb254_verify_device(pb254_ctx* c, int kind, const pb254_config* cfg_in, const uint64_t* proof_words,
                        size_t n_words, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs) {
  return guarded([&] {
    need_ctx(c);
    need_kind(kind);
    need(proof_words && inputs && timestamps, "null argument");
    const pb254_config cfg = config_or_default(cfg_in, -1);
    const uint64_t starts[2] = {0, n_inputs};
    verify_dev::Outcome o;
    // the batch of one: the round's coordinator sizes the arena once the walk knows the proof's shape, and drains the
    // stream before the walk reads its results
    on_context(c, 0, [&] {
      verify_dev::verify_many(c, kind, cfg, &proof_words, &n_words, 1, inputs, timestamps, starts, &o);
    });
    if (o.code) throw Pb254Error(o.code, o.msg);
  });
}

// pb254_verify_device on n_proofs proofs in rounds of verify_dev::ROUND: one launch per stage per round.
int pb254_verify_many_device(pb254_ctx* c, int kind, const pb254_config* cfg_in, const uint64_t* const* proof_words,
                             const size_t* n_words, size_t n_proofs, const uint64_t* inputs, const uint64_t* timestamps,
                             const uint64_t* input_starts, int* codes_out, char* messages_out) {
  std::vector<verify_dev::Outcome> out;
  const int rc = guarded([&] {
    need_ctx(c);
    need_kind(kind);
    need(n_proofs <= verify_dev::MAX_PROOFS, "more than 2^12 proofs");
    need(proof_words && n_words && inputs && timestamps && input_starts && codes_out, "null argument");
    for (size_t b = 0; b < n_proofs; b++) need(proof_words[b] != nullptr, "null proof_words entry");
    need(input_starts[0] == 0, "input_starts[0] must be 0");
    for (size_t b = 0; b < n_proofs; b++) need(input_starts[b] <= input_starts[b + 1], "input_starts must not decrease");
    const pb254_config cfg = config_or_default(cfg_in, -1);
    out.resize(n_proofs);
    try {
      on_context(c, 0, [&] {
        verify_dev::verify_many(c, kind, cfg, proof_words, n_words, n_proofs, inputs, timestamps, input_starts,
                                out.data());
      });
    } catch (const Pb254Error& e) {  // PB254_E_CUDA / PB254_E_OOM fail every proof
      for (auto& o : out) o = verify_dev::Outcome{e.code, e.what()};
      throw;
    }
  });
  if (out.empty()) return rc;  // bad arguments (outputs untouched), or no proofs
  for (size_t b = 0; b < n_proofs; b++) {
    codes_out[b] = out[b].code;
    if (messages_out) {
      char* m = messages_out + b * PB254_VERIFY_MESSAGE_BYTES;
      const size_t len = std::min(out[b].msg.size(), (size_t)PB254_VERIFY_MESSAGE_BYTES - 1);
      memcpy(m, out[b].msg.data(), len);
      m[len] = 0;
    }
  }
  if (rc) return rc;
  for (size_t b = 0; b < n_proofs; b++)
    if (out[b].code) {
      g_last_error = "proof " + std::to_string(b) + ": " + out[b].msg;
      return out[b].code;
    }
  return PB254_OK;
}

void pb254_proof_free(pb254_proof* p) { delete p; }
size_t pb254_proof_results_words(const pb254_proof* p) { return p->results.size(); }
const uint64_t* pb254_proof_results_data(const pb254_proof* p) { return p->results.data(); }
int pb254_proof_parse(const uint64_t* proof_words, size_t n_words, pb254_proof_layout* out) {
  return guarded([&] {
    if (!proof_words || !out) throw Pb254Error(PB254_E_BAD_ARG, "null argument");
    proofview::parse(proof_words, n_words, *out);
  });
}

size_t pb254_proof_words(const pb254_proof* p) { return p->data.blob.size(); }
const uint64_t* pb254_proof_data(const pb254_proof* p) { return p->data.blob.data(); }
size_t pb254_proof_debug_words(const pb254_proof* p, int which) {
  const std::vector<u64>* v = debug_slot(p, which);
  return v ? v->size() : 0;
}
const uint64_t* pb254_proof_debug_data(const pb254_proof* p, int which) {
  const std::vector<u64>* v = debug_slot(p, which);
  return v ? v->data() : nullptr;
}

}  // extern "C"
