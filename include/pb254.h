/* pb254.h — C ABI of the B200-native starky prover for plonky2_bn254's BN254 STARKs.
 *
 * Drop-in boundary (SURVEY.md §8b): the entry points below are what an FFI crate binds in place of
 * the bodies of
 *   G1ScalarMulStark::generate_trace   src/starks/curves/g1/scalar_mul_stark.rs:55-69
 *   G2ScalarMulStark::generate_trace   src/starks/curves/g2/scalar_mul_stark.rs:55-69
 *   FqExpStark::generate_trace         src/starks/fields/exp_stark.rs:53-67
 *   prove()                            src/starks/common/prover.rs:18-72
 *   verify()                           src/starks/common/verifier.rs:32-98
 * as called from G1/G2/FqStarkProofGenerator::run_once
 *   (src/generators/g1/stark_proof.rs:136-179, g2/stark_proof.rs:136, fq/stark_proof.rs:135).
 *
 * Plain pointers and sizes only. All field elements are canonical little-endian u64 (< p).
 * Input wire format, one row per instance, each 256-bit value as 4 little-endian u64 words:
 *   kind G1: s, x.x, x.y, offset.x, offset.y                                   (20 words)
 *   kind G2: s, x.x.c0, x.x.c1, x.y.c0, x.y.c1, offset.x.c0, ... offset.y.c1   (36 words)
 *   kind FQ: s, x                                                              (8 words)
 * `s` is any value < 2^256 (not reduced); coordinates must be canonical (< p) affine, non-infinity.
 * `timestamps[i]` is the CTL timestamp of instance i (the reference uses the batch index).
 */
#ifndef PB254_H
#define PB254_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum { PB254_KIND_G1 = 0, PB254_KIND_G2 = 1, PB254_KIND_FQ = 2 };

/* return codes (the reference panics / returns anyhow::Error at these points, SURVEY.md §5) */
enum {
  PB254_OK = 0,
  PB254_E_SCALAR_RANGE = 1,  /* common/utils.rs:4   scalar wider than 256 bits (unreachable on this wire format) */
  PB254_E_INFINITY = 2,      /* g1/add.rs:49-51     an intermediate a = -b (point at infinity) */
  PB254_E_NOT_CANONICAL = 3, /* coordinate >= p */
  PB254_E_CUDA = 4,          /* CUDA runtime failure */
  PB254_E_OOM = 5,           /* device allocation failure */
  PB254_E_BAD_ARG = 6,
  PB254_E_VERIFY = 7,        /* verifier.rs: proof rejected */
  PB254_E_NOT_ON_CURVE = 8   /* an input point is not on the curve: G1Affine / G2Affine are curve points by construction
                                in the reference (ark-ec); the device chains re-associate additions and need the group law */
};

/* StarkConfig (starky config.rs; the reference hard-wires standard_fast_config() at
 * src/generators/g1/stark_proof.rs:85,152) */
typedef struct pb254_config {
  uint32_t rate_bits;        /* 1 */
  uint32_t cap_height;       /* 4 */
  uint32_t num_challenges;   /* 2 */
  uint32_t num_query_rounds; /* 84 */
  uint32_t pow_bits;         /* 16 */
  uint32_t arity_bits;       /* 4  (FriReductionStrategy::ConstantArityBits(4, 5)) */
  uint32_t final_poly_bits;  /* 5 */
} pb254_config;

typedef struct pb254_ctx pb254_ctx;
typedef struct pb254_proof pb254_proof;

void pb254_config_standard_fast(pb254_config* out);

/* One context per GPU; a context may be used by one thread at a time. `stream` is a cudaStream_t
 * (0 / NULL = the library creates its own stream). */
int pb254_ctx_create(int device, void* stream, pb254_ctx** out);
void pb254_ctx_destroy(pb254_ctx* ctx);
const char* pb254_last_error(void);
/* number of CUDA kernels this library has launched in this process */
uint64_t pb254_launch_count(void);

/* device time (CUDA events on the context's stream) of the stages of the last call, in ms */
int pb254_timing_count(pb254_ctx* ctx);
const char* pb254_timing_name(pb254_ctx* ctx, int i);
double pb254_timing_ms(pb254_ctx* ctx, int i);

/* shapes */
int pb254_trace_width(int kind);                  /* 781 / 1295 / 427 */
int pb254_input_words(int kind);                  /* 20 / 36 / 8 */
int pb254_num_aux(int kind, uint32_t num_challenges); /* 456 / 906 / 134 for 2 challenges */
size_t pb254_trace_rows(size_t n_inputs, size_t min_rows);

/* ---- building blocks (exposed for parity tests and reuse) ----------------------------------- */
/* Poseidon permutation of n states (12 words each), on the device. */
int pb254_poseidon_permute(pb254_ctx* ctx, const uint64_t* states_in, size_t n, uint64_t* states_out);
/* K3: LDE of a host column-major matrix (cols x n) -> host (cols x n<<rate_bits), natural order. */
int pb254_lde_batch(pb254_ctx* ctx, const uint64_t* values, size_t cols, size_t n, uint32_t rate_bits,
                    int from_coeffs, uint64_t* lde_out);
/* K3+K4+K5: PolynomialBatch::from_values / from_coeffs of a host column-major matrix: Merkle cap
 * (2^cap_height x 4 words) and, optionally, all digest levels bottom-up. */
int pb254_commit(pb254_ctx* ctx, const uint64_t* values, size_t cols, size_t n, uint32_t rate_bits,
                 uint32_t cap_height, int from_coeffs, uint64_t* cap_out, uint64_t* digests_out);

/* ---- oversized single trace across GPUs (SURVEY.md 8e): device-pointer building blocks ------------------
 * One committed matrix too large or too slow for one GPU is column-sharded for the LDE (no communication),
 * exchanged once (NCCL all-to-all over NVLink, done by the host language with its own communicator) into
 * contiguous row blocks, leaf-hashed row-locally, and the digests are all-gathered so that every rank builds
 * the subtree under its own Merkle-cap entries. All pointers are device pointers on the context's GPU. */
/* LDE of `cols` device-resident columns [col][n] -> [col][n << rate_bits], natural order. */
int pb254_lde_dev(pb254_ctx* ctx, const uint64_t* d_values, size_t cols, size_t n, uint32_t rate_bits,
                  int from_coeffs, uint64_t* d_lde_out);
/* d_digests_out[i] = hash_or_noop(row i) for `rows` rows of the column-major matrix [cols][stride]. */
int pb254_leaf_hash_rows_dev(pb254_ctx* ctx, const uint64_t* d_matrix, size_t stride, size_t cols, size_t rows,
                             uint64_t* d_digests_out);
/* 2^log_roots roots of the subtree over tree positions [first, first + 2^log_sub) of a tree with 2^log_total
 * leaves, leaf(q) = d_all_digests[bit_reverse(q)] (digests of all rows in natural row order). */
int pb254_merkle_subtree_dev(pb254_ctx* ctx, const uint64_t* d_all_digests, uint32_t log_total, size_t first,
                             uint32_t log_sub, uint32_t log_roots, uint64_t* d_roots_out);

/* ---- ONE proof across the GPUs of a node (SURVEY.md 8e, BASELINE config 5) ----------------------------------
 * prove() of src/starks/common/prover.rs:18-72 for a single oversized trace, one process per GPU, every rank calling
 * pb254_prove_sharded with the same inputs. The transcript is replicated (every rank derives the same challenges from
 * the same caps), the heavy stages are sharded:
 *   commitments (trace, auxiliary)  LDE of a column shard -> all_to_all -> leaf hashing of a row block -> all_gather of
 *                                   the digests -> inner levels
 *   quotient evaluation             row blocks of the LDE with a next-row halo -> all_gather of the values
 *   FRI combination                 row blocks -> all_gather
 *   query openings                  rows from the rank that owns them -> all_gather
 *   trace generation, auxiliary     by instances / row blocks when n / world is a multiple of 512 and >= 2^16 (every
 *   columns                         BASELINE size), with one all_to_all of values per matrix; replicated otherwise
 * and the proof is byte-identical to the single-GPU proof on every rank (pb254_proof_results_* is empty when the trace
 * is generated by instances: the native outputs are then spread over the ranks). An input error of any instance fails
 * the call on EVERY rank with the same code. The collectives are the CALLER's (its own
 * NCCL communicator: torch.distributed in plonky2_bn254_b200/dist.py, an NCCL binding in a Rust caller): the library
 * calls back with device pointers on the context's GPU; the callee must enqueue the collective on the context's
 * stream (or order it after prior and before later work of that stream) and return 0 on success. */
typedef struct pb254_comm {
  uint32_t rank, world; /* world: a power of two, <= 2^cap_height, dividing the LDE height */
  void* user;
  /* send: world chunks of bytes_per_peer, chunk q goes to rank q; recv: chunk q came from rank q */
  int (*all_to_all)(void* user, const void* d_send, void* d_recv, size_t bytes_per_peer);
  /* recv: world chunks of bytes_per_rank in rank order */
  int (*all_gather)(void* user, const void* d_send, void* d_recv, size_t bytes_per_rank);
} pb254_comm;
int pb254_prove_sharded(pb254_ctx* ctx, int kind, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs,
                        size_t min_rows, const pb254_config* cfg, const pb254_comm* comm, pb254_proof** out);

/* ---- trace generation (K1 + K2) -------------------------------------------------------------- */
/* generate_trace(&inputs, min_rows): fills cols_out, column-major pb254_trace_width(kind) x
 * pb254_trace_rows(n_inputs, min_rows), with the bit-exact trace of the reference. min_rows must make
 * the trace at least 2^16 rows (the reference passes 1 << 16). */
int pb254_generate_trace(pb254_ctx* ctx, int kind, const uint64_t* inputs, const uint64_t* timestamps,
                         size_t n_inputs, size_t min_rows, uint64_t* cols_out);

/* ---- witness before proving (K13) ------------------------------------------------------------ */
/* Chained scalar multiplications, the witness G1/G2SingleGenerator computes natively before run_once
 * (src/generators/g1/single.rs:48-52) and g1_msm threads through `offset` (src/utils/g1_msm.rs:22-36).
 * kind: PB254_KIND_G1 or PB254_KIND_G2. terms: n_terms rows of s, x (G1 12 words, G2 20 words), in chain order.
 * chain_starts: n_chains + 1 indices, chain_starts[0] = 0, non-decreasing, chain_starts[n_chains] = n_terms.
 * offsets: n_chains affine points (G1 8 words, G2 16 words). For chain c: acc = offsets[c]; for each term i of the
 * chain, row i of inputs_out = (s_i, x_i, acc) and acc = s_i * x_i + acc; sums_out[c] = acc (may be NULL).
 * inputs_out is in the pb254_prove wire format. At most 2^17 terms and 2^17 chains. PB254_E_INFINITY if an
 * accumulator after the first is the point at infinity (pb254_last_error() names the lowest such chain and term);
 * PB254_E_NOT_CANONICAL / PB254_E_NOT_ON_CURVE as pb254_prove. */
int pb254_scalar_mul_chains(pb254_ctx* ctx, int kind, const uint64_t* terms, size_t n_terms,
                            const uint64_t* chain_starts, size_t n_chains, const uint64_t* offsets,
                            uint64_t* inputs_out, uint64_t* sums_out);

/* The Shallue-van de Woestijne map of HashToG2::map_to_g2 (src/utils/hash_to_g2.rs:113-147), before cofactor
 * clearing. us: n values u in Fq2, 8 words each (c0, c1). points_out: n affine points of the G2 curve, 16 words each
 * (x.c0, x.c1, y.c0, y.c1). Square roots as ark-ff computes them: a^((p+1)/4) in Fq, the complex method in Fq2; the
 * sign of y follows sgn(u) (src/fields/sgn.rs:20-27). At most 2^17 values. PB254_E_NOT_CANONICAL for a coordinate
 * >= p, PB254_E_BAD_ARG for an exceptional u (tv1 * tv2 = 0); pb254_last_error() names the lowest such index. */
int pb254_map_to_g2(pb254_ctx* ctx, const uint64_t* us, size_t n, uint64_t* points_out);

/* HashToG2::hash_to_g2 (src/utils/hash_to_g2.rs:76-148) of n messages of msg_len canonical Goldilocks elements each
 * (row-major; msg_len = 0 is valid), with the cofactor clearing of the circuit (:195-208) as pb254_prove G2 rows.
 * u_i = hash_to_fq2(m_i) (the plonky2 Challenger, :76-87), x_i = map_to_g2(u_i), k_i = the 254 low bits of the
 * SplitMix64(seed) draws 4i+1 .. 4i+4 (little endian), offset_i = k_i * G2.
 * inputs_out: n rows of 36 words (s = the G2 cofactor, x_i, offset_i). hashes_out: n affine points of 16 words,
 * cofactor * x_i, the hash_to_g2 output. At most 2^17 messages and 2^24 message elements in all. Errors name the
 * lowest failing message: PB254_E_NOT_CANONICAL (an element >= 2^64 - 2^32 + 1), PB254_E_BAD_ARG (an exceptional u,
 * or k_i = 0 mod r), PB254_E_INFINITY (cofactor * x_i + offset_i or cofactor * x_i at infinity). */
int pb254_hash_to_g2(pb254_ctx* ctx, const uint64_t* messages, size_t n, size_t msg_len, uint64_t seed,
                     uint64_t* inputs_out, uint64_t* hashes_out);

/* ---- proving ------------------------------------------------------------------------------- */
/* generate_trace + prove in one call, the body of run_once between
 * src/generators/g1/stark_proof.rs:154 and :163; the trace stays on the device.
 * cfg == NULL selects StarkConfig::standard_fast_config(). The proof-of-work witness is the MINIMAL
 * one (the reference's rayon find_any returns an arbitrary valid witness). */
int pb254_prove(pb254_ctx* ctx, int kind, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs,
                size_t min_rows, const pb254_config* cfg, int keep_debug, pb254_proof** out);
/* pb254_prove with `d_inputs` / `d_timestamps` already resident in the memory of the context's GPU
 * (same wire format); the batched-pipeline form, where a producer kernel wrote the work items. */
int pb254_prove_dev(pb254_ctx* ctx, int kind, const uint64_t* d_inputs, const uint64_t* d_timestamps,
                    size_t n_inputs, size_t min_rows, const pb254_config* cfg, int keep_debug, pb254_proof** out);
/* A stream of independent proofs through several contexts of the SAME GPU (one stream and one workspace each), the
 * software pipeline of a witness generator that has many batches to prove (the circuit builder registers one
 * G1/G2/FqStarkProofGenerator per 128-1024 operations, src/generators/g1/stark_proof.rs:136): batch b is proved by
 * pb254_prove on ctxs[b % n_ctx], the contexts run on their own host threads, so the host-side transcript, the small
 * kernels and the tail waves of one proof overlap the big kernels of the next. inputs / timestamps: n_batches
 * consecutive batches of n_inputs instances each (wire format as above). proofs_out: n_batches handles, in batch
 * order; identical to what pb254_prove returns for each batch. On failure nothing is returned and the first
 * error is reported. */
int pb254_prove_many(pb254_ctx* const* ctxs, size_t n_ctx, int kind, const uint64_t* inputs, const uint64_t* timestamps,
                     size_t n_inputs, size_t n_batches, size_t min_rows, const pb254_config* cfg, pb254_proof** proofs_out);
/* prove(stark, config, trace, ctls, public_inputs = []) on a host trace, column-major
 * pb254_trace_width(kind) x n_rows (src/starks/common/prover.rs:18-30). */
int pb254_prove_trace(pb254_ctx* ctx, int kind, const uint64_t* trace_cols, size_t n_rows, const pb254_config* cfg,
                      int keep_debug, pb254_proof** out);
void pb254_proof_free(pb254_proof* proof);

/* ---- verification (pb254_verify on the host, as the reference; pb254_verify_device on a context) ---- */
/* verify(stark, config, ctls, proof, public_inputs = [], extra_looking_values)
 * (src/starks/common/verifier.rs:32-98) on a serialized proof. As in the reference, the STARK (`kind`) and the
 * StarkConfig (`cfg`, NULL = standard_fast_config) are the CALLER's: a proof whose header names another kind or
 * other parameters (fewer query rounds, no grinding, ...) is rejected; only degree_bits is taken from the proof.
 * `inputs` holds n_inputs rows of pb254_input_words(kind) words. The extra looking values are recomputed natively
 * from the batch (inputs / timestamps, same wire format as pb254_prove), as run_once does with
 * g1_generate_ctl_values (src/starks/curves/g1/scalar_mul_ctl.rs:57-80). Returns PB254_OK or PB254_E_VERIFY
 * (pb254_last_error() names the failed check). Needs no context and no GPU. */
int pb254_verify(int kind, const pb254_config* cfg, const uint64_t* proof_words, size_t n_words,
                 const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs);
/* pb254_verify with the native CTL values and all Merkle openings computed on the context's GPU. Same arguments
 * and the same result as pb254_verify: for every input it returns the same code and pb254_last_error() names the
 * same failed check. PB254_E_CUDA / PB254_E_OOM are the only additional outcomes. The transcript, the quotient
 * identity at zeta and the FRI folds run on the calling thread; stage times are "verify native ctl" and
 * "verify merkle" (pb254_timing_*). */
int pb254_verify_device(pb254_ctx* ctx, int kind, const pb254_config* cfg, const uint64_t* proof_words,
                        size_t n_words, const uint64_t* inputs, const uint64_t* timestamps, size_t n_inputs);
#define PB254_VERIFY_MESSAGE_BYTES 256
/* pb254_verify_device on n_proofs proofs of ONE kind under ONE StarkConfig (the caller's, NULL = standard_fast), the
 * batched counterpart of pb254_prove_many: one launch per stage for every 64 proofs.
 * proof_words[b] / n_words[b]: proof b. inputs / timestamps: the batches of all proofs concatenated in the pb254_prove
 * wire format; proof b's rows are input_starts[b] .. input_starts[b+1] (n_proofs + 1 indices, input_starts[0] = 0,
 * non-decreasing). codes_out[b]: what pb254_verify returns for proof b alone (0 = accepted). messages_out: NULL, or
 * n_proofs slots of PB254_VERIFY_MESSAGE_BYTES; slot b receives pb254_last_error() of that pb254_verify call,
 * NUL-terminated and truncated to fit ("" for an accepted proof).
 * Returns PB254_OK if every proof is accepted. Otherwise it returns the code of the lowest rejected proof, and
 * pb254_last_error() is "proof <b>: <its message>". PB254_E_CUDA / PB254_E_OOM fail the whole call and are written
 * to every codes_out entry. PB254_E_BAD_ARG for bad arguments leaves the outputs untouched. At most 2^12 proofs. */
int pb254_verify_many_device(pb254_ctx* ctx, int kind, const pb254_config* cfg, const uint64_t* const* proof_words,
                             const size_t* n_words, size_t n_proofs, const uint64_t* inputs, const uint64_t* timestamps,
                             const uint64_t* input_starts, int* codes_out, char* messages_out);
/* Serialized StarkProofWithMetadata: little-endian u64 words, field order of SURVEY.md C.7 behind a
 * 10-word header {magic, kind, degree_bits, config[7]} (layout in DESIGN.md). */
size_t pb254_proof_words(const pb254_proof* proof);
const uint64_t* pb254_proof_data(const pb254_proof* proof);
/* ---- proof fields (the consumer of the proof, set_stark_proof_target at src/generators/g1/stark_proof.rs:173-178
 * and src/starks/common/ctl_values.rs:10-26, walks StarkProofWithMetadata field by field) ------------------------
 * Where every field of StarkProofWithMetadata lives in a serialized proof: offsets and sizes in u64 words from the
 * start of the blob. An extension element is 2 words, a Merkle cap 4 * 2^cap_height words, a hash 4 words.
 * Field names are starky's (proof.rs: StarkProof, StarkOpeningSet) and plonky2's (fri/proof.rs: FriProof,
 * FriQueryRound, FriInitialTreeProof, FriQueryStep). Needs no context and no GPU. */
#define PB254_MAX_FRI_LAYERS 16
typedef struct pb254_proof_layout {
  uint32_t kind, degree_bits;
  pb254_config config;              /* as stamped into the header */
  uint32_t trace_width;             /* W */
  uint32_t aux_width;               /* A: lookup helper columns, lookup Z and CTL Z columns */
  uint32_t quotient_width;          /* Q = 2 * num_challenges */
  uint32_t num_ctl_zs;              /* 2 * num_challenges (two cross-table lookups) */
  uint32_t num_fri_layers;          /* commit-phase reductions */
  uint32_t fri_arity_bits[PB254_MAX_FRI_LAYERS];
  uint64_t words;                   /* total length of the blob */
  uint64_t cap_words;               /* 4 * 2^cap_height */
  uint64_t init_challenger_state;   /* 12 words  (StarkProofWithMetadata::init_challenger_state) */
  uint64_t trace_cap, auxiliary_polys_cap, quotient_polys_cap;  /* cap_words each */
  uint64_t local_values, next_values;                   /* 2 W each   (openings) */
  uint64_t auxiliary_polys, auxiliary_polys_next;       /* 2 A each */
  uint64_t ctl_zs_first;                                /* num_ctl_zs base-field words */
  uint64_t quotient_polys;                              /* 2 Q */
  uint64_t commit_phase_merkle_caps;                    /* num_fri_layers x cap_words */
  uint64_t query_round_proofs;                          /* config.num_query_rounds records of query_words */
  uint64_t query_words;
  uint64_t final_poly, final_poly_words;                /* 2 words per coefficient */
  uint64_t pow_witness;                                 /* 1 word */
  /* inside one query record (offsets from the start of the record): initial_trees_proof = the three oracles'
   * (leaf values, Merkle siblings bottom-up), then one FriQueryStep (evals, siblings) per layer */
  uint32_t initial_path_words;      /* 4 * (degree_bits + rate_bits - cap_height) */
  uint32_t q_trace_leaf, q_trace_path, q_aux_leaf, q_aux_path, q_quotient_leaf, q_quotient_path;
  uint32_t q_step_evals[PB254_MAX_FRI_LAYERS], q_step_evals_words[PB254_MAX_FRI_LAYERS];
  uint32_t q_step_path[PB254_MAX_FRI_LAYERS], q_step_path_words[PB254_MAX_FRI_LAYERS];
} pb254_proof_layout;
/* Checks the header and the length of a serialized proof and fills the layout. PB254_E_BAD_ARG if the words are
 * not a proof blob or the length does not match the header. */
int pb254_proof_parse(const uint64_t* proof_words, size_t n_words, pb254_proof_layout* out);

/* The batch's native outputs, read from the trace instead of being recomputed on the CPU: for instance k the
 * 16-bit limbs (one per word) of s*x + offset (G1: x, y; G2: x.c0, x.c1, y.c0, y.c1) or x^s (Fq). run_once
 * computes exactly these with arkworks before proving (src/generators/g1/stark_proof.rs:143-149) and the MSM
 * helpers chain them (src/utils/g1_msm.rs:22-36). Only filled by pb254_prove / pb254_prove_dev. */
size_t pb254_proof_results_words(const pb254_proof* proof);
const uint64_t* pb254_proof_results_data(const pb254_proof* proof);
/* intermediate artefacts for parity tests: which = 0 auxiliary values (A x n), 1 quotient chunk coefficients
 * (2*num_challenges x n), 2 challenges [betas, gammas, alphas, zeta, fri_alpha, fri_betas], 3 query indices,
 * 5 the running quotient total of challenge 0 after every constraint group at quotient point 5 (64 words per pass of
 * the quotient kernel, 4096 words). Slots 0-2 and 5 are filled only when keep_debug != 0, slot 3 always; any other
 * `which` gives 0 words and NULL. */
size_t pb254_proof_debug_words(const pb254_proof* proof, int which);
const uint64_t* pb254_proof_debug_data(const pb254_proof* proof, int which);

#ifdef __cplusplus
}
#endif
#endif /* PB254_H */
