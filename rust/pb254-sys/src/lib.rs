//! Raw bindings of `include/pb254.h`. One item per C declaration, same order.
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_double, c_int, c_void};

pub const PB254_KIND_G1: c_int = 0;
pub const PB254_KIND_G2: c_int = 1;
pub const PB254_KIND_FQ: c_int = 2;

pub const PB254_OK: c_int = 0;
pub const PB254_E_SCALAR_RANGE: c_int = 1;
pub const PB254_E_INFINITY: c_int = 2;
pub const PB254_E_NOT_CANONICAL: c_int = 3;
pub const PB254_E_CUDA: c_int = 4;
pub const PB254_E_OOM: c_int = 5;
pub const PB254_E_BAD_ARG: c_int = 6;
pub const PB254_E_VERIFY: c_int = 7;
pub const PB254_E_NOT_ON_CURVE: c_int = 8;
pub const PB254_MAX_FRI_LAYERS: usize = 16;
pub const PB254_VERIFY_MESSAGE_BYTES: usize = 256;

/// `StarkConfig` (starky config.rs); `standard_fast_config()` = {1, 4, 2, 84, 16, 4, 5}.
#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct pb254_config {
    pub rate_bits: u32,
    pub cap_height: u32,
    pub num_challenges: u32,
    pub num_query_rounds: u32,
    pub pow_bits: u32,
    pub arity_bits: u32,
    pub final_poly_bits: u32,
}

/// `pb254_proof_layout`: where every field of `StarkProofWithMetadata` lives in a serialized proof
/// (offsets and sizes in u64 words), filled by `pb254_proof_parse`.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct pb254_proof_layout {
    pub kind: u32,
    pub degree_bits: u32,
    pub config: pb254_config,
    pub trace_width: u32,
    pub aux_width: u32,
    pub quotient_width: u32,
    pub num_ctl_zs: u32,
    pub num_fri_layers: u32,
    pub fri_arity_bits: [u32; PB254_MAX_FRI_LAYERS],
    pub words: u64,
    pub cap_words: u64,
    pub init_challenger_state: u64,
    pub trace_cap: u64,
    pub auxiliary_polys_cap: u64,
    pub quotient_polys_cap: u64,
    pub local_values: u64,
    pub next_values: u64,
    pub auxiliary_polys: u64,
    pub auxiliary_polys_next: u64,
    pub ctl_zs_first: u64,
    pub quotient_polys: u64,
    pub commit_phase_merkle_caps: u64,
    pub query_round_proofs: u64,
    pub query_words: u64,
    pub final_poly: u64,
    pub final_poly_words: u64,
    pub pow_witness: u64,
    pub initial_path_words: u32,
    pub q_trace_leaf: u32,
    pub q_trace_path: u32,
    pub q_aux_leaf: u32,
    pub q_aux_path: u32,
    pub q_quotient_leaf: u32,
    pub q_quotient_path: u32,
    pub q_step_evals: [u32; PB254_MAX_FRI_LAYERS],
    pub q_step_evals_words: [u32; PB254_MAX_FRI_LAYERS],
    pub q_step_path: [u32; PB254_MAX_FRI_LAYERS],
    pub q_step_path_words: [u32; PB254_MAX_FRI_LAYERS],
}

/// `pb254_comm` (include/pb254.h): the caller's collectives for ONE proof across the GPUs of a node. The callbacks get
/// device pointers on the context's GPU and must enqueue on (or order with) the context's stream; 0 = success.
#[repr(C)]
pub struct pb254_comm {
    pub rank: u32,
    pub world: u32,
    pub user: *mut c_void,
    pub all_to_all: Option<unsafe extern "C" fn(user: *mut c_void, d_send: *const c_void, d_recv: *mut c_void, bytes_per_peer: usize) -> c_int>,
    pub all_gather: Option<unsafe extern "C" fn(user: *mut c_void, d_send: *const c_void, d_recv: *mut c_void, bytes_per_rank: usize) -> c_int>,
}

#[repr(C)]
pub struct pb254_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct pb254_proof {
    _private: [u8; 0],
}

extern "C" {
    pub fn pb254_config_standard_fast(out: *mut pb254_config);
    pub fn pb254_ctx_create(device: c_int, stream: *mut c_void, out: *mut *mut pb254_ctx) -> c_int;
    pub fn pb254_ctx_destroy(ctx: *mut pb254_ctx);
    pub fn pb254_last_error() -> *const c_char;
    pub fn pb254_launch_count() -> u64;
    pub fn pb254_timing_count(ctx: *mut pb254_ctx) -> c_int;
    pub fn pb254_timing_name(ctx: *mut pb254_ctx, i: c_int) -> *const c_char;
    pub fn pb254_timing_ms(ctx: *mut pb254_ctx, i: c_int) -> c_double;
    pub fn pb254_trace_width(kind: c_int) -> c_int;
    pub fn pb254_input_words(kind: c_int) -> c_int;
    pub fn pb254_num_aux(kind: c_int, num_challenges: u32) -> c_int;
    pub fn pb254_trace_rows(n_inputs: usize, min_rows: usize) -> usize;
    pub fn pb254_poseidon_permute(ctx: *mut pb254_ctx, states_in: *const u64, n: usize, states_out: *mut u64) -> c_int;
    pub fn pb254_lde_batch(ctx: *mut pb254_ctx, values: *const u64, cols: usize, n: usize, rate_bits: u32,
                           from_coeffs: c_int, lde_out: *mut u64) -> c_int;
    pub fn pb254_commit(ctx: *mut pb254_ctx, values: *const u64, cols: usize, n: usize, rate_bits: u32,
                        cap_height: u32, from_coeffs: c_int, cap_out: *mut u64, digests_out: *mut u64) -> c_int;
    pub fn pb254_generate_trace(ctx: *mut pb254_ctx, kind: c_int, inputs: *const u64, timestamps: *const u64,
                                n_inputs: usize, min_rows: usize, cols_out: *mut u64) -> c_int;
    pub fn pb254_scalar_mul_chains(ctx: *mut pb254_ctx, kind: c_int, terms: *const u64, n_terms: usize,
                                   chain_starts: *const u64, n_chains: usize, offsets: *const u64,
                                   inputs_out: *mut u64, sums_out: *mut u64) -> c_int;
    pub fn pb254_map_to_g2(ctx: *mut pb254_ctx, us: *const u64, n: usize, points_out: *mut u64) -> c_int;
    pub fn pb254_hash_to_g2(ctx: *mut pb254_ctx, messages: *const u64, n: usize, msg_len: usize, seed: u64,
                            inputs_out: *mut u64, hashes_out: *mut u64) -> c_int;
    pub fn pb254_prove(ctx: *mut pb254_ctx, kind: c_int, inputs: *const u64, timestamps: *const u64, n_inputs: usize,
                       min_rows: usize, cfg: *const pb254_config, keep_debug: c_int, out: *mut *mut pb254_proof) -> c_int;
    pub fn pb254_prove_dev(ctx: *mut pb254_ctx, kind: c_int, d_inputs: *const u64, d_timestamps: *const u64,
                           n_inputs: usize, min_rows: usize, cfg: *const pb254_config, keep_debug: c_int,
                           out: *mut *mut pb254_proof) -> c_int;
    pub fn pb254_prove_trace(ctx: *mut pb254_ctx, kind: c_int, trace_cols: *const u64, n_rows: usize,
                             cfg: *const pb254_config, keep_debug: c_int, out: *mut *mut pb254_proof) -> c_int;
    pub fn pb254_prove_many(ctxs: *const *mut pb254_ctx, n_ctx: usize, kind: c_int, inputs: *const u64, timestamps: *const u64,
                            n_inputs: usize, n_batches: usize, min_rows: usize, cfg: *const pb254_config,
                            proofs_out: *mut *mut pb254_proof) -> c_int;
    pub fn pb254_prove_sharded(ctx: *mut pb254_ctx, kind: c_int, inputs: *const u64, timestamps: *const u64, n_inputs: usize,
                               min_rows: usize, cfg: *const pb254_config, comm: *const pb254_comm,
                               out: *mut *mut pb254_proof) -> c_int;
    pub fn pb254_proof_free(proof: *mut pb254_proof);
    pub fn pb254_verify(kind: c_int, cfg: *const pb254_config, proof_words: *const u64, n_words: usize,
                        inputs: *const u64, timestamps: *const u64, n_inputs: usize) -> c_int;
    pub fn pb254_verify_device(ctx: *mut pb254_ctx, kind: c_int, cfg: *const pb254_config, proof_words: *const u64,
                               n_words: usize, inputs: *const u64, timestamps: *const u64, n_inputs: usize) -> c_int;
    pub fn pb254_verify_many_device(ctx: *mut pb254_ctx, kind: c_int, cfg: *const pb254_config,
                                    proof_words: *const *const u64, n_words: *const usize, n_proofs: usize,
                                    inputs: *const u64, timestamps: *const u64, input_starts: *const u64,
                                    codes_out: *mut c_int, messages_out: *mut c_char) -> c_int;
    pub fn pb254_proof_parse(proof_words: *const u64, n_words: usize, out: *mut pb254_proof_layout) -> c_int;
    pub fn pb254_proof_results_words(proof: *const pb254_proof) -> usize;
    pub fn pb254_proof_results_data(proof: *const pb254_proof) -> *const u64;
    pub fn pb254_lde_dev(ctx: *mut pb254_ctx, d_values: *const u64, cols: usize, n: usize, rate_bits: u32,
                         from_coeffs: c_int, d_lde_out: *mut u64) -> c_int;
    pub fn pb254_leaf_hash_rows_dev(ctx: *mut pb254_ctx, d_matrix: *const u64, stride: usize, cols: usize, rows: usize,
                                    d_digests_out: *mut u64) -> c_int;
    pub fn pb254_merkle_subtree_dev(ctx: *mut pb254_ctx, d_all_digests: *const u64, log_total: u32, first: usize,
                                    log_sub: u32, log_roots: u32, d_roots_out: *mut u64) -> c_int;
    pub fn pb254_proof_words(proof: *const pb254_proof) -> usize;
    pub fn pb254_proof_data(proof: *const pb254_proof) -> *const u64;
    pub fn pb254_proof_debug_words(proof: *const pb254_proof, which: c_int) -> usize;
    pub fn pb254_proof_debug_data(proof: *const pb254_proof, which: c_int) -> *const u64;
}
