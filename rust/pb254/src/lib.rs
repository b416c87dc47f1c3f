//! Safe wrapper over `pb254-sys` with the reference's types at the surface.
//!
//! UNCOMPILED (no Rust toolchain in the build image). It mirrors the call sites
//!   G1/G2/FqStarkProofGenerator::run_once   src/generators/{g1,g2,fq}/stark_proof.rs:135-179
//!   prove()                                 src/starks/common/prover.rs:18-72
//!   verify()                                src/starks/common/verifier.rs:32-98
//! and rebuilds `StarkProofWithMetadata<F, C, D>` from the proof blob through `pb254_proof_parse`
//! (layout: include/pb254.h `pb254_proof_layout`, INTEGRATION.md §3).
use anyhow::{anyhow, Result};
use ark_bn254::{Fq, Fq2, G1Affine, G2Affine};
use ark_ff::{BigInt, PrimeField};
use num_bigint::BigUint;
use pb254_sys as sys;
use plonky2::field::extension::quadratic::QuadraticExtension;
use plonky2::field::extension::FieldExtension;
use plonky2::field::goldilocks_field::GoldilocksField;
use plonky2::field::polynomial::PolynomialCoeffs;
use plonky2::field::types::Field;
use plonky2::fri::proof::{FriInitialTreeProof, FriProof, FriQueryRound, FriQueryStep};
use plonky2::hash::hash_types::HashOut;
use plonky2::hash::hashing::PlonkyPermutation;
use plonky2::hash::merkle_proofs::MerkleProof;
use plonky2::hash::merkle_tree::MerkleCap;
use plonky2::hash::poseidon::{PoseidonHash, PoseidonPermutation};
use plonky2::plonk::config::PoseidonGoldilocksConfig;
use starky::config::StarkConfig;
use starky::proof::{StarkOpeningSet, StarkProof, StarkProofWithMetadata};
use std::ffi::CStr;

pub use sys::{PB254_KIND_FQ, PB254_KIND_G1, PB254_KIND_G2};

type F = GoldilocksField;
type C = PoseidonGoldilocksConfig;
type FE = QuadraticExtension<F>;
const D: usize = 2;

/// One prover context per GPU (not `Sync`: one thread at a time, like the reference's generator loop).
pub struct Context(*mut sys::pb254_ctx);
unsafe impl Send for Context {}

fn last_error() -> String {
    unsafe { CStr::from_ptr(sys::pb254_last_error()).to_string_lossy().into_owned() }
}
fn check(rc: i32) -> Result<()> {
    if rc == sys::PB254_OK { Ok(()) } else { Err(anyhow!("pb254 error {rc}: {}", last_error())) }
}

/// `StarkConfig` -> `pb254_config` (starky config.rs; `ConstantArityBits(arity_bits, final_poly_bits)`).
pub fn config_of(c: &StarkConfig) -> Result<sys::pb254_config> {
    use plonky2::fri::reduction_strategies::FriReductionStrategy::ConstantArityBits;
    let (arity_bits, final_poly_bits) = match c.fri_config.reduction_strategy {
        ConstantArityBits(a, f) => (a as u32, f as u32),
        _ => return Err(anyhow!("only FriReductionStrategy::ConstantArityBits is supported")),
    };
    Ok(sys::pb254_config {
        rate_bits: c.fri_config.rate_bits as u32,
        cap_height: c.fri_config.cap_height as u32,
        num_challenges: c.num_challenges as u32,
        num_query_rounds: c.fri_config.num_query_rounds as u32,
        pow_bits: c.fri_config.proof_of_work_bits,
        arity_bits,
        final_poly_bits,
    })
}

fn push_biguint(out: &mut Vec<u64>, x: &BigUint) {
    let mut d = x.to_u64_digits();
    assert!(d.len() <= 4, "scalar wider than 256 bits (common/utils.rs:4)");
    d.resize(4, 0);
    out.extend_from_slice(&d);
}
fn push_fq(out: &mut Vec<u64>, x: &Fq) {
    out.extend_from_slice(&x.into_bigint().0); // canonical little-endian 4 x u64
}
fn push_fq2(out: &mut Vec<u64>, x: &Fq2) {
    push_fq(out, &x.c0);
    push_fq(out, &x.c1);
}

/// Wire format of `G1ScalarMulInput {s, x, offset}` (src/starks/curves/g1/scalar_mul_stark.rs:37-41): 20 words.
pub fn pack_g1(inputs: &[(BigUint, G1Affine, G1Affine)]) -> Vec<u64> {
    let mut w = Vec::with_capacity(inputs.len() * 20);
    for (s, x, off) in inputs {
        push_biguint(&mut w, s);
        push_fq(&mut w, &x.x);
        push_fq(&mut w, &x.y);
        push_fq(&mut w, &off.x);
        push_fq(&mut w, &off.y);
    }
    w
}
/// Wire format of `G2ScalarMulInput {s, x, offset}` (src/starks/curves/g2/scalar_mul_stark.rs:36-40): 36 words,
/// every Fq2 coordinate as c0 then c1.
pub fn pack_g2(inputs: &[(BigUint, G2Affine, G2Affine)]) -> Vec<u64> {
    let mut w = Vec::with_capacity(inputs.len() * 36);
    for (s, x, off) in inputs {
        push_biguint(&mut w, s);
        push_fq2(&mut w, &x.x);
        push_fq2(&mut w, &x.y);
        push_fq2(&mut w, &off.x);
        push_fq2(&mut w, &off.y);
    }
    w
}
/// Wire format of `FqExpInput {s, x}` (src/starks/fields/exp_stark.rs:36-39): 8 words.
pub fn pack_fq(inputs: &[(BigUint, Fq)]) -> Vec<u64> {
    let mut w = Vec::with_capacity(inputs.len() * 8);
    for (s, x) in inputs {
        push_biguint(&mut w, s);
        push_fq(&mut w, x);
    }
    w
}

/// 16 limbs of 16 bits (one per word, little-endian) -> Fq: the limb convention of src/starks/mod.rs:13-20.
pub fn fq_from_limbs(limbs: &[u64]) -> Fq {
    assert_eq!(limbs.len(), 16);
    let mut w = [0u64; 4];
    for (i, l) in limbs.iter().enumerate() {
        w[i / 4] |= (l & 0xffff) << (16 * (i % 4));
    }
    Fq::from_bigint(BigInt(w)).expect("canonical limbs")
}

/// A proof together with the batch's native outputs (read from the trace on the device).
pub struct Proved {
    pub proof: StarkProofWithMetadata<F, C, D>,
    pub blob: Vec<u64>,
    /// `pb254_proof_results_data`: per instance 32 (G1), 64 (G2) or 16 (Fq) limbs.
    pub results: Vec<u64>,
}
impl Proved {
    /// `s * x + offset` per instance — what run_once computes with arkworks at stark_proof.rs:143-149.
    pub fn g1_outputs(&self) -> Vec<G1Affine> {
        self.results.chunks(32).map(|r| G1Affine::new_unchecked(fq_from_limbs(&r[..16]), fq_from_limbs(&r[16..]))).collect()
    }
    pub fn g2_outputs(&self) -> Vec<G2Affine> {
        self.results
            .chunks(64)
            .map(|r| {
                let x = Fq2::new(fq_from_limbs(&r[..16]), fq_from_limbs(&r[16..32]));
                let y = Fq2::new(fq_from_limbs(&r[32..48]), fq_from_limbs(&r[48..]));
                G2Affine::new_unchecked(x, y)
            })
            .collect()
    }
    /// `x^s` per instance (src/generators/fq/stark_proof.rs:143-146).
    pub fn fq_outputs(&self) -> Vec<Fq> {
        self.results.chunks(16).map(fq_from_limbs).collect()
    }
}

impl Context {
    pub fn new(device: i32) -> Result<Self> {
        let mut p = std::ptr::null_mut();
        check(unsafe { sys::pb254_ctx_create(device, std::ptr::null_mut(), &mut p) })?;
        Ok(Context(p))
    }

    fn take(h: *mut sys::pb254_proof) -> Result<Proved> {
        let blob = unsafe { std::slice::from_raw_parts(sys::pb254_proof_data(h), sys::pb254_proof_words(h)) }.to_vec();
        let nres = unsafe { sys::pb254_proof_results_words(h) };
        let results = if nres == 0 { vec![] } else { unsafe { std::slice::from_raw_parts(sys::pb254_proof_results_data(h), nres) }.to_vec() };
        unsafe { sys::pb254_proof_free(h) };
        Ok(Proved { proof: decode_proof(&blob)?, blob, results })
    }

    /// `pb254_scalar_mul_chains`: the witness `G1SingleGenerator` / `G2SingleGenerator` compute before run_once
    /// (src/generators/g1/single.rs:48-52). `terms` holds n rows of s, x (G1 12 words, G2 20 words) in chain order,
    /// `chain_starts` n_chains + 1 indices (first 0, last n, non-decreasing), `offsets` one affine point per chain
    /// (G1 8 words, G2 16 words). Returns (inputs, sums): the `pack_*` wire rows (s, x, accumulator before the term),
    /// ready for `prove`, and the final accumulator of every chain.
    pub fn scalar_mul_chains(&self, kind: i32, terms: &[u64], chain_starts: &[u64], offsets: &[u64]) -> Result<(Vec<u64>, Vec<u64>)> {
        let fw = match kind {
            sys::PB254_KIND_G1 => 4,
            sys::PB254_KIND_G2 => 8,
            _ => return Err(anyhow!("scalar_mul_chains: kind must be PB254_KIND_G1 or PB254_KIND_G2")),
        };
        let n_chains = chain_starts.len().checked_sub(1).ok_or_else(|| anyhow!("empty chain_starts"))?;
        if terms.len() % (4 + 2 * fw) != 0 || offsets.len() != n_chains * 2 * fw {
            return Err(anyhow!("scalar_mul_chains: terms / offsets do not match the kind and chain_starts"));
        }
        let n_terms = terms.len() / (4 + 2 * fw);
        let mut inputs = vec![0u64; n_terms * (4 + 4 * fw)];
        let mut sums = vec![0u64; n_chains * 2 * fw];
        check(unsafe {
            sys::pb254_scalar_mul_chains(self.0, kind, terms.as_ptr(), n_terms, chain_starts.as_ptr(), n_chains,
                                         offsets.as_ptr(), inputs.as_mut_ptr(), sums.as_mut_ptr())
        })?;
        Ok((inputs, sums))
    }

    /// `pb254_map_to_g2`: the SvdW map of `HashToG2::map_to_g2` (src/utils/hash_to_g2.rs:113-147) before cofactor
    /// clearing. `us` holds n values u in Fq2, 8 words each (c0, c1); returns n affine points of the G2 curve, 16 words
    /// each (x.c0, x.c1, y.c0, y.c1).
    pub fn map_to_g2(&self, us: &[u64]) -> Result<Vec<u64>> {
        if us.len() % 8 != 0 {
            return Err(anyhow!("map_to_g2: {} words are not whole Fq2 values", us.len()));
        }
        let n = us.len() / 8;
        let mut points = vec![0u64; n * 16];
        check(unsafe { sys::pb254_map_to_g2(self.0, us.as_ptr(), n, points.as_mut_ptr()) })?;
        Ok(points)
    }

    /// `pb254_hash_to_g2`: `HashToG2::hash_to_g2` (src/utils/hash_to_g2.rs:76-148) of `n` equally long messages of
    /// canonical Goldilocks elements, concatenated in `messages` (empty messages are valid), with the circuit's
    /// cofactor clearing (:195-208). Returns (inputs, hashes): the `pack_g2` rows (cofactor, mapped point, offset
    /// k_i G2 with k_i drawn from SplitMix64(seed)), ready for `prove`, and the n hash_to_g2 outputs (16 words each).
    pub fn hash_to_g2(&self, messages: &[u64], n: usize, seed: u64) -> Result<(Vec<u64>, Vec<u64>)> {
        if n == 0 {
            return Ok((Vec::new(), Vec::new()));
        }
        if messages.len() % n != 0 {
            return Err(anyhow!("hash_to_g2: {} words are not {} equally long messages", messages.len(), n));
        }
        let msg_len = messages.len() / n;
        let mut inputs = vec![0u64; n * 36];
        let mut hashes = vec![0u64; n * 16];
        check(unsafe {
            sys::pb254_hash_to_g2(self.0, messages.as_ptr(), n, msg_len, seed, inputs.as_mut_ptr(), hashes.as_mut_ptr())
        })?;
        Ok((inputs, hashes))
    }

    /// The G1ScalarMulInput batch of `g1_msm(scalars, points)` (src/utils/g1_msm.rs:22-36) as one chain from a
    /// random subgroup point `offset`: returns (the `pack_g1` words of the batch, sum s_i x_i), the MSM being
    /// acc_N - acc_0. An accumulator at infinity is an error, as in the reference (g1_msm.rs:20-21).
    pub fn g1_msm(&self, scalars: &[BigUint], points: &[G1Affine], offset: &G1Affine) -> Result<(Vec<u64>, G1Affine)> {
        use ark_ec::{AffineRepr, CurveGroup};
        if scalars.len() != points.len() {
            return Err(anyhow!("g1_msm: {} scalars for {} points", scalars.len(), points.len()));
        }
        let mut terms = Vec::with_capacity(points.len() * 12);
        for (s, x) in scalars.iter().zip(points) {
            push_biguint(&mut terms, s);
            push_fq(&mut terms, &x.x);
            push_fq(&mut terms, &x.y);
        }
        let mut off = Vec::with_capacity(8);
        push_fq(&mut off, &offset.x);
        push_fq(&mut off, &offset.y);
        let (inputs, sums) = self.scalar_mul_chains(sys::PB254_KIND_G1, &terms, &[0, points.len() as u64], &off)?;
        let fq = |w: &[u64]| Fq::from_bigint(BigInt([w[0], w[1], w[2], w[3]])).expect("canonical");
        let acc = G1Affine::new_unchecked(fq(&sums[..4]), fq(&sums[4..]));
        Ok((inputs, (acc.into_group() - offset.into_group()).into_affine()))
    }

    /// `generate_trace(&inputs, min_rows)` + `prove` (run_once lines 154-163) for `kind`; `words` as produced by
    /// `pack_*`; `config` None = `StarkConfig::standard_fast_config()`.
    pub fn prove(&self, kind: i32, words: &[u64], timestamps: &[u64], min_rows: usize, config: Option<&StarkConfig>) -> Result<Proved> {
        let cfg = config.map(config_of).transpose()?;
        let mut h = std::ptr::null_mut();
        check(unsafe {
            sys::pb254_prove(self.0, kind, words.as_ptr(), timestamps.as_ptr(), timestamps.len(), min_rows,
                             cfg.as_ref().map_or(std::ptr::null(), |c| c as *const _), 0, &mut h)
        })?;
        Self::take(h)
    }

    /// ONE proof across the GPUs of a node (`pb254_prove_sharded`): every rank (one process per GPU) calls this with the
    /// same `words` / `timestamps` and its own collectives - e.g. closures over an NCCL communicator created on the
    /// stream this context was created with. All ranks return the same proof, byte-identical to `prove` on one GPU.
    /// (No native outputs in this mode: the trace is spread over the ranks.)
    pub fn prove_sharded(&self, kind: i32, words: &[u64], timestamps: &[u64], min_rows: usize, config: Option<&StarkConfig>,
                         rank: u32, world: u32, collectives: &mut dyn Collectives) -> Result<Proved> {
        unsafe extern "C" fn a2a(user: *mut std::ffi::c_void, s: *const std::ffi::c_void, r: *mut std::ffi::c_void, n: usize) -> i32 {
            let c = &mut **(user as *mut &mut dyn Collectives);
            c.all_to_all(s as *const u8, r as *mut u8, n).map_or(1, |_| 0)
        }
        unsafe extern "C" fn ag(user: *mut std::ffi::c_void, s: *const std::ffi::c_void, r: *mut std::ffi::c_void, n: usize) -> i32 {
            let c = &mut **(user as *mut &mut dyn Collectives);
            c.all_gather(s as *const u8, r as *mut u8, n).map_or(1, |_| 0)
        }
        let cfg = config.map(config_of).transpose()?;
        let mut fat: &mut dyn Collectives = collectives;
        let comm = sys::pb254_comm { rank, world, user: &mut fat as *mut _ as *mut std::ffi::c_void,
                                     all_to_all: Some(a2a), all_gather: Some(ag) };
        let mut h = std::ptr::null_mut();
        check(unsafe {
            sys::pb254_prove_sharded(self.0, kind, words.as_ptr(), timestamps.as_ptr(), timestamps.len(), min_rows,
                                     cfg.as_ref().map_or(std::ptr::null(), |c| c as *const _), &comm, &mut h)
        })?;
        Self::take(h)
    }

    /// `generate_trace` alone: column-major `width x rows` (the transpose `trace_rows_to_poly_values` builds).
    pub fn generate_trace(&self, kind: i32, words: &[u64], timestamps: &[u64], min_rows: usize) -> Result<Vec<Vec<F>>> {
        let width = unsafe { sys::pb254_trace_width(kind) } as usize;
        let rows = unsafe { sys::pb254_trace_rows(timestamps.len(), min_rows) };
        let mut cols = vec![0u64; width * rows];
        check(unsafe { sys::pb254_generate_trace(self.0, kind, words.as_ptr(), timestamps.as_ptr(), timestamps.len(), min_rows, cols.as_mut_ptr()) })?;
        Ok(cols.chunks(rows).map(|c| c.iter().map(|&v| F::from_canonical_u64(v)).collect()).collect())
    }

    /// The literal `prove(stark, config, trace, ctls, &[], timing)` on a host trace (prover.rs:18-30).
    pub fn prove_trace(&self, kind: i32, trace: &[Vec<F>], config: Option<&StarkConfig>) -> Result<Proved> {
        use plonky2::field::types::PrimeField64;
        let rows = trace[0].len();
        let flat: Vec<u64> = trace.iter().flat_map(|c| c.iter().map(|v| v.to_canonical_u64())).collect();
        let cfg = config.map(config_of).transpose()?;
        let mut h = std::ptr::null_mut();
        check(unsafe {
            sys::pb254_prove_trace(self.0, kind, flat.as_ptr(), rows, cfg.as_ref().map_or(std::ptr::null(), |c| c as *const _), 0, &mut h)
        })?;
        Self::take(h)
    }

    /// `verify` with the native CTL values and the Merkle openings computed on this context's GPU
    /// (`pb254_verify_device`): the same checks in the same order, so the same result and error for every input.
    pub fn verify(&self, kind: i32, config: Option<&StarkConfig>, blob: &[u64], words: &[u64], timestamps: &[u64]) -> Result<()> {
        let cfg = config.map(config_of).transpose()?;
        check(unsafe {
            sys::pb254_verify_device(self.0, kind, cfg.as_ref().map_or(std::ptr::null(), |c| c as *const _), blob.as_ptr(),
                                     blob.len(), words.as_ptr(), timestamps.as_ptr(), timestamps.len())
        })
    }
}
impl Drop for Context {
    fn drop(&mut self) {
        unsafe { sys::pb254_ctx_destroy(self.0) }
    }
}

/// `verify()` on the serialized proof (host side of libpb254; kind and config are the caller's).
pub fn verify(kind: i32, config: Option<&StarkConfig>, blob: &[u64], words: &[u64], timestamps: &[u64]) -> Result<()> {
    let cfg = config.map(config_of).transpose()?;
    check(unsafe {
        sys::pb254_verify(kind, cfg.as_ref().map_or(std::ptr::null(), |c| c as *const _), blob.as_ptr(), blob.len(),
                          words.as_ptr(), timestamps.as_ptr(), timestamps.len())
    })
}

pub fn layout_of(blob: &[u64]) -> Result<sys::pb254_proof_layout> {
    let mut l = std::mem::MaybeUninit::<sys::pb254_proof_layout>::zeroed();
    check(unsafe { sys::pb254_proof_parse(blob.as_ptr(), blob.len(), l.as_mut_ptr()) })?;
    Ok(unsafe { l.assume_init() })
}

fn fs(w: &[u64]) -> Vec<F> { w.iter().map(|&v| F::from_canonical_u64(v)).collect() }
fn exts(w: &[u64]) -> Vec<FE> {
    w.chunks(2).map(|c| FE::from_basefield_array([F::from_canonical_u64(c[0]), F::from_canonical_u64(c[1])])).collect()
}
fn hashes(w: &[u64]) -> Vec<HashOut<F>> {
    w.chunks(4).map(|c| HashOut { elements: [fs(c)[0], fs(c)[1], fs(c)[2], fs(c)[3]] }).collect()
}

/// Blob -> `StarkProofWithMetadata`, field by field from the parsed layout.
pub fn decode_proof(blob: &[u64]) -> Result<StarkProofWithMetadata<F, C, D>> {
    let l = layout_of(blob)?;
    let at = |off: u64, n: u64| &blob[off as usize..(off + n) as usize];
    let cap = |off: u64| MerkleCap::<F, PoseidonHash>(hashes(at(off, l.cap_words)));
    let (w, a, q) = (l.trace_width as u64, l.aux_width as u64, l.quotient_width as u64);
    let init_challenger_state = PoseidonPermutation::<F>::new(fs(at(l.init_challenger_state, 12)));
    let openings = StarkOpeningSet {
        local_values: exts(at(l.local_values, 2 * w)),
        next_values: exts(at(l.next_values, 2 * w)),
        auxiliary_polys: Some(exts(at(l.auxiliary_polys, 2 * a))),
        auxiliary_polys_next: Some(exts(at(l.auxiliary_polys_next, 2 * a))),
        ctl_zs_first: Some(fs(at(l.ctl_zs_first, l.num_ctl_zs as u64))),
        quotient_polys: Some(exts(at(l.quotient_polys, 2 * q))),
    };
    let nl = l.num_fri_layers as usize;
    let commit_phase_merkle_caps = (0..nl).map(|i| cap(l.commit_phase_merkle_caps + i as u64 * l.cap_words)).collect();
    let mut query_round_proofs = Vec::with_capacity(l.config.num_query_rounds as usize);
    for k in 0..l.config.num_query_rounds as u64 {
        let rec = at(l.query_round_proofs + k * l.query_words, l.query_words);
        let part = |off: u32, n: u32| &rec[off as usize..(off + n) as usize];
        let ip = l.initial_path_words;
        let evals_proofs = [(l.q_trace_leaf, l.trace_width, l.q_trace_path), (l.q_aux_leaf, l.aux_width, l.q_aux_path),
                            (l.q_quotient_leaf, l.quotient_width, l.q_quotient_path)]
            .iter()
            .map(|&(leaf, n, path)| (fs(part(leaf, n)), MerkleProof::<F, PoseidonHash> { siblings: hashes(part(path, ip)) }))
            .collect();
        let steps = (0..nl)
            .map(|i| FriQueryStep {
                evals: exts(part(l.q_step_evals[i], l.q_step_evals_words[i])),
                merkle_proof: MerkleProof { siblings: hashes(part(l.q_step_path[i], l.q_step_path_words[i])) },
            })
            .collect();
        query_round_proofs.push(FriQueryRound { initial_trees_proof: FriInitialTreeProof { evals_proofs }, steps });
    }
    let opening_proof = FriProof {
        commit_phase_merkle_caps,
        query_round_proofs,
        final_poly: PolynomialCoeffs::new(exts(at(l.final_poly, l.final_poly_words))),
        pow_witness: F::from_canonical_u64(blob[l.pow_witness as usize]),
    };
    let proof = StarkProof {
        trace_cap: cap(l.trace_cap),
        auxiliary_polys_cap: Some(cap(l.auxiliary_polys_cap)),
        quotient_polys_cap: Some(cap(l.quotient_polys_cap)),
        openings,
        opening_proof,
    };
    Ok(StarkProofWithMetadata { init_challenger_state, proof })
}


/// The two collectives `Context::prove_sharded` needs, on DEVICE pointers of the context's GPU (sizes in bytes).
/// `all_to_all`: `world` chunks of `bytes_per_peer`, chunk q goes to rank q, chunk q of `recv` came from rank q;
/// `all_gather`: `recv` = `world` chunks of `bytes_per_rank` in rank order. Enqueue on the context's stream.
pub trait Collectives {
    fn all_to_all(&mut self, d_send: *const u8, d_recv: *mut u8, bytes_per_peer: usize) -> Result<()>;
    fn all_gather(&mut self, d_send: *const u8, d_recv: *mut u8, bytes_per_rank: usize) -> Result<()>;
}

/// A stream of independent batches through several contexts of one GPU (`pb254_prove_many`): batch b is proved on
/// `contexts[b % contexts.len()]` by the library's own host threads; proofs come back in batch order.
/// `words`: the batches' `pack_*` rows back to back, `timestamps`: `n_batches * n_inputs` values.
pub fn prove_many(contexts: &[&Context], kind: i32, words: &[u64], timestamps: &[u64], n_inputs: usize, min_rows: usize,
                  config: Option<&StarkConfig>) -> Result<Vec<Proved>> {
    let n_batches = timestamps.len() / n_inputs;
    let cfg = config.map(config_of).transpose()?;
    let ctxs: Vec<*mut sys::pb254_ctx> = contexts.iter().map(|c| c.0).collect();
    let mut handles = vec![std::ptr::null_mut(); n_batches];
    check(unsafe {
        sys::pb254_prove_many(ctxs.as_ptr(), ctxs.len(), kind, words.as_ptr(), timestamps.as_ptr(), n_inputs, n_batches, min_rows,
                              cfg.as_ref().map_or(std::ptr::null(), |c| c as *const _), handles.as_mut_ptr())
    })?;
    handles.into_iter().map(Context::take).collect()
}
