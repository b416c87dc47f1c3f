"""ctypes binding of the C ABI in include/pb254.h (libpb254.so, CUDA sm_100a).

There is no CPU fallback: if the CUDA library is missing or no GPU is present, loading / context
creation raises. (Tests for host-side logic may bind the test-only host-simulation build by passing
an explicit path to :class:`Library`; the product never does.)
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libpb254.so")

KIND_G1, KIND_G2, KIND_FQ = 0, 1, 2
MESSAGE_BYTES = 256  # PB254_VERIFY_MESSAGE_BYTES

ERROR_NAMES = {
    0: "OK", 1: "E_SCALAR_RANGE", 2: "E_INFINITY", 3: "E_NOT_CANONICAL", 4: "E_CUDA", 5: "E_OOM", 6: "E_BAD_ARG",
    7: "E_VERIFY", 8: "E_NOT_ON_CURVE",
}


class Pb254Error(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"pb254 error {code} ({ERROR_NAMES.get(code, '?')}): {msg}")
        self.code = code


class Config(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in
                ("rate_bits", "cap_height", "num_challenges", "num_query_rounds", "pow_bits", "arity_bits",
                 "final_poly_bits")]

    def as_tuple(self):
        return tuple(getattr(self, n) for n, _ in self._fields_)


def _u64(a):
    return np.ascontiguousarray(a, dtype=np.uint64)


def _p(a):
    return a.ctypes.data_as(C.c_void_p) if a is not None else None


_COLL_FN = C.CFUNCTYPE(C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_size_t)


class Comm(C.Structure):
    """pb254_comm (include/pb254.h): the caller's collectives for ONE proof across the GPUs of a node."""
    _fields_ = [("rank", C.c_uint32), ("world", C.c_uint32), ("user", C.c_void_p),
                ("all_to_all", _COLL_FN), ("all_gather", _COLL_FN)]


class ProofLayout(C.Structure):
    """pb254_proof_layout (include/pb254.h): offsets and sizes, in u64 words, of the fields of a serialized proof."""
    _fields_ = ([("kind", C.c_uint32), ("degree_bits", C.c_uint32), ("config", Config)] +
                [(n, C.c_uint32) for n in ("trace_width", "aux_width", "quotient_width", "num_ctl_zs", "num_fri_layers")] +
                [("fri_arity_bits", C.c_uint32 * 16)] +
                [(n, C.c_uint64) for n in (
                    "words", "cap_words", "init_challenger_state", "trace_cap", "auxiliary_polys_cap",
                    "quotient_polys_cap", "local_values", "next_values", "auxiliary_polys", "auxiliary_polys_next",
                    "ctl_zs_first", "quotient_polys", "commit_phase_merkle_caps", "query_round_proofs", "query_words",
                    "final_poly", "final_poly_words", "pow_witness")] +
                [(n, C.c_uint32) for n in ("initial_path_words", "q_trace_leaf", "q_trace_path", "q_aux_leaf",
                                           "q_aux_path", "q_quotient_leaf", "q_quotient_path")] +
                [(n, C.c_uint32 * 16) for n in ("q_step_evals", "q_step_evals_words", "q_step_path", "q_step_path_words")])


class Library:
    """A loaded libpb254 (product) or, for host-logic tests only, the hostsim build."""

    def __init__(self, path: str | None = None):
        path = path or LIB_PATH
        if not os.path.exists(path):
            raise FileNotFoundError(
                f"{path} not found: build it with `python -m plonky2_bn254_b200.build` "
                "(there is no CPU fallback for the prover)")
        self.path = path
        self.lib = C.CDLL(path)
        L = self.lib
        L.pb254_last_error.restype = C.c_char_p
        L.pb254_launch_count.restype = C.c_uint64
        L.pb254_trace_rows.restype = C.c_size_t
        L.pb254_trace_rows.argtypes = [C.c_size_t, C.c_size_t]
        L.pb254_ctx_create.argtypes = [C.c_int, C.c_void_p, C.POINTER(C.c_void_p)]
        L.pb254_ctx_destroy.argtypes = [C.c_void_p]
        L.pb254_timing_count.argtypes = [C.c_void_p]
        L.pb254_timing_name.argtypes = [C.c_void_p, C.c_int]
        L.pb254_timing_name.restype = C.c_char_p
        L.pb254_timing_ms.argtypes = [C.c_void_p, C.c_int]
        L.pb254_timing_ms.restype = C.c_double
        L.pb254_proof_words.restype = C.c_size_t
        L.pb254_proof_words.argtypes = [C.c_void_p]
        L.pb254_proof_data.restype = C.POINTER(C.c_uint64)
        L.pb254_proof_data.argtypes = [C.c_void_p]
        L.pb254_proof_debug_words.restype = C.c_size_t
        L.pb254_proof_debug_words.argtypes = [C.c_void_p, C.c_int]
        L.pb254_proof_debug_data.restype = C.POINTER(C.c_uint64)
        L.pb254_proof_debug_data.argtypes = [C.c_void_p, C.c_int]
        L.pb254_proof_free.argtypes = [C.c_void_p]
        L.pb254_proof_results_words.restype = C.c_size_t
        L.pb254_proof_results_words.argtypes = [C.c_void_p]
        L.pb254_proof_results_data.restype = C.POINTER(C.c_uint64)
        L.pb254_proof_results_data.argtypes = [C.c_void_p]

        L.pb254_proof_parse.argtypes = [C.c_void_p, C.c_size_t, C.POINTER(ProofLayout)]
        L.pb254_verify_many_device.restype = C.c_int
        L.pb254_verify_many_device.argtypes = [
            C.c_void_p, C.c_int, C.POINTER(Config), C.POINTER(C.c_void_p), C.POINTER(C.c_size_t), C.c_size_t,
            C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int), C.POINTER(C.c_char)]

    def check(self, rc):
        if rc != 0:
            raise Pb254Error(rc, self.lib.pb254_last_error().decode())

    def standard_fast_config(self) -> Config:
        c = Config()
        self.lib.pb254_config_standard_fast(C.byref(c))
        return c

    def launch_count(self) -> int:
        return int(self.lib.pb254_launch_count())

    def trace_width(self, kind):
        return self.lib.pb254_trace_width(kind)

    def input_words(self, kind):
        return self.lib.pb254_input_words(kind)

    def num_aux(self, kind, num_challenges=2):
        return self.lib.pb254_num_aux(kind, num_challenges)

    def trace_rows(self, n_inputs, min_rows):
        return self.lib.pb254_trace_rows(n_inputs, min_rows)


    def verify(self, kind, proof_words, inputs, timestamps, config: "Config | None" = None) -> bool:
        """pb254_verify(kind, config, ...): True, or raises Pb254Error(E_VERIFY / ...) naming the failed check.
        `kind` and `config` (None = standard_fast_config) are the verifier's own, never the proof's."""
        w, inputs, timestamps = self._verify_args(kind, proof_words, inputs, timestamps)
        self.check(self.lib.pb254_verify(C.c_int(kind), C.byref(config) if config is not None else None, _p(w),
                                         C.c_size_t(w.size), _p(inputs), _p(timestamps), C.c_size_t(inputs.shape[0])))
        return True

    def _verify_args(self, kind, proof_words, inputs, timestamps):
        w = _u64(proof_words)
        inputs = _u64(inputs)
        timestamps = _u64(timestamps)
        if inputs.ndim != 2 or inputs.shape[1] != self.input_words(kind) or timestamps.size != inputs.shape[0]:
            raise Pb254Error(6, "inputs must be (n, input_words(kind)) with one timestamp per row")
        return w, inputs, timestamps


    def parse_proof(self, proof_words) -> "ProofView":
        """pb254_proof_parse: the fields of StarkProofWithMetadata as views into the serialized proof."""
        w = _u64(proof_words)
        lay = ProofLayout()
        self.check(self.lib.pb254_proof_parse(_p(w), C.c_size_t(w.size), C.byref(lay)))
        return ProofView(w, lay)


class ProofView:
    """StarkProofWithMetadata rebuilt from the blob, field names of starky's StarkProof / StarkOpeningSet and
    plonky2's FriProof (what set_stark_proof_target consumes, src/generators/g1/stark_proof.rs:173-178). Every
    attribute is a numpy view of the blob: extension elements as (.., 2), hashes as (.., 4)."""

    def __init__(self, words: np.ndarray, lay: "ProofLayout"):
        self.words, self.layout = words, lay
        w, l = words, lay
        cw = int(l.cap_words)

        def sl(off, n):
            return w[int(off):int(off) + int(n)]

        self.kind, self.degree_bits = int(l.kind), int(l.degree_bits)
        self.config = l.config
        self.init_challenger_state = sl(l.init_challenger_state, 12)
        self.trace_cap = sl(l.trace_cap, cw).reshape(-1, 4)
        self.auxiliary_polys_cap = sl(l.auxiliary_polys_cap, cw).reshape(-1, 4)
        self.quotient_polys_cap = sl(l.quotient_polys_cap, cw).reshape(-1, 4)
        W, A, Q = int(l.trace_width), int(l.aux_width), int(l.quotient_width)
        self.openings = {
            "local_values": sl(l.local_values, 2 * W).reshape(-1, 2),
            "next_values": sl(l.next_values, 2 * W).reshape(-1, 2),
            "auxiliary_polys": sl(l.auxiliary_polys, 2 * A).reshape(-1, 2),
            "auxiliary_polys_next": sl(l.auxiliary_polys_next, 2 * A).reshape(-1, 2),
            "ctl_zs_first": sl(l.ctl_zs_first, l.num_ctl_zs),
            "quotient_polys": sl(l.quotient_polys, 2 * Q).reshape(-1, 2),
        }
        nl = int(l.num_fri_layers)
        self.commit_phase_merkle_caps = sl(l.commit_phase_merkle_caps, nl * cw).reshape(nl, -1, 4)
        self.final_poly = sl(l.final_poly, l.final_poly_words).reshape(-1, 2)
        self.pow_witness = int(w[int(l.pow_witness)])
        ip = int(l.initial_path_words)
        self.query_round_proofs = []
        for q in range(int(l.config.num_query_rounds)):
            rec = sl(int(l.query_round_proofs) + q * int(l.query_words), l.query_words)
            initial = [(rec[a:a + n], rec[b:b + ip].reshape(-1, 4)) for a, n, b in
                       ((l.q_trace_leaf, W, l.q_trace_path), (l.q_aux_leaf, A, l.q_aux_path),
                        (l.q_quotient_leaf, Q, l.q_quotient_path))]
            steps = [(rec[l.q_step_evals[i]:l.q_step_evals[i] + l.q_step_evals_words[i]].reshape(-1, 2),
                      rec[l.q_step_path[i]:l.q_step_path[i] + l.q_step_path_words[i]].reshape(-1, 4)) for i in range(nl)]
            self.query_round_proofs.append({"initial_trees_proof": initial, "steps": steps})

    def serialize(self) -> np.ndarray:
        """The blob rebuilt field by field (round trip of parse)."""
        l = self.layout
        c = l.config
        out = [self.words[:1], np.array([l.kind, l.degree_bits, c.rate_bits, c.cap_height, c.num_challenges,
                                         c.num_query_rounds, c.pow_bits, c.arity_bits, c.final_poly_bits], dtype=np.uint64),
               self.init_challenger_state, self.trace_cap.ravel(), self.auxiliary_polys_cap.ravel(),
               self.quotient_polys_cap.ravel()]
        o = self.openings
        out += [o[k].ravel() for k in ("local_values", "next_values", "auxiliary_polys", "auxiliary_polys_next",
                                       "ctl_zs_first", "quotient_polys")]
        out.append(self.commit_phase_merkle_caps.ravel())
        for q in self.query_round_proofs:
            for leaf, path in q["initial_trees_proof"]:
                out += [leaf, path.ravel()]
            for ev, path in q["steps"]:
                out += [ev.ravel(), path.ravel()]
        out += [self.final_poly.ravel(), np.array([self.pow_witness], dtype=np.uint64)]
        return np.concatenate(out)


_default = None


def prove_many(contexts, kind, batches, min_rows=1 << 16, config: "Config | None" = None):
    """pb254_prove_many: `batches` = list of (inputs, timestamps) of equal size, proved round-robin on `contexts` (all on
    one GPU) by the library's own host threads; returns the proofs in batch order."""
    L = contexts[0].L
    inp = np.ascontiguousarray(np.stack([_u64(b[0]) for b in batches]))
    ts = np.ascontiguousarray(np.stack([_u64(b[1]) for b in batches]))
    nb, n_inputs = inp.shape[0], inp.shape[1]
    assert inp.shape[2] == L.input_words(kind) and ts.shape == (nb, n_inputs)
    handles = (C.c_void_p * nb)()
    ctxs = (C.c_void_p * len(contexts))(*[c._h for c in contexts])
    L.check(L.lib.pb254_prove_many(ctxs, C.c_size_t(len(contexts)), C.c_int(kind), _p(inp), _p(ts), C.c_size_t(n_inputs),
                                   C.c_size_t(nb), C.c_size_t(min_rows),
                                   C.byref(config) if config is not None else None, handles))
    return [Proof(L, C.c_void_p(h)) for h in handles]


def default_library() -> Library:
    global _default
    if _default is None:
        _default = Library()
    return _default


class Context:
    """One prover context per GPU (pb254_ctx)."""

    def __init__(self, device: int = 0, stream: int | None = None, library: Library | None = None):
        self.L = library or default_library()
        h = C.c_void_p()
        self.L.check(self.L.lib.pb254_ctx_create(device, C.c_void_p(stream or 0), C.byref(h)))
        self._h = h

    def close(self):
        if getattr(self, "_h", None):
            self.L.lib.pb254_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def timings(self):
        """[(stage name, device ms)] of the last call on this context."""
        n = self.L.lib.pb254_timing_count(self._h)
        return [(self.L.lib.pb254_timing_name(self._h, i).decode(), self.L.lib.pb254_timing_ms(self._h, i))
                for i in range(n)]

    # ---- building blocks ------------------------------------------------------------------
    def poseidon_permute(self, states):
        s = _u64(states).reshape(-1, 12)
        out = np.empty_like(s)
        self.L.check(self.L.lib.pb254_poseidon_permute(self._h, _p(s), C.c_size_t(s.shape[0]), _p(out)))
        return out

    def lde_batch(self, values, rate_bits, from_coeffs=False):
        v = _u64(values)
        cols, n = v.shape
        out = np.empty((cols, n << rate_bits), dtype=np.uint64)
        self.L.check(self.L.lib.pb254_lde_batch(self._h, _p(v), C.c_size_t(cols), C.c_size_t(n), C.c_uint32(rate_bits),
                                                C.c_int(int(from_coeffs)), _p(out)))
        return out

    def commit(self, values, rate_bits, cap_height, from_coeffs=False, want_digests=False):
        v = _u64(values)
        cols, n = v.shape
        cap = np.empty((1 << cap_height, 4), dtype=np.uint64)
        dig = None
        if want_digests:
            N = n << rate_bits
            total, m = 0, N
            while m >= (1 << cap_height):
                total += m
                m //= 2
            dig = np.empty((total, 4), dtype=np.uint64)
        self.L.check(self.L.lib.pb254_commit(self._h, _p(v), C.c_size_t(cols), C.c_size_t(n), C.c_uint32(rate_bits),
                                             C.c_uint32(cap_height), C.c_int(int(from_coeffs)), _p(cap), _p(dig)))
        return (cap, dig) if want_digests else cap

    # ---- device-pointer building blocks (oversized-trace mode, see dist.py) ---------------------
    def lde_dev(self, d_values: int, cols: int, n: int, rate_bits: int, d_out: int, from_coeffs=False):
        self.L.check(self.L.lib.pb254_lde_dev(self._h, C.c_void_p(d_values), C.c_size_t(cols), C.c_size_t(n),
                                              C.c_uint32(rate_bits), C.c_int(int(from_coeffs)), C.c_void_p(d_out)))

    def leaf_hash_rows_dev(self, d_matrix: int, stride: int, cols: int, rows: int, d_digests: int):
        self.L.check(self.L.lib.pb254_leaf_hash_rows_dev(self._h, C.c_void_p(d_matrix), C.c_size_t(stride),
                                                         C.c_size_t(cols), C.c_size_t(rows), C.c_void_p(d_digests)))

    def merkle_subtree_dev(self, d_all_digests: int, log_total: int, first: int, log_sub: int, log_roots: int,
                           d_roots: int):
        self.L.check(self.L.lib.pb254_merkle_subtree_dev(self._h, C.c_void_p(d_all_digests), C.c_uint32(log_total),
                                                         C.c_size_t(first), C.c_uint32(log_sub),
                                                         C.c_uint32(log_roots), C.c_void_p(d_roots)))

    # ---- trace generation -----------------------------------------------------------------
    def generate_trace(self, kind, inputs, timestamps, min_rows=1 << 16):
        inputs = _u64(inputs)
        timestamps = _u64(timestamps)
        k = inputs.shape[0]
        assert inputs.shape[1] == self.L.input_words(kind)
        n = self.L.trace_rows(k, min_rows)
        cols = np.empty((self.L.trace_width(kind), n), dtype=np.uint64)
        self.L.check(self.L.lib.pb254_generate_trace(self._h, C.c_int(kind), _p(inputs), _p(timestamps), C.c_size_t(k),
                                                     C.c_size_t(min_rows), _p(cols)))
        return cols

    # ---- witness before proving -------------------------------------------------------------
    def scalar_mul_chains(self, kind, terms, chain_starts, offsets):
        """pb254_scalar_mul_chains: chain c starts at offsets[c] and each of its terms (s, x) adds s * x.
        terms (n_terms, 12 | 20) rows of s, x in chain order; chain_starts (n_chains + 1,) with chain_starts[0] = 0 and
        chain_starts[-1] = n_terms; offsets (n_chains, 8 | 16) affine points. Returns (inputs, sums): inputs
        (n_terms, input_words(kind)) pb254_prove rows (s, x, accumulator before the term), sums (n_chains, 8 | 16) the
        final accumulators."""
        fw = 4 if kind == KIND_G1 else 8             # any other kind is rejected by the library
        terms = _u64(terms)
        starts = _u64(chain_starts).reshape(-1)
        offsets = _u64(offsets)
        n_chains = starts.size - 1
        if kind in (KIND_G1, KIND_G2) and (terms.ndim != 2 or terms.shape[1] != 4 + 2 * fw or n_chains < 0 or
                                           offsets.size != n_chains * 2 * fw):
            raise Pb254Error(6, f"terms must be (n, {4 + 2 * fw}) and offsets (len(chain_starts) - 1, {2 * fw})")
        inputs = np.empty((terms.shape[0], 4 + 4 * fw), dtype=np.uint64)
        sums = np.empty((n_chains, 2 * fw), dtype=np.uint64)
        self.L.check(self.L.lib.pb254_scalar_mul_chains(self._h, C.c_int(kind), _p(terms), C.c_size_t(terms.shape[0]),
                                                        _p(starts), C.c_size_t(n_chains), _p(offsets), _p(inputs),
                                                        _p(sums)))
        return inputs, sums

    def map_to_g2(self, us):
        """pb254_map_to_g2: the SvdW map of ``workloads.map_to_curve``. us (n, 8) canonical words of u (c0, c1) in Fq2.
        Returns (n, 16): x.c0, x.c1, y.c0, y.c1 of each point of the G2 curve."""
        us = _u64(us).reshape(-1, 8)
        out = np.empty((us.shape[0], 16), dtype=np.uint64)
        self.L.check(self.L.lib.pb254_map_to_g2(self._h, _p(us), C.c_size_t(us.shape[0]), _p(out)))
        return out

    def hash_to_g2(self, messages, seed: int):
        """pb254_hash_to_g2 over messages (n, msg_len) canonical Goldilocks elements. Returns (inputs, hashes): inputs
        (n, 36) the pb254_prove G2 rows (cofactor, map_to_g2(hash_to_fq2(m)), offset = k * G2 with k drawn from
        SplitMix64(seed) as ``workloads.hash_to_g2_inputs`` draws it), hashes (n, 16) cofactor * x, the hash_to_g2
        outputs."""
        m = _u64(messages)
        if m.ndim != 2:
            raise Pb254Error(6, "messages must be (n, msg_len)")
        inputs = np.empty((m.shape[0], 36), dtype=np.uint64)
        hashes = np.empty((m.shape[0], 16), dtype=np.uint64)
        self.L.check(self.L.lib.pb254_hash_to_g2(self._h, _p(m), C.c_size_t(m.shape[0]), C.c_size_t(m.shape[1]),
                                                 C.c_uint64(seed & (2**64 - 1)), _p(inputs), _p(hashes)))
        return inputs, hashes

    # ---- proving --------------------------------------------------------------------------
    def prove(self, kind, inputs, timestamps, min_rows=1 << 16, config: Config | None = None, keep_debug=False):
        """generate_trace + prove on the device; returns a :class:`Proof`."""
        inputs = _u64(inputs)
        timestamps = _u64(timestamps)
        assert inputs.ndim == 2 and inputs.shape[1] == self.L.input_words(kind)
        h = C.c_void_p()
        self.L.check(self.L.lib.pb254_prove(self._h, C.c_int(kind), _p(inputs), _p(timestamps),
                                            C.c_size_t(inputs.shape[0]), C.c_size_t(min_rows),
                                            C.byref(config) if config is not None else None, C.c_int(int(keep_debug)),
                                            C.byref(h)))
        return Proof(self.L, h)

    def verify(self, kind, proof_words, inputs, timestamps, config: Config | None = None) -> bool:
        """pb254_verify_device: :meth:`Library.verify` with the native CTL values and the Merkle openings computed on
        this context's GPU. Same checks, same outcome for every input: True, or raises the same Pb254Error."""
        w, inputs, timestamps = self.L._verify_args(kind, proof_words, inputs, timestamps)
        self.L.check(self.L.lib.pb254_verify_device(self._h, C.c_int(kind),
                                                    C.byref(config) if config is not None else None, _p(w),
                                                    C.c_size_t(w.size), _p(inputs), _p(timestamps),
                                                    C.c_size_t(inputs.shape[0])))
        return True

    def verify_many(self, kind, proofs, batches, config: Config | None = None):
        """pb254_verify_many_device: :meth:`verify` on every proof, with one launch per stage for every 64 proofs.
        `batches` is one (inputs, timestamps) per proof, of any sizes. Returns one entry per proof: None if accepted,
        else (code, message), what :meth:`Library.verify` reports for that proof alone. Raises Pb254Error for bad
        arguments and for a CUDA or out-of-memory error, which fails the whole call."""
        if len(proofs) != len(batches):
            raise Pb254Error(6, "one (inputs, timestamps) batch per proof")
        args = [self.L._verify_args(kind, w, inp, ts) for w, (inp, ts) in zip(proofs, batches)]
        n = len(args)
        iw = self.L.input_words(kind)
        inputs = np.concatenate([a[1] for a in args]) if n else np.empty((0, iw), dtype=np.uint64)
        timestamps = np.concatenate([a[2] for a in args]) if n else np.empty(0, dtype=np.uint64)
        starts = np.zeros(n + 1, dtype=np.uint64)
        starts[1:] = np.cumsum([a[1].shape[0] for a in args])
        words = (C.c_void_p * max(n, 1))(*[a[0].ctypes.data for a in args])
        sizes = (C.c_size_t * max(n, 1))(*[a[0].size for a in args])
        codes = (C.c_int * max(n, 1))(*([-1] * max(n, 1)))
        msgs = C.create_string_buffer(max(n, 1) * MESSAGE_BYTES)
        rc = self.L.lib.pb254_verify_many_device(self._h, kind, C.byref(config) if config is not None else None, words,
                                                 sizes, n, _p(inputs), _p(timestamps), _p(starts), codes, msgs)
        if rc in (4, 5) or any(codes[b] == -1 for b in range(n)):
            self.L.check(rc)
        return [None if codes[b] == 0 else
                (codes[b], msgs.raw[b * MESSAGE_BYTES:(b + 1) * MESSAGE_BYTES].split(b"\0", 1)[0].decode())
                for b in range(n)]

    def prove_sharded(self, kind, inputs, timestamps, rank: int, world: int, all_to_all, all_gather,
                      min_rows=1 << 16, config: Config | None = None):
        """pb254_prove_sharded: one proof across `world` ranks, every rank calling with the same inputs.
        all_to_all(send_ptr, recv_ptr, bytes_per_peer) / all_gather(send_ptr, recv_ptr, bytes_per_rank) get raw pointers
        on this context's device and must run on (or be ordered with) the context's stream; see dist.TorchCollectives."""
        inputs = _u64(inputs)
        timestamps = _u64(timestamps)
        assert inputs.ndim == 2 and inputs.shape[1] == self.L.input_words(kind)
        errors = []

        def wrap(fn):
            def cb(_user, send, recv, nbytes):
                try:
                    fn(int(send), int(recv), int(nbytes))
                    return 0
                except Exception as e:  # an exception must not cross the C frames
                    errors.append(e)
                    return 1
            return _COLL_FN(cb)
        comm = Comm(rank, world, None, wrap(all_to_all), wrap(all_gather))
        h = C.c_void_p()
        rc = self.L.lib.pb254_prove_sharded(self._h, C.c_int(kind), _p(inputs), _p(timestamps),
                                            C.c_size_t(inputs.shape[0]), C.c_size_t(min_rows),
                                            C.byref(config) if config is not None else None, C.byref(comm), C.byref(h))
        if errors:
            raise errors[0]
        self.L.check(rc)
        return Proof(self.L, h)

    def prove_dev(self, kind, d_inputs_ptr: int, d_timestamps_ptr: int, n_inputs: int, min_rows=1 << 16,
                  config: Config | None = None):
        """pb254_prove_dev: inputs and timestamps are device pointers on this context's GPU."""
        h = C.c_void_p()
        self.L.check(self.L.lib.pb254_prove_dev(self._h, C.c_int(kind), C.c_void_p(d_inputs_ptr),
                                                C.c_void_p(d_timestamps_ptr), C.c_size_t(n_inputs),
                                                C.c_size_t(min_rows),
                                                C.byref(config) if config is not None else None, C.c_int(0),
                                                C.byref(h)))
        return Proof(self.L, h)

    def prove_trace(self, kind, trace_cols, config: Config | None = None, keep_debug=False):
        t = _u64(trace_cols)
        assert t.shape[0] == self.L.trace_width(kind)
        h = C.c_void_p()
        self.L.check(self.L.lib.pb254_prove_trace(self._h, C.c_int(kind), _p(t), C.c_size_t(t.shape[1]),
                                                  C.byref(config) if config is not None else None,
                                                  C.c_int(int(keep_debug)), C.byref(h)))
        return Proof(self.L, h)


class Proof:
    """Owned pb254_proof handle."""

    def __init__(self, library: Library, handle):
        self.L = library
        self._h = handle

    def close(self):
        if getattr(self, "_h", None):
            self.L.lib.pb254_proof_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def words(self) -> np.ndarray:
        n = self.L.lib.pb254_proof_words(self._h)
        p = self.L.lib.pb254_proof_data(self._h)
        return np.ctypeslib.as_array(p, shape=(n,)).copy()

    def bytes(self) -> bytes:
        return self.words().tobytes()

    def results(self) -> np.ndarray:
        """(n_inputs, L) 16-bit limbs of the native outputs s*x + offset / x^s, read from the trace."""
        n = self.L.lib.pb254_proof_results_words(self._h)
        if n == 0:
            return np.zeros((0, 0), dtype=np.uint64)
        p = self.L.lib.pb254_proof_results_data(self._h)
        return np.ctypeslib.as_array(p, shape=(n,)).copy()

    def debug(self, which: int) -> np.ndarray:
        n = self.L.lib.pb254_proof_debug_words(self._h, which)
        if n == 0:
            return np.zeros(0, dtype=np.uint64)
        p = self.L.lib.pb254_proof_debug_data(self._h, which)
        return np.ctypeslib.as_array(p, shape=(n,)).copy()
