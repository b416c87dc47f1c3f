"""pb254_verify_device (ffi.Context.verify) against pb254_verify (ffi.Library.verify): on every input both return the
same outcome - both accept, or both raise with the same code and the same message. The CPU tests run the
host-simulation build, where the device stages run one work item per thread; the GPU tests run the product library."""
import ctypes as C

import numpy as np
import pytest

from plonky2_bn254_b200 import ffi, inputs as I, workloads as Wk
from util import GL_P


def both(ctx, kind, words, inp, ts, config=None):
    """None if both verifiers accept, else the common (code, message)."""
    outs = []
    for verify in (ctx.L.verify, ctx.verify):
        try:
            assert verify(kind, words, inp, ts, config=config) is True
            outs.append(None)
        except ffi.Pb254Error as e:
            outs.append((e.code, str(e)))
    assert outs[0] == outs[1], outs
    return outs[0]


def bump(words, pos):
    w = words.copy()
    w[pos] = np.uint64((int(w[pos]) + 1) % GL_P)
    return w


def tamper_positions(lib, words):
    """(name, word offset) of one word of every section of the proof, from the ProofView layout: caps, challenger
    state, openings, commit-phase caps, the first and last query record (leaves, paths, layer evals and paths),
    final polynomial and proof-of-work witness. Query-record entries are marked with query=True."""
    lay = lib.parse_proof(words).layout
    out = [(n, int(getattr(lay, n)), False) for n in (
        "trace_cap", "auxiliary_polys_cap", "quotient_polys_cap", "init_challenger_state", "local_values",
        "next_values", "auxiliary_polys", "auxiliary_polys_next", "ctl_zs_first", "quotient_polys")]
    out += [(f"commit_phase_cap{i}", int(lay.commit_phase_merkle_caps) + i * int(lay.cap_words), False)
            for i in range(lay.num_fri_layers)]
    nq = int(lay.config.num_query_rounds)
    for q in (0, nq - 1):
        rec = int(lay.query_round_proofs) + q * int(lay.query_words)
        for n in ("q_trace_leaf", "q_trace_path", "q_aux_leaf", "q_aux_path", "q_quotient_leaf", "q_quotient_path"):
            out.append((f"query{q}.{n}", rec + int(getattr(lay, n)), True))
        for i in range(lay.num_fri_layers):
            out.append((f"query{q}.step{i}.evals", rec + int(lay.q_step_evals[i]), True))
            if lay.q_step_path_words[i]:
                out.append((f"query{q}.step{i}.path", rec + int(lay.q_step_path[i]), True))
    out += [("final_poly", int(lay.final_poly), False), ("pow_witness", int(lay.pow_witness), False)]
    return out


def sweep(ctx, kind, words, inp, ts, config=None):
    for name, pos, in_query in tamper_positions(ctx.L, words):
        got = both(ctx, kind, bump(words, pos), inp, ts, config)
        assert got is not None and got[0] == 7, (name, got)
        if in_query:
            assert "Merkle path" in got[1] or "FRI layer" in got[1], (name, got)


def ordering(ctx, kind, words, inp, ts):
    """A FRI-layer sibling of query 2 and a trace leaf of query 5: the earlier query's failure is reported."""
    lay = ctx.L.parse_proof(words).layout
    rec = lambda q: int(lay.query_round_proofs) + q * int(lay.query_words)
    w = bump(bump(words, rec(2) + int(lay.q_step_path[0])), rec(5) + int(lay.q_trace_leaf))
    assert both(ctx, kind, w, inp, ts) == (7, "pb254 error 7 (E_VERIFY): verify: Merkle path of the FRI layer tree")


def zero_combination_timestamp(words_debug_challenges, inp_row, nch=2):
    """The timestamp that makes instance's input combination under challenge 0 zero: the input tuple is the limbs of
    words 4.. then of words 0..4 then the timestamp, combined as sum t_i beta^i + gamma."""
    beta, gamma = int(words_debug_challenges[0]), int(words_debug_challenges[nch])
    words = [int(v) for v in inp_row[4:]] + [int(v) for v in inp_row[:4]]
    limbs = [(wd >> (16 * i)) & 0xFFFF for wd in words for i in range(4)]
    acc = sum(l * pow(beta, i, GL_P) for i, l in enumerate(limbs)) + gamma
    return (-acc * pow(pow(beta, len(limbs), GL_P), -1, GL_P)) % GL_P


# ---- CPU (host-simulation build) -------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def g1_case(oracle):
    inp, ts = I.make_inputs(I.KIND_G1, 2, I.config_seed(70))
    pf, _, _ = oracle.prove_inputs(I.KIND_G1, inp, ts)
    return {"words": pf.words(), "inputs": inp, "timestamps": ts}


def test_accepts_oracle_proofs(hostsim_ctx, fq_case, g1_case):
    assert both(hostsim_ctx, I.KIND_FQ, fq_case["words"], fq_case["inputs"], fq_case["timestamps"]) is None
    assert both(hostsim_ctx, I.KIND_G1, g1_case["words"], g1_case["inputs"], g1_case["timestamps"]) is None
    names = [n for n, _ in hostsim_ctx.timings()]
    assert names == ["verify native ctl", "verify merkle"]


def test_tampering_sweep(hostsim_ctx, fq_case):
    sweep(hostsim_ctx, I.KIND_FQ, fq_case["words"], fq_case["inputs"], fq_case["timestamps"])


def test_earlier_query_wins(hostsim_ctx, fq_case):
    ordering(hostsim_ctx, I.KIND_FQ, fq_case["words"], fq_case["inputs"], fq_case["timestamps"])


def test_wrong_public_inputs(hostsim_ctx, g1_case):
    c, w, inp, ts = hostsim_ctx, g1_case["words"], g1_case["inputs"], g1_case["timestamps"]
    for row, col in ((1, 4), (1, 0), (0, 13)):  # x coordinate, scalar, offset coordinate
        bad = inp.copy()
        bad[row, col] ^= np.uint64(1)
        assert both(c, I.KIND_G1, w, bad, ts) == (7, "pb254 error 7 (E_VERIFY): verify: cross-table lookup sum")
    assert both(c, I.KIND_G1, w, inp, ts + np.uint64(1))[1].endswith("cross-table lookup sum")


def test_non_canonical_and_infinity_instances(hostsim_ctx, g1_case):
    c, w, inp, ts = hostsim_ctx, g1_case["words"], g1_case["inputs"], g1_case["timestamps"]
    non_canonical = inp.copy()
    non_canonical[1, 8:12] = np.uint64(0xFFFFFFFFFFFFFFFF)
    assert both(c, I.KIND_G1, w, non_canonical, ts)[0] == 3
    s_is_r = inp.copy()
    s_is_r[1, 0:4] = I._words(I.BN254_R)  # r * x reaches infinity inside the ladder
    got = both(c, I.KIND_G1, w, s_is_r, ts)
    assert got[0] == 2 and "intermediate point at infinity" in got[1]
    # two bad instances: the lower one's error is reported, whichever kind it is
    two = s_is_r.copy()
    two[0, 8:12] = np.uint64(0xFFFFFFFFFFFFFFFF)
    assert both(c, I.KIND_G1, w, two, ts)[0] == 3
    two = non_canonical.copy()
    two[0, 0:4] = I._words(I.BN254_R)
    assert both(c, I.KIND_G1, w, two, ts)[0] == 2


def test_zero_combination(hostsim_ctx, fq_case):
    ch = fq_case["proof"].debug(2)
    ts = fq_case["timestamps"].copy()
    ts[1] = np.uint64(zero_combination_timestamp(ch, fq_case["inputs"][1]))
    got = both(hostsim_ctx, I.KIND_FQ, fq_case["words"], fq_case["inputs"], ts)
    assert got == (7, "pb254 error 7 (E_VERIFY): verify: CTL combination is zero")


@pytest.mark.parametrize("field,value", [(6, 1), (7, 0), (5, 1), (3, 2), (4, 3), (8, 3), (9, 4)])
def test_weakened_header(hostsim_ctx, fq_case, field, value):
    w = fq_case["words"].copy()
    w[field] = np.uint64(value)
    got = both(hostsim_ctx, I.KIND_FQ, w, fq_case["inputs"], fq_case["timestamps"])
    assert got[0] == 7 and "header" in got[1]


def test_kind_config_truncation_and_periods(hostsim_ctx, fq_case):
    c, w, inp, ts = hostsim_ctx, fq_case["words"], fq_case["inputs"], fq_case["timestamps"]
    assert both(c, I.KIND_FQ, w[:-5], inp, ts)[0] == 7
    assert both(c, I.KIND_FQ, np.zeros(100, dtype=np.uint64), inp, ts)[0] == 7
    g1_inp, g1_ts = I.make_inputs(I.KIND_G1, 3, I.config_seed(71))
    assert both(c, I.KIND_G1, w, g1_inp, g1_ts)[0] == 7
    w2 = w.copy()
    w2[1] = np.uint64(I.KIND_G2)
    assert both(c, I.KIND_FQ, w2, inp, ts)[0] == 7
    with pytest.raises(ffi.Pb254Error) as e:  # wrong shape for the caller's kind: refused on the Python side
        c.verify(I.KIND_G2, w2, inp, ts)
    assert e.value.code == 6
    cfg = c.L.standard_fast_config()
    cfg.num_query_rounds = 100
    assert both(c, I.KIND_FQ, w, inp, ts, config=cfg)[0] == 7
    assert both(c, I.KIND_FQ, w, inp, ts, config=c.L.standard_fast_config()) is None
    many, many_ts = I.make_inputs(I.KIND_FQ, 129, I.config_seed(72))  # a 2^16-row trace holds 128 instances
    assert both(c, I.KIND_FQ, w, many, many_ts)[0] == 7


def test_argument_errors(hostsim_ctx, fq_case):
    L = hostsim_ctx.L
    w, inp, ts = fq_case["words"], fq_case["inputs"], fq_case["timestamps"]
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    call = lambda ctx, kind, pw, pi, pt: L.lib.pb254_verify_device(ctx, C.c_int(kind), None, pw, C.c_size_t(w.size),
                                                                   pi, pt, C.c_size_t(inp.shape[0]))
    assert call(hostsim_ctx._h, I.KIND_FQ, p(w), p(inp), p(ts)) == 0
    assert call(None, I.KIND_FQ, p(w), p(inp), p(ts)) == 6
    assert L.lib.pb254_last_error() == b"null context"
    for args in ((None, p(inp), p(ts)), (p(w), None, p(ts)), (p(w), p(inp), None)):
        assert call(hostsim_ctx._h, I.KIND_FQ, *args) == 6
        assert L.lib.pb254_last_error() == b"null argument"
    assert call(hostsim_ctx._h, 3, p(w), p(inp), p(ts)) == 6
    assert b"unknown STARK kind" in L.lib.pb254_last_error()


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def config2(gpu_ctx):
    inp, ts = I.make_inputs(I.KIND_G1, 1024, I.config_seed(2))
    return gpu_ctx.prove(I.KIND_G1, inp, ts).words(), inp, ts


@pytest.mark.gpu
def test_gpu_config2_g1_1024(gpu_ctx, config2):
    w, inp, ts = config2
    assert both(gpu_ctx, I.KIND_G1, w, inp, ts) is None
    assert [n for n, _ in gpu_ctx.timings()] == ["verify native ctl", "verify merkle"]


@pytest.mark.gpu
def test_gpu_config2_wrong_public_inputs(gpu_ctx, config2):
    w, inp, ts = config2
    bad = inp.copy()
    bad[700, 0] ^= np.uint64(4)
    assert both(gpu_ctx, I.KIND_G1, w, bad, ts)[1].endswith("cross-table lookup sum")
    bad = inp.copy()
    bad[900, 0:4] = I._words(I.BN254_R)
    bad[901, 4:8] = np.uint64(0xFFFFFFFFFFFFFFFF)
    assert both(gpu_ctx, I.KIND_G1, w, bad, ts)[0] == 2
    assert both(gpu_ctx, I.KIND_G1, w, inp, ts + np.uint64(1))[1].endswith("cross-table lookup sum")


@pytest.mark.gpu
def test_gpu_config3_g2_1024(gpu_ctx):
    inp, ts = I.make_inputs(I.KIND_G2, 1024, I.config_seed(3))
    assert both(gpu_ctx, I.KIND_G2, gpu_ctx.prove(I.KIND_G2, inp, ts).words(), inp, ts) is None


@pytest.mark.gpu
def test_gpu_config4_fq_4096_blowup8(gpu_ctx):
    cfg = gpu_ctx.L.standard_fast_config()
    cfg.rate_bits, cfg.num_query_rounds = 3, 28
    inp, ts = I.make_inputs(I.KIND_FQ, 4096, I.config_seed(4))
    w = gpu_ctx.prove(I.KIND_FQ, inp, ts, config=cfg).words()
    assert both(gpu_ctx, I.KIND_FQ, w, inp, ts, config=cfg) is None


@pytest.mark.gpu
def test_gpu_hash_to_g2_batch(gpu_ctx):
    """x = map_to_curve(...) lies outside the prime-order subgroup: the ladder handles it as the host does."""
    msgs = np.random.default_rng(6).integers(0, 1 << 32, size=(256, 4), dtype=np.uint64)
    inputs, ts, _, _ = Wk.hash_to_g2_inputs_device(gpu_ctx, msgs, seed=6)
    assert both(gpu_ctx, I.KIND_G2, gpu_ctx.prove(I.KIND_G2, inputs, ts).words(), inputs, ts) is None


@pytest.mark.gpu
def test_gpu_g1_msm_chain(gpu_ctx):
    rng = I.SplitMix64(15)
    pts = [I.scalar_mul_gen(I.KIND_G1, rng.bits256() % I.BN254_R) for _ in range(64)]
    scalars = [rng.bits256() for _ in range(64)]
    inputs, ts, _ = Wk.g1_msm_inputs(gpu_ctx, scalars, pts, seed=15)
    assert both(gpu_ctx, I.KIND_G1, gpu_ctx.prove(I.KIND_G1, inputs, ts).words(), inputs, ts) is None


@pytest.mark.gpu
def test_gpu_tampering_sweep_and_ordering(gpu_ctx):
    inp, ts = I.make_inputs(I.KIND_G1, 5, I.config_seed(73))
    w = gpu_ctx.prove(I.KIND_G1, inp, ts).words()
    assert int(w[2]) == 16
    assert both(gpu_ctx, I.KIND_G1, w, inp, ts) is None
    sweep(gpu_ctx, I.KIND_G1, w, inp, ts)
    ordering(gpu_ctx, I.KIND_G1, w, inp, ts)
