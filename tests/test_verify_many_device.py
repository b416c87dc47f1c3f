"""pb254_verify_many_device (ffi.Context.verify_many): every proof of a batch gets exactly the outcome pb254_verify
(ffi.Library.verify) gives it alone, whatever the other proofs contain and in any order; the return code and
pb254_last_error() name the lowest rejected proof. The CPU tests run the host-simulation build; the GPU tests run the
product library."""
import ctypes as C
import os
import re
import time

import numpy as np
import pytest

from plonky2_bn254_b200 import ffi, inputs as I, workloads as Wk
from test_verify_device import bump, zero_combination_timestamp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ["verify native ctl", "verify merkle"]


def alone(verify, L, kind, words, inp, ts, config=None):
    """None if `verify` accepts the proof, else (code, pb254_last_error())."""
    try:
        assert verify(kind, words, inp, ts, config=config) is True
        return None
    except ffi.Pb254Error as e:
        return e.code, L.lib.pb254_last_error().decode()


def check_batch(ctx, kind, entries, config=None, reference=None):
    """verify_many on entries [(words, inputs, timestamps)] against `reference` (Library.verify by default) on each
    entry alone; also checks the last error names the lowest rejected proof. Returns the outcomes."""
    reference = reference or ctx.L.verify
    want = [alone(reference, ctx.L, kind, w, i, t, config) for w, i, t in entries]
    got = ctx.verify_many(kind, [e[0] for e in entries], [(e[1], e[2]) for e in entries], config=config)
    assert got == want
    bad = [b for b, o in enumerate(want) if o is not None]
    if bad:
        assert ctx.L.lib.pb254_last_error().decode() == f"proof {bad[0]}: {want[bad[0]][1]}"
    return got


class Raw:
    """The C entry point with caller-built arrays, for the argument checks."""

    def __init__(self, L, words, n_inputs, n):
        self.L, self.w = L, words
        self.words = (C.c_void_p * n)(*[words.ctypes.data] * n)
        self.sizes = (C.c_size_t * n)(*[words.size] * n)
        self.starts = np.arange(n + 1, dtype=np.uint64) * np.uint64(n_inputs)
        self.codes = (C.c_int * n)(*[-7] * n)
        self.msgs = C.create_string_buffer(n * ffi.MESSAGE_BYTES)

    def __call__(self, ctx, kind, inp, ts, n, words="default", sizes="default", starts=None):
        words = self.words if isinstance(words, str) else words
        sizes = self.sizes if isinstance(sizes, str) else sizes
        starts = self.starts if starts is None else starts
        return self.L.lib.pb254_verify_many_device(ctx, kind, None, words, sizes, n, ffi._p(inp), ffi._p(ts),
                                                   ffi._p(starts), self.codes, self.msgs)


# ---- CPU (host-simulation build) -------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def g1_case(oracle):
    inp, ts = I.make_inputs(I.KIND_G1, 2, I.config_seed(70))
    pf, _, _ = oracle.prove_inputs(I.KIND_G1, inp, ts)
    return {"words": pf.words(), "inputs": inp, "timestamps": ts}


def fq_entries(L, case):
    """Valid copies and one rejection of every kind the walk has, for the fq oracle proof."""
    w, inp, ts = case["words"], case["inputs"], case["timestamps"]
    lay = L.parse_proof(w).layout
    rec0 = int(lay.query_round_proofs)
    bumped = [bump(w, int(getattr(lay, n))) for n in ("trace_cap", "init_challenger_state", "local_values",
                                                      "ctl_zs_first", "final_poly", "pow_witness")]
    bumped += [bump(w, rec0 + int(lay.q_trace_leaf)), bump(w, rec0 + int(lay.q_step_path[0]))]
    header = w.copy()
    header[7] = np.uint64(0)  # no grinding
    zts = ts.copy()
    zts[1] = np.uint64(zero_combination_timestamp(case["proof"].debug(2), inp[1]))
    wrong = inp.copy()
    wrong[0, 4] ^= np.uint64(1)
    entries = [(w, inp, ts)] + [(b, inp, ts) for b in bumped[:4]] + [(w, inp, ts)] + [(b, inp, ts) for b in bumped[4:]]
    entries += [(header, inp, ts), (w[:-5], inp, ts), (w, wrong, ts), (w, inp, zts),
                (w, inp[:0], ts[:0]), (w, inp, ts)]
    return entries


def g1_entries(case):
    w, inp, ts = case["words"], case["inputs"], case["timestamps"]
    wrong = inp.copy()
    wrong[1, 4] ^= np.uint64(1)
    non_canonical = inp.copy()
    non_canonical[1, 8:12] = np.uint64(0xFFFFFFFFFFFFFFFF)
    s_is_r = inp.copy()
    s_is_r[1, 0:4] = I._words(I.BN254_R)
    two = s_is_r.copy()
    two[0, 8:12] = np.uint64(0xFFFFFFFFFFFFFFFF)
    return [(w, inp, ts), (w, wrong, ts), (w, non_canonical, ts), (w, inp, ts), (w, s_is_r, ts), (w, two, ts),
            (w, inp, ts + np.uint64(1)), (w, inp[:0], ts[:0]), (w, inp, ts)]


def test_mixed_batch_matches_the_host_verifier(hostsim_ctx, fq_case):
    entries = fq_entries(hostsim_ctx.L, fq_case)
    got = check_batch(hostsim_ctx, I.KIND_FQ, entries)
    assert got[0] is None and got[5] is None and got[-1] is None
    assert sum(o is not None for o in got) == len(entries) - 3
    assert [n for n, _ in hostsim_ctx.timings()] == NAMES
    check_batch(hostsim_ctx, I.KIND_FQ, entries[::-1])
    rng = np.random.default_rng(5)
    check_batch(hostsim_ctx, I.KIND_FQ, [entries[i] for i in rng.permutation(len(entries))])


def test_native_failures_stay_with_their_proof(hostsim_ctx, g1_case):
    entries = g1_entries(g1_case)
    got = check_batch(hostsim_ctx, I.KIND_G1, entries)
    assert [o and o[0] for o in got] == [None, 7, 3, None, 2, 3, 7, 7, None]
    check_batch(hostsim_ctx, I.KIND_G1, entries[::-1])
    rng = np.random.default_rng(6)
    check_batch(hostsim_ctx, I.KIND_G1, [entries[i] for i in rng.permutation(len(entries))])


def test_no_walk_is_left_waiting(hostsim_ctx, fq_case):
    w, inp, ts = fq_case["words"], fq_case["inputs"], fq_case["timestamps"]
    t0 = time.monotonic()
    got = check_batch(hostsim_ctx, I.KIND_FQ, [(w[:-1], inp, ts)] * 5)  # every walk ends before start()
    assert all(o[0] == 7 for o in got)
    assert hostsim_ctx.timings() == []  # no device round
    got = check_batch(hostsim_ctx, I.KIND_FQ, [(w[:-1], inp, ts)] * 4 + [(w, inp, ts)])  # only the last starts
    assert got[-1] is None
    assert check_batch(hostsim_ctx, I.KIND_FQ, [(w, inp, ts)]) == [None]
    assert hostsim_ctx.verify_many(I.KIND_FQ, [], []) == []
    assert time.monotonic() - t0 < 300


def test_two_rounds(hostsim_ctx, fq_case):
    """66 proofs are two rounds of at most 64: each has its own device stages, and proofs keep their indices."""
    w, inp, ts = fq_case["words"], fq_case["inputs"], fq_case["timestamps"]
    valid = {0, 63, 64, 65}
    entries = [(w, inp, ts) if b in valid else (w[:-1], inp, ts) for b in range(66)]
    entries[65] = (w, inp, ts + np.uint64(1))
    got = check_batch(hostsim_ctx, I.KIND_FQ, entries)
    assert [b for b, o in enumerate(got) if o is None] == [0, 63, 64]
    assert got[65][1].endswith("cross-table lookup sum")
    assert [n for n, _ in hostsim_ctx.timings()] == NAMES * 2


def test_argument_errors(hostsim_ctx, fq_case):
    L = hostsim_ctx.L
    w, inp, ts = fq_case["words"], fq_case["inputs"], fq_case["timestamps"]
    raw = Raw(L, w, inp.shape[0], 2)
    both_inp, both_ts = np.concatenate([inp, inp]), np.concatenate([ts, ts])
    call = lambda *a, **k: raw(hostsim_ctx._h, I.KIND_FQ, both_inp, both_ts, 2, *a, **k)
    assert call() == 0 and list(raw.codes) == [0, 0]
    raw.codes[0] = raw.codes[1] = -7

    def refused(rc, message):
        assert rc == 6 and L.lib.pb254_last_error().decode() == message
        assert list(raw.codes) == [-7, -7]

    refused(raw(None, I.KIND_FQ, both_inp, both_ts, 2), "null context")
    refused(call(words=None), "null argument")
    refused(call(sizes=None), "null argument")
    refused(call(words=(C.c_void_p * 2)(w.ctypes.data, None)), "null proof_words entry")
    refused(call(starts=np.array([0, 4, 3], dtype=np.uint64)), "input_starts must not decrease")
    refused(call(starts=np.array([1, 3, 6], dtype=np.uint64)), "input_starts[0] must be 0")
    refused(raw(hostsim_ctx._h, 3, both_inp, both_ts, 2), "unknown STARK kind (0 = G1, 1 = G2, 2 = Fq)")
    refused(raw(hostsim_ctx._h, I.KIND_FQ, both_inp, both_ts, (1 << 12) + 1), "more than 2^12 proofs")
    with pytest.raises(ffi.Pb254Error) as e:  # shapes are refused on the Python side
        hostsim_ctx.verify_many(I.KIND_G1, [w], [(inp, ts)])
    assert e.value.code == 6
    with pytest.raises(ffi.Pb254Error) as e:
        hostsim_ctx.verify_many(I.KIND_FQ, [w, w], [(inp, ts)])
    assert e.value.code == 6


def test_messages_out_may_be_null(hostsim_ctx, fq_case):
    L = hostsim_ctx.L
    w, inp, ts = fq_case["words"], fq_case["inputs"], fq_case["timestamps"]
    raw = Raw(L, w, inp.shape[0], 1)
    rc = L.lib.pb254_verify_many_device(hostsim_ctx._h, I.KIND_FQ, None, raw.words, raw.sizes, 1, ffi._p(inp),
                                        ffi._p(ts + np.uint64(1)), ffi._p(raw.starts), raw.codes, None)
    assert rc == 7 and list(raw.codes) == [7]
    assert L.lib.pb254_last_error().decode() == "proof 0: verify: cross-table lookup sum"


def test_ctypes_declaration_matches_the_header():
    src = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "pb254.h")).read(), flags=re.S)
    params = re.search(r"int\s+pb254_verify_many_device\s*\(([^)]*)\)", src).group(1)
    types = [re.sub(r"\s+", " ", re.sub(r"\s*\b\w+$", "", p.strip())).replace(" *", "*") for p in params.split(",")]
    to_ctypes = {"pb254_ctx*": C.c_void_p, "int": C.c_int, "const pb254_config*": C.POINTER(ffi.Config),
                 "const uint64_t* const*": C.POINTER(C.c_void_p), "const size_t*": C.POINTER(C.c_size_t),
                 "size_t": C.c_size_t, "const uint64_t*": C.c_void_p, "int*": C.POINTER(C.c_int),
                 "char*": C.POINTER(C.c_char)}
    assert "#define PB254_VERIFY_MESSAGE_BYTES 256" in src and ffi.MESSAGE_BYTES == 256
    from plonky2_bn254_b200 import build
    L = ffi.Library(build.build_hostsim())
    assert L.lib.pb254_verify_many_device.argtypes == [to_ctypes[t] for t in types]
    assert L.lib.pb254_verify_many_device.restype == C.c_int


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_gpu_32_batches_one_launch_per_stage(gpu_ctx):
    batches = [I.make_inputs(I.KIND_G1, 128, I.config_seed(800 + b)) for b in range(32)]
    proofs = [p.words() for p in ffi.prove_many([gpu_ctx], I.KIND_G1, batches)]
    n0 = gpu_ctx.L.launch_count()
    assert gpu_ctx.verify(I.KIND_G1, proofs[0], *batches[0])
    one = gpu_ctx.L.launch_count() - n0
    n0 = gpu_ctx.L.launch_count()
    assert gpu_ctx.verify_many(I.KIND_G1, proofs, batches) == [None] * 32
    assert gpu_ctx.L.launch_count() - n0 == one == 4
    assert [n for n, _ in gpu_ctx.timings()] == NAMES


@pytest.mark.gpu
def test_gpu_mixed_sizes_and_tampering(gpu_ctx):
    L = gpu_ctx.L
    cases = []
    for n, seed in ((1024, 2), (5, 810), (1024, 811), (200, 812), (128, 813), (256, 814)):
        inp, ts = I.make_inputs(I.KIND_G1, n, I.config_seed(seed))
        cases.append((gpu_ctx.prove(I.KIND_G1, inp, ts).words(), inp, ts))
    assert sorted({int(c[0][2]) for c in cases}) == [16, 17, 19]
    entries = list(cases)
    for w, inp, ts in cases[:4]:
        lay = L.parse_proof(w).layout
        rec = int(lay.query_round_proofs) + 7 * int(lay.query_words)
        entries.append((bump(w, rec + int(lay.q_step_path[1])), inp, ts))
        wrong = inp.copy()
        wrong[-1, 0] ^= np.uint64(4)
        entries.append((w, wrong, ts))
    bad = cases[0][1].copy()
    bad[900, 0:4] = I._words(I.BN254_R)
    bad[901, 4:8] = np.uint64(0xFFFFFFFFFFFFFFFF)
    entries.append((cases[0][0], bad, cases[0][2]))
    entries.append((cases[2][0][:-3], cases[2][1], cases[2][2]))
    order = np.random.default_rng(7).permutation(len(entries))
    entries = [entries[i] for i in order]
    got = check_batch(gpu_ctx, I.KIND_G1, entries, reference=gpu_ctx.verify)
    assert sum(o is None for o in got) == len(cases)
    small = [e for e in entries if int(e[0][2]) == 16]
    assert len(small) >= 4
    check_batch(gpu_ctx, I.KIND_G1, small)


@pytest.mark.gpu
def test_gpu_g2_batch_with_hash_to_g2(gpu_ctx):
    batches = [I.make_inputs(I.KIND_G2, 128, I.config_seed(820 + b)) for b in range(3)]
    msgs = np.random.default_rng(8).integers(0, 1 << 32, size=(128, 4), dtype=np.uint64)
    inputs, ts, _, _ = Wk.hash_to_g2_inputs_device(gpu_ctx, msgs, seed=8)
    batches.append((inputs, ts))
    proofs = [gpu_ctx.prove(I.KIND_G2, i, t).words() for i, t in batches]
    assert gpu_ctx.verify_many(I.KIND_G2, proofs, batches) == [None] * 4


@pytest.mark.gpu
def test_gpu_fq_batch_blowup8(gpu_ctx):
    cfg = gpu_ctx.L.standard_fast_config()
    cfg.rate_bits, cfg.num_query_rounds = 3, 28
    batches = [I.make_inputs(I.KIND_FQ, n, I.config_seed(830 + n)) for n in (128, 1000, 4096)]
    proofs = [gpu_ctx.prove(I.KIND_FQ, i, t, config=cfg).words() for i, t in batches]
    assert gpu_ctx.verify_many(I.KIND_FQ, proofs, batches, config=cfg) == [None] * 3
    assert check_batch(gpu_ctx, I.KIND_FQ, [(proofs[0], *batches[0]), (proofs[1], *batches[0])], config=cfg,
                       reference=gpu_ctx.verify)[1] is not None
