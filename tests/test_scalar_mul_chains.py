"""pb254_scalar_mul_chains (K13): chained scalar multiplications, the witness G1/G2SingleGenerator computes before
run_once (src/generators/g1/single.rs:48-52) and g1_msm threads through its offsets (src/utils/g1_msm.rs:22-36).
The reference is the oracle's native_result applied serially, term by term, exactly as the generator loop runs:
acc_(i+1) = native_result(s_i, x_i, acc_i). CPU part on the host-simulation build, GPU part on the product library."""
import numpy as np
import pytest

from plonky2_bn254_b200 import ffi, inputs as I, workloads as Wk

P = I.BN254_P
FW = {I.KIND_G1: 4, I.KIND_G2: 8}


def limbs_to_words(limbs):
    """16-bit limbs (native_result / Proof.results() layout) -> little-endian u64 words."""
    l = np.asarray(limbs, dtype=np.uint64).reshape(-1, 4)
    return l[:, 0] | (l[:, 1] << np.uint64(16)) | (l[:, 2] << np.uint64(32)) | (l[:, 3] << np.uint64(48))


def serial_chains(oracle, kind, terms, starts, offsets):
    rows, sums = [], []
    for c in range(len(starts) - 1):
        acc = np.asarray(offsets[c], dtype=np.uint64)
        for i in range(int(starts[c]), int(starts[c + 1])):
            row = np.concatenate([terms[i], acc])
            rows.append(row)
            acc = limbs_to_words(oracle.native_result(kind, row))
        sums.append(acc)
    tw = 4 + 4 * FW[kind]
    return np.array(rows, dtype=np.uint64).reshape(-1, tw), np.array(sums, dtype=np.uint64).reshape(-1, 2 * FW[kind])


def random_case(kind, lengths, seed):
    """terms, chain_starts, offsets for chains of the given lengths (points k * G, random 256-bit scalars)."""
    n = sum(lengths)
    inp, _ = I.make_inputs(kind, max(n, len(lengths)), seed)
    tw = 4 + 2 * FW[kind]
    terms = inp[:n, :tw].copy()
    offsets = inp[:len(lengths), tw:].copy()
    starts = np.concatenate([[0], np.cumsum(lengths)]).astype(np.uint64)
    return terms, starts, offsets


def check(ctx, oracle, kind, terms, starts, offsets):
    rows, sums = ctx.scalar_mul_chains(kind, terms, starts, offsets)
    want_rows, want_sums = serial_chains(oracle, kind, terms, starts, offsets)
    assert rows.shape == want_rows.shape and (rows == want_rows).all()
    assert (sums == want_sums).all()
    return rows, sums


def g1_point(words):
    return (Wk._int256(words[0:4]), Wk._int256(words[4:8]))


# ---- CPU: host-simulation build ------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind", [I.KIND_G1, I.KIND_G2])
@pytest.mark.parametrize("lengths", [[40], [1] * 6, [3, 0, 7, 1, 0, 12]], ids=["one_chain", "singletons", "mixed"])
def test_chains_equal_serial_oracle_hostsim(hostsim_ctx, oracle, kind, lengths):
    terms, starts, offsets = random_case(kind, lengths, 1000 + len(lengths))
    check(hostsim_ctx, oracle, kind, terms, starts, offsets)


def test_chains_cross_checked_with_python_curve_arithmetic(hostsim_ctx):
    terms, starts, offsets = random_case(I.KIND_G1, [4], 77)
    rows, sums = hostsim_ctx.scalar_mul_chains(I.KIND_G1, terms, starts, offsets)
    acc = g1_point(offsets[0])
    for i in range(4):
        assert g1_point(rows[i, 12:20]) == acc
        acc = Wk.g1_add(Wk.g1_mul(Wk._int256(terms[i, :4]), g1_point(terms[i, 4:12])), acc)
    assert g1_point(sums[0]) == acc
    # G2: one singleton
    t2, s2, o2 = random_case(I.KIND_G2, [1], 78)
    _, sums2 = hostsim_ctx.scalar_mul_chains(I.KIND_G2, t2, s2, o2)
    want = Wk.g2_add(Wk.g2_mul(Wk._int256(t2[0, :4]), Wk._g2_from_words(t2[0, 4:20])), Wk._g2_from_words(o2[0]))
    assert Wk._g2_from_words(sums2[0]) == want


@pytest.mark.parametrize("kind", [I.KIND_G1, I.KIND_G2])
def test_special_scalars(hostsim_ctx, oracle, kind):
    """s = 0 and s = r give s * x = infinity (the accumulator stays), s = 2^256 - 1 is not reduced."""
    terms, starts, offsets = random_case(kind, [5, 2], 31)
    for i, s in ((0, 0), (1, I.BN254_R), (3, (1 << 256) - 1), (5, 0), (6, (1 << 256) - 1)):
        terms[i, :4] = I._words(s)
    rows, sums = check(hostsim_ctx, oracle, kind, terms, starts, offsets)
    assert (rows[1, -2 * FW[kind]:] == rows[0, -2 * FW[kind]:]).all() and (rows[2, -2 * FW[kind]:] == offsets[0]).all()


@pytest.mark.parametrize("kind", [I.KIND_G1, I.KIND_G2])
def test_infinity_names_the_term(hostsim_ctx, oracle, kind):
    terms, starts, offsets = random_case(kind, [2, 4, 3], 55)
    rows, _ = serial_chains(oracle, kind, terms, starts, offsets)
    bad = 4  # chain 1, index 2 in the chain: x = -acc_4, s = 1
    fw = FW[kind]
    acc = rows[bad, 4 + 2 * fw:]
    neg_y = [(P - Wk._int256(acc[fw + 4 * k:fw + 4 * k + 4])) % P for k in range(fw // 4)]
    terms[bad, :4] = I._words(1)
    terms[bad, 4:4 + fw] = acc[:fw]
    terms[bad, 4 + fw:] = np.array(sum((I._words(v) for v in neg_y), []), dtype=np.uint64)
    with pytest.raises(ffi.Pb254Error) as e:
        hostsim_ctx.scalar_mul_chains(kind, terms, starts, offsets)
    assert e.value.code == 2
    assert "chain 1, term 4 (index 2 in the chain)" in str(e.value)


def test_input_errors(hostsim_ctx):
    kind = I.KIND_G1
    terms, starts, offsets = random_case(kind, [3, 2], 9)

    def code(t=terms, s=starts, o=offsets, k=kind):
        with pytest.raises(ffi.Pb254Error) as e:
            hostsim_ctx.scalar_mul_chains(k, t, s, o)
        return e.value.code

    t = terms.copy()
    t[1, 4:8] = I._words(P)                       # x.x = p: not canonical
    assert code(t=t) == 3
    t = terms.copy()
    t[2, 4:12] = I._words(1) + I._words(1)        # (1, 1): not on y^2 = x^3 + 3
    assert code(t=t) == 8
    o = offsets.copy()
    o[1, :8] = I._words(1) + I._words(1)          # an offset off the curve
    assert code(o=o) == 8
    for bad in ([0, 4, 3, 5], [1, 3, 5], [0, 3, 4]):   # decreasing, not starting at 0, not ending at n_terms
        assert code(s=np.array(bad, dtype=np.uint64), o=np.resize(offsets, (len(bad) - 1, 8))) == 6
    assert code(k=I.KIND_FQ) == 6
    big = np.zeros(((1 << 17) + 1, 12), dtype=np.uint64)
    assert code(t=big, s=np.array([0, big.shape[0]], dtype=np.uint64), o=offsets[:1]) == 6


def test_g1_msm_inputs_hostsim(hostsim_ctx):
    rng = I.SplitMix64(5)
    pts = [I.scalar_mul_gen(I.KIND_G1, rng.bits256() % I.BN254_R) for _ in range(6)]
    scalars = [rng.bits256() for _ in range(6)]
    inputs, ts, msm = Wk.g1_msm_inputs(hostsim_ctx, scalars, pts, seed=3)
    want = None
    for s, p in zip(scalars, pts):
        want = Wk.g1_add(want, Wk.g1_mul(s, p))
    assert msm == want and inputs.shape == (6, 20) and (ts == np.arange(6)).all()
    assert Wk.g1_msm_inputs(hostsim_ctx, [0, I.BN254_R], pts[:2], seed=3)[2] is None


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("lengths", [[1024], [128] * 64], ids=["g1_msm_1024", "64x128"])
def test_g1_chains_gpu(gpu_ctx, oracle, lengths):
    terms, starts, offsets = random_case(I.KIND_G1, lengths, 2024)
    check(gpu_ctx, oracle, I.KIND_G1, terms, starts, offsets)


@pytest.mark.gpu
@pytest.mark.parametrize("lengths", [
    [128, 3],                         # the second chain's head is element 129: a block boundary is the first term
    [127, 1, 5],                      # chain 1's head exactly at element 128, the start of block 1
    [1000],                           # one chain through every block of the first level
    [0, 300, 0, 0, 17, 1, 2000, 0],   # empty chains, n_terms + n_chains not a multiple of the block size
    [5] * 3000 + [1],                 # a second and a third scan level (18001 + 3001 elements)
], ids=["head_after_boundary", "head_on_boundary", "spanning", "mixed_empty", "three_levels"])
def test_scan_edge_cases_gpu(gpu_ctx, oracle, lengths):
    terms, starts, offsets = random_case(I.KIND_G1, lengths, 7 + len(lengths))
    check(gpu_ctx, oracle, I.KIND_G1, terms, starts, offsets)


@pytest.mark.gpu
def test_g1_chain_end_to_end_proof(gpu_ctx, oracle):
    """The chained 1024-term batch proves and verifies, and the trace's own outputs continue the chain."""
    terms, starts, offsets = random_case(I.KIND_G1, [1024], 2024)
    rows, sums = gpu_ctx.scalar_mul_chains(I.KIND_G1, terms, starts, offsets)
    ts = np.arange(1024, dtype=np.uint64)
    pf = gpu_ctx.prove(I.KIND_G1, rows, ts)
    assert gpu_ctx.L.verify(I.KIND_G1, pf.words(), rows, ts)
    res = pf.results().reshape(1024, 32)
    out = np.array([limbs_to_words(r) for r in res])
    assert (out[:-1] == rows[1:, 12:20]).all()
    assert (out[-1] == sums[0]).all()


@pytest.mark.gpu
def test_g2_singletons_from_hash_to_g2_gpu(gpu_ctx, oracle):
    rng = np.random.default_rng(3)
    msgs = rng.integers(0, Wk.GOLDILOCKS_P, size=(1024, 8), dtype=np.uint64)
    inp, ts, _ = Wk.hash_to_g2_inputs(msgs, gpu_ctx.poseidon_permute, seed=4)
    terms, offsets = inp[:, :20].copy(), inp[:, 20:].copy()
    starts = np.arange(1025, dtype=np.uint64)
    rows, sums = check(gpu_ctx, oracle, I.KIND_G2, terms, starts, offsets)
    assert (rows == inp).all()
    pf = gpu_ctx.prove(I.KIND_G2, rows, ts)
    res = pf.results().reshape(1024, 64)
    assert (np.array([limbs_to_words(r) for r in res]) == sums).all()


@pytest.mark.gpu
def test_g1_msm_inputs_gpu(gpu_ctx):
    rng = I.SplitMix64(8)
    pts = [I.scalar_mul_gen(I.KIND_G1, rng.bits256() % I.BN254_R) for _ in range(16)]
    scalars = [rng.bits256() for _ in range(16)]
    inputs, ts, msm = Wk.g1_msm_inputs(gpu_ctx, scalars, pts, seed=9)
    want = None
    for s, p in zip(scalars, pts):
        want = Wk.g1_add(want, Wk.g1_mul(s, p))
    assert msm == want
