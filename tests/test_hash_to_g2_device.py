"""pb254_map_to_g2 / pb254_hash_to_g2 (K14): the hash_to_g2 witness (src/utils/hash_to_g2.rs:76-148, cofactor clearing
:195-208) built on the device. The contract is the Python restatement in workloads.py, word for word: map_to_curve,
hash_to_g2_inputs with the oracle's Poseidon, and the oracle's native_result minus the offset for the hashes.
CPU part on the host-simulation build, GPU part on the product library."""
import ctypes as C

import numpy as np
import pytest

from plonky2_bn254_b200 import ffi, inputs as I, workloads as Wk
from util import rand_field

P = I.BN254_P
F2 = I._Fq2
GAMMA = 0x9E3779B97F4A7C15


def oracle_permute(oracle):
    return lambda st: np.stack([oracle.poseidon_permute(r) for r in np.asarray(st, dtype=np.uint64).reshape(-1, 12)])


def u_words(us):
    return np.array([I._words(u[0]) + I._words(u[1]) for u in us], dtype=np.uint64).reshape(-1, 8)


def limbs_to_words(limbs):
    """16-bit limbs (native_result layout) -> little-endian u64 words."""
    l = np.asarray(limbs, dtype=np.uint64).reshape(-1, 4)
    return l[:, 0] | (l[:, 1] << np.uint64(16)) | (l[:, 2] << np.uint64(32)) | (l[:, 3] << np.uint64(48))


def point_words(pts):
    return np.array([Wk._g2_words(p) for p in pts], dtype=np.uint64).reshape(-1, 16)


def svdw_branch(u):
    """Which of x1, x2, x3 workloads._map_with_tv4 takes for u (recomputed, not read from the code under test)."""
    one = (1, 0)
    t = F2.mul(F2.mul(u, u), Wk._GZ)
    tv1, tv2 = F2.sub(one, t), F2.add(one, t)
    tv5 = F2.mul(F2.mul(F2.mul(u, tv1), F2.inv(F2.mul(tv1, tv2))), Wk._TV4)
    if Wk._fq2_is_qr(Wk._g(F2.sub(Wk._NEG_Z_BY_TWO, tv5))):
        return 1
    return 2 if Wk._fq2_is_qr(Wk._g(F2.add(Wk._NEG_Z_BY_TWO, tv5))) else 3


def exceptional_us():
    """The four u with tv1 * tv2 = 0: u^2 = +-1 / g(Z)."""
    out = []
    for sign in (1, -1):
        r = I.fq2_sqrt(F2.mul((sign % P, 0), F2.inv(Wk._GZ)))
        assert r is not None                           # 1/g(Z) and -1/g(Z) are squares in Fq2
        out += [r, F2.sub((0, 0), r)]
    assert len(set(out)) == 4
    return out


def hashes_from_rows(oracle, rows, offsets):
    """native_result(G2, row) - offset: the hash_to_g2 outputs of the serial reference."""
    res = np.array([oracle.native_result(I.KIND_G2, r) for r in rows])
    return point_words(Wk.hash_to_g2_outputs(res, offsets))


def check_hash_to_g2(ctx, oracle, msgs, seed):
    rows, ts, offs = Wk.hash_to_g2_inputs(msgs, oracle_permute(oracle), seed)
    inputs, hashes = ctx.hash_to_g2(msgs, seed)
    assert inputs.shape == rows.shape and (inputs == rows).all()
    assert (hashes == hashes_from_rows(oracle, rows, offs)).all()
    return inputs, hashes


def code_of(fn, *args):
    with pytest.raises(ffi.Pb254Error) as e:
        fn(*args)
    return e.value.code, str(e.value)


# ---- CPU: host-simulation build ------------------------------------------------------------------------------------
def test_map_to_g2_random_u_all_branches_hostsim(hostsim_ctx):
    rng = I.SplitMix64(2025)
    us = [(rng.bits256() % P, rng.bits256() % P) for _ in range(64)]
    assert {svdw_branch(u) for u in us} == {1, 2, 3}
    got = hostsim_ctx.map_to_g2(u_words(us))
    assert (got == point_words([Wk.map_to_curve(u) for u in us])).all()


def test_map_to_g2_chosen_u_hostsim(hostsim_ctx):
    c = 0x1234567890ABCDEF1234567890ABCDEF1234567890ABCDEF
    us = [(0, 0), (0, c), (c, 0), (0, 1), (1, 0), (P - 1, P - 1)]
    got = hostsim_ctx.map_to_g2(u_words(us))
    assert (got == point_words([Wk.map_to_curve(u) for u in us])).all()


def test_map_to_g2_exceptional_u_hostsim(hostsim_ctx):
    rng = I.SplitMix64(5)
    for u in exceptional_us():
        with pytest.raises(ValueError):
            Wk.map_to_curve(u)
        us = [(rng.bits256() % P, rng.bits256() % P) for _ in range(5)]
        us[2] = us[4] = u
        code, msg = code_of(hostsim_ctx.map_to_g2, u_words(us))
        assert code == 6 and "index 2:" in msg and "exceptional" in msg


def test_map_to_g2_argument_errors_hostsim(hostsim_ctx):
    us = u_words([(3, 4), (5, 6), (7, 8)])
    for col in (0, 4):                                 # c0 = p, c1 = p
        bad = us.copy()
        bad[1, col:col + 4] = I._words(P)
        code, msg = code_of(hostsim_ctx.map_to_g2, bad)
        assert code == 3 and "index 1:" in msg
    assert hostsim_ctx.map_to_g2(np.zeros((0, 8), dtype=np.uint64)).shape == (0, 16)
    code, _ = code_of(hostsim_ctx.map_to_g2, np.zeros(((1 << 17) + 1, 8), dtype=np.uint64))
    assert code == 6
    lib, out = hostsim_ctx.L.lib, np.empty((3, 16), dtype=np.uint64)
    assert lib.pb254_map_to_g2(hostsim_ctx._h, None, C.c_size_t(3), out.ctypes.data_as(C.c_void_p)) == 6
    assert lib.pb254_map_to_g2(hostsim_ctx._h, us.ctypes.data_as(C.c_void_p), C.c_size_t(3), None) == 6
    assert lib.pb254_map_to_g2(None, us.ctypes.data_as(C.c_void_p), C.c_size_t(3),
                               out.ctypes.data_as(C.c_void_p)) == 6


@pytest.mark.parametrize("seed", [7, 0xFFFFFFFFFFFFFFF0])
@pytest.mark.parametrize("ln", [0, 3, 8, 13, 16])
def test_hash_to_g2_equals_python_hostsim(hostsim_ctx, oracle, ln, seed):
    msgs = rand_field(np.random.default_rng(ln + 10), (5, ln))
    msgs[0, :min(ln, 2)] = Wk.GOLDILOCKS_P - 1             # the largest canonical element
    check_hash_to_g2(hostsim_ctx, oracle, msgs, seed)


def test_hash_to_g2_inputs_device_hostsim(hostsim_ctx, oracle):
    msgs = rand_field(np.random.default_rng(3), (4, 6))
    inputs, ts, offs, hashes = Wk.hash_to_g2_inputs_device(hostsim_ctx, msgs, seed=11)
    rows, ts_py, offs_py = Wk.hash_to_g2_inputs(msgs, oracle_permute(oracle), 11)
    assert (inputs == rows).all() and (ts == ts_py).all() and offs == offs_py
    for row, off, h in zip(inputs, offs, hashes):
        x = Wk._g2_from_words(row[4:20])
        assert h == Wk.g2_mul(Wk.G2_COFACTOR, x)
        assert Wk.g2_add(h, off) == Wk._g2_from_words(
            limbs_to_words(oracle.native_result(I.KIND_G2, row)))


def test_hash_to_g2_argument_errors_hostsim(hostsim_ctx):
    msgs = rand_field(np.random.default_rng(1), (6, 5))
    bad = msgs.copy()
    bad[4, 2] = Wk.GOLDILOCKS_P
    bad[5, 0] = 2**64 - 1
    code, msg = code_of(hostsim_ctx.hash_to_g2, bad, 1)
    assert code == 3 and "index 4:" in msg
    inputs, hashes = hostsim_ctx.hash_to_g2(np.zeros((0, 5), dtype=np.uint64), 1)
    assert inputs.shape == (0, 36) and hashes.shape == (0, 16)
    for shape in (((1 << 17) + 1, 0), (1, (1 << 24) + 1), (2, (1 << 23) + 1)):   # n, msg_len, n * msg_len caps
        code, _ = code_of(hostsim_ctx.hash_to_g2, np.zeros(shape, dtype=np.uint64), 1)
        assert code == 6
    lib = hostsim_ctx.L.lib
    out36, out16 = np.empty((6, 36), dtype=np.uint64), np.empty((6, 16), dtype=np.uint64)
    p = lambda a: a.ctypes.data_as(C.c_void_p)
    call = lambda ctx, m, a, b: lib.pb254_hash_to_g2(ctx, m, C.c_size_t(6), C.c_size_t(5), C.c_uint64(1), a, b)
    assert call(hostsim_ctx._h, None, p(out36), p(out16)) == 6
    assert call(hostsim_ctx._h, p(msgs), None, p(out16)) == 6
    assert call(hostsim_ctx._h, p(msgs), p(out36), None) == 6
    assert call(None, p(msgs), p(out36), p(out16)) == 6


# ---- GPU ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n", [1024, 300])           # 300 singleton chains: 600 scan elements cross block boundaries
def test_hash_to_g2_parity_gpu(gpu_ctx, oracle, n):
    msgs = rand_field(np.random.default_rng(n), (n, 8))
    check_hash_to_g2(gpu_ctx, oracle, msgs, seed=n + 1)


@pytest.mark.gpu
def test_map_to_g2_gpu(gpu_ctx):
    rng = I.SplitMix64(77)
    us = [(rng.bits256() % P, rng.bits256() % P) for _ in range(256)] + [(0, 0), (0, 5), (5, 0)]
    assert (gpu_ctx.map_to_g2(u_words(us)) == point_words([Wk.map_to_curve(u) for u in us])).all()
    code, msg = code_of(gpu_ctx.map_to_g2, u_words(us[:3] + exceptional_us()[:1]))
    assert code == 6 and "index 3:" in msg


@pytest.mark.gpu
def test_hash_to_g2_largest_batch_gpu(gpu_ctx, oracle):
    n, seed = 1 << 17, 99
    msgs = rand_field(np.random.default_rng(17), (n, 3))
    inputs, hashes = gpu_ctx.hash_to_g2(msgs, seed)
    assert inputs.shape == (n, 36) and hashes.shape == (n, 16)
    idx = np.random.default_rng(5).choice(n, size=64, replace=False)
    idx[:2] = [0, n - 1]
    us = Wk.hash_to_fq2(msgs[idx], oracle_permute(oracle))
    for i, u in zip(idx, us):
        rng = I.SplitMix64(seed + 4 * int(i) * GAMMA)    # counter-based: the state after 4i draws
        k = rng.bits256() & ((1 << 254) - 1)
        x = Wk.map_to_curve(u)
        want = I._words(Wk.G2_COFACTOR) + Wk._g2_words(x) + Wk._g2_words(I.scalar_mul_gen(I.KIND_G2, k))
        assert list(inputs[i]) == want
        assert list(hashes[i]) == Wk._g2_words(Wk.g2_mul(Wk.G2_COFACTOR, x))


@pytest.mark.gpu
def test_hash_to_g2_end_to_end_proof_gpu(gpu_ctx, oracle):
    msgs = rand_field(np.random.default_rng(128), (128, 5))
    inputs, ts, offs, hashes = Wk.hash_to_g2_inputs_device(gpu_ctx, msgs, seed=128)
    pf = gpu_ctx.prove(I.KIND_G2, inputs, ts)
    assert Wk.hash_to_g2_outputs(pf.results(), offs) == hashes
    assert all(h is not None and Wk.g2_mul(I.BN254_R, h) is None for h in hashes)
    assert oracle.verify(pf.words(), inputs, ts)
