"""The fused operand table of the tensor-core Poseidon (csrc/poseidon_constants_tcf.inc: two partial rounds per
u8 x u8 -> s32 product, read by csrc/poseidon_tc.cuh) checked without a GPU. The tile is un-swizzled, its entries are
compared with M P M, M e0 and the fused round constants, and the kernel's schedule - 4 full rounds through the
one-round tile (poseidon_constants_tcb.inc), 11 fused layers, 4 full rounds - is replayed with numpy integers,
including the A row the kernel writes, the thread's own row-0 product (dp2a pieces) and the byte-weight fold, bit for
bit as the kernel does them. Whole permutations must equal the oracle's Poseidon."""
import os
import re

import numpy as np

from util import rand_field

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
P = 0xFFFFFFFF00000001
M32, M64 = (1 << 32) - 1, (1 << 64) - 1
CIRC = [17, 15, 41, 16, 2, 28, 13, 13, 39, 18, 34, 20]
MDS = np.array([[CIRC[(i - r) % 12] + (8 if r == i == 0 else 0) for i in range(12)] for r in range(12)], dtype=np.int64)
PZ = np.diag([0] + [1] * 11).astype(np.int64)      # zeroes lane 0
MPM = MDS @ PZ @ MDS
FUSED_ROUNDS = list(range(4, 26, 2))                  # a fused layer j takes partial rounds 4 + 2 j and 5 + 2 j


def load_tile(name):
    txt = open(os.path.join(ROOT, "plonky2_bn254_b200", "csrc", name)).read()
    words = [int(w, 16) for w in re.findall(r"0x([0-9a-fA-F]{8})u", txt)]
    assert len(words) == 96 * 128 // 4
    img = np.array(words, dtype="<u4").view(np.uint8)
    tile = np.zeros((96, 128), dtype=np.int64)
    for n in range(96):                       # 16-byte chunk c of row n is stored at chunk position c ^ (n & 7)
        for c in range(8):
            pos = n * 128 + ((c ^ (n & 7)) << 4)
            tile[n, 16 * c:16 * c + 16] = img[pos:pos + 16]
    return tile


def fused_constants(rc):
    """C_j = M P RC[r + 1] + RC[r + 2] - 255 sum_i hi(M P M [.][i]), r = 4 + 2 j, per output lane, mod p."""
    out = []
    for r in FUSED_ROUNDS:
        c1 = [0] + rc[12 * (r + 1) + 1:12 * (r + 2)]
        out.append([(sum(int(MDS[ro][k]) * c1[k] for k in range(12)) + rc[12 * (r + 2) + ro]
                     - 255 * sum(int(v) >> 8 for v in MPM[ro])) % P for ro in range(12)])
    return out


def test_fused_tile_entries(oracle):
    B = load_tile("poseidon_constants_tcf.inc")
    rc = [int(x) for x in oracle.poseidon_round_constants()]
    consts = fused_constants(rc)
    assert MPM.min() == 3872 and MPM.max() == 6520     # non-negative, < 2^13: one lo byte and a hi byte <= 25
    for ro in range(12):
        for w in range(8):
            row = B[8 * ro + w]
            for i in range(12):
                lo, hi = int(MPM[ro][i]) & 0xFF, int(MPM[ro][i]) >> 8
                for q in range(8):
                    want = lo if q == w else hi if q == w - 1 or (w == 4 and q == 7) else 0
                    assert row[8 * i + q] == want, (ro, w, i, q)
                assert row[115 + i] == (hi if w == 0 else 0)
            assert (row[96:104] == [MDS[ro][0] if q == w else 0 for q in range(8)]).all()
            for j in range(11):
                assert row[104 + j] == (consts[j][ro] >> (8 * w)) & 0xFF
            assert row[127] == 0


def recombine4(a0, a1, a2, a3):
    """poseidon_tc.cuh recombine4, instruction for instruction (u32 registers, carry flags)."""
    lo = a0 + ((a1 & 0xFFFF) << 16)
    hi = (a1 >> 16) + a2 + (lo >> 32)
    lo &= M32
    assert hi <= M32
    hi += (a3 & 0xFFFF) << 16
    w2 = (a3 >> 16) + (hi >> 32)
    hi = (hi & M32) + w2
    c = hi >> 32
    x = ((((hi & M32) << 32) | lo) - w2) & M64
    return (x + (M32 if c else 0)) & M64


def fold(acc):
    out = []
    for r in range(12):
        q = [int(v) for v in acc[8 * r:8 * r + 8]]
        a = [q[2 * k] + (q[2 * k + 1] << 8) for k in range(4)]
        assert max(a) <= M32
        out.append(recombine4(*a))
    return out


def row0_plus(s, rc, r):
    """u0 = row 0 of MDS s + RC[r + 1][0] as the thread computes it: dp2a on 16-bit pieces seeded by the constant."""
    k = rc[12 * (r + 1)]
    acc = [((k >> (16 * q)) & 0xFFFF) + sum(int(MDS[0][i]) * ((s[i] >> (16 * q)) & 0xFFFF) for i in range(12))
           for q in range(4)]
    assert max(acc) < 1 << 25
    return recombine4(*acc)


def sbox(x):
    return pow(x, 7, P)


def bytes_of(x):
    return [(x >> (8 * q)) & 0xFF for q in range(8)]


def fused_high(t, j, s):
    """k = 96 .. 127 of a fused layer: sbox(u0), the one-hot of the layer, the complement bytes, a zero."""
    hi = [0] * 32
    hi[0:8] = bytes_of(t)
    hi[8 + j] = 1
    for i in range(12):
        hi[19 + i] = 255 - (s[i] >> 56)
    return hi


def product(B, s, high, stats):
    a = np.array([b for x in s for b in bytes_of(x)] + high, dtype=np.int64)
    acc = B @ a
    stats["max"] = max(stats["max"], int(acc.max()))
    assert acc.max() < 1 << 20
    return fold(acc)


def test_fused_layer_equals_two_partial_rounds_on_lazy_states(oracle):
    Bf = load_tile("poseidon_constants_tcf.inc")
    rc = [int(x) for x in oracle.poseidon_round_constants()]
    rng = np.random.default_rng(5)
    edges = [0, 1, P - 1, P, P + 1, M64, M64 - 1, M32, M32 << 32, (1 << 63)]
    stats = {"max": 0}
    def lane():  # any u64 representative: random, non-canonical (>= p), or an edge value
        kind = int(rng.integers(0, 3))
        if kind == 0:
            return (int(rng.integers(0, 1 << 32)) << 32) | int(rng.integers(0, 1 << 32))
        if kind == 1:
            return P + int(rng.integers(0, M32))
        return edges[int(rng.integers(0, len(edges)))]

    for trial in range(44):
        s = [lane() for _ in range(12)]
        j = trial % 11
        r = FUSED_ROUNDS[j]
        s1 = [sbox(s[0])] + s[1:]                          # round r's S-box (its constant is already in s)
        t = sbox(row0_plus(s1, rc, r))
        got = [x % P for x in product(Bf, s1, fused_high(t, j, s1), stats)]
        v = [x % P for x in s1]
        for rr in (r, r + 1):                              # two plain partial rounds, from the MDS of round r on
            if rr == r + 1:
                v[0] = sbox(v[0])
            v = [(int(sum(int(MDS[ro][i]) * v[i] for i in range(12))) + rc[12 * (rr + 1) + ro]) % P for ro in range(12)]
        assert got == v, (trial, j)
    assert 0 < stats["max"] < 1 << 20


def test_replayed_fused_permutation_equals_the_oracle(oracle):
    B, Bf = load_tile("poseidon_constants_tcb.inc"), load_tile("poseidon_constants_tcf.inc")
    rc = [int(x) for x in oracle.poseidon_round_constants()]
    rng = np.random.default_rng(17)
    states = [list(map(int, s)) for s in rand_field(rng, (5, 12))]
    states[0] = [0] * 12
    states[1] = [P - 1] * 12
    stats = {"max": 0}
    for st in states:
        # three permutations back to back through the same A row, as a sponge hashes a long row
        want = np.array(st, dtype=np.uint64)
        s = list(st)
        high = [0] * 32                                    # k = 96 .. 127 of this thread's A row
        for _ in range(3):
            want = oracle.poseidon_permute(want)
            s = [(x + rc[i]) % P for i, x in enumerate(s)]
            for L in range(19):
                if L < 4 or L >= 15:
                    R = L if L < 4 else L + 11             # full rounds 0-3 and 26-29
                    s = [sbox(x) for x in s]
                    high = [0] * 32
                    if R < 29:
                        high[R] = 1                        # adds the constants of round R + 1
                    s = product(B, s, high, stats)
                else:
                    j = L - 4
                    s[0] = sbox(s[0])
                    high = fused_high(sbox(row0_plus(s, rc, FUSED_ROUNDS[j])), j, s)
                    s = product(Bf, s, high, stats)
            assert high == [0] * 32                        # the row ends every permutation without layer bytes
            s = [x % P for x in s]
            assert s == [int(x) for x in want]
    assert 0 < stats["max"] < 1 << 20
