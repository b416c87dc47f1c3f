"""Batch workload generators for the G2 and fq_exp STARKs (SURVEY.md section 8f, rank 4): the two places of the
reference that produce large batches of hot-path work items.

* ``is_square`` (src/fields/fq.rs:283-295): the Legendre symbol ``x^((p-1)/2)`` of every value goes through
  ``fq_exp``; a batch of values is a batch of ``FqExpInput {s: (p-1)/2, x}`` and the STARK's native results are the
  symbols (1 = square, p-1 = non-square, 0 = zero).
* ``hash_to_g2`` (src/utils/hash_to_g2.rs:68-148 native, :151-209 circuit): ``hash_to_fq2`` (a Poseidon challenger over
  the message, 2 x 16 challenges, low 32 bits each, reduced mod p) -> Shallue-van de Woestijne map to the curve
  y^2 = x^3 + 3/(9+u) -> cofactor clearing, which the circuit does as ``g2_scalar_mul(cofactor, point, offset)``
  with a random offset (:195-208) followed by ``- offset``. A batch of messages is a batch of
  ``G2ScalarMulInput {s: cofactor, x: mapped point, offset}``; ``hash_to_g2_outputs`` removes the offsets from the
  STARK's native results. ``hash_to_g2_inputs_device`` builds the same batch, and the hashes, on the device
  (``Context.hash_to_g2``).
* ``g1_msm`` (src/utils/g1_msm.rs:22-36): a chain of G1 scalar-muls threaded through ``offset`` from a random subgroup
  point; ``g1_msm_inputs`` builds the batch on the device (``Context.scalar_mul_chains``) and returns the MSM.

Host-side, pure Python / numpy: this is workload generation (what the reference's witness generators do on the CPU
before they reach ``run_once``), not part of the prover. The Poseidon permutation is injected (``Context.poseidon_permute``
on the GPU; the tests also run it against the CPU oracle's permutation).
"""
from __future__ import annotations

import numpy as np

from . import inputs as I
from .inputs import BN254_P, BN254_R, _Fq2 as F2

GOLDILOCKS_P = 0xFFFFFFFF00000001
LEGENDRE_EXPONENT = (BN254_P - 1) // 2            # (Fq::from(-1) / Fq::from(2)).into(), fq.rs:290
G2_COFACTOR = 21888242871839275222246405745257275088844257914179612981679871602714643921549  # hash_to_g2.rs:68-74
NUM_MODULUS_LIMBS = 8                              # 256-bit modulus in u32 limbs


# ---- is_square -----------------------------------------------------------------------------------------------
def is_square_inputs(xs):
    """FqExpInput batch for the Legendre symbols of ``xs`` (ints mod p): (inputs[n, 8], timestamps[n])."""
    rows = [I._words(LEGENDRE_EXPONENT) + I._words(int(x) % BN254_P) for x in xs]
    return np.array(rows, dtype=np.uint64).reshape(len(rows), 8), np.arange(len(rows), dtype=np.uint64)


def _int256(words) -> int:
    return sum(int(w) << (64 * i) for i, w in enumerate(words))


def _from_limbs16(limbs) -> int:
    """A 256-bit value from the 16 little-endian 16-bit limbs of the trace (src/starks/mod.rs:13-20)."""
    return sum(int(w) << (16 * i) for i, w in enumerate(limbs))


def is_square_outputs(results) -> np.ndarray:
    """``legendre.is_equal(one)`` (fq.rs:293-294) for the native results ``x^((p-1)/2)`` of an fq_exp proof
    (``Proof.results()``: 16 limbs of 16 bits per instance, as they stand in the trace)."""
    return np.array([_from_limbs16(r) == 1 for r in np.asarray(results).reshape(-1, 16)], dtype=bool)


# ---- hash_to_fq2 ---------------------------------------------------------------------------------------------
def hash_to_fq2(messages, permute):
    """``HashToG2::hash_to_fq2`` (hash_to_g2.rs:76-87) for a batch of equally long messages.

    messages: [n, len] canonical Goldilocks elements; permute: callable [n, 12] uint64 -> [n, 12] uint64, the Poseidon
    permutation. plonky2 0.2.2 ``Challenger``: observed elements overwrite the rate lanes 8 at a time (duplexing =
    overwrite + permute), challenges are popped from the END of the 8 rate lanes, an empty output buffer triggers one
    more permutation. Returns a list of n (c0, c1) pairs."""
    m = np.ascontiguousarray(np.asarray(messages, dtype=np.uint64))
    n, ln = m.shape
    state = np.zeros((n, 12), dtype=np.uint64)
    perm = lambda st: np.ascontiguousarray(np.asarray(permute(st), dtype=np.uint64).reshape(n, 12))
    buf, have, pending = None, 0, 0                   # output buffer (the 8 rate lanes), how many are left, buffered inputs
    for pos in range(0, ln, 8):                       # observe_elements
        take = min(8, ln - pos)
        state[:, :take] = m[:, pos:pos + take]
        have = 0                                      # observe_element clears the output buffer
        if take == 8:                                 # a full input buffer is absorbed at once: duplexing
            state = perm(state)
            buf, have = state[:, :8].copy(), 8
        else:
            pending = take
    out = []                                          # challenges in the order get_challenge returns them
    for _ in range(4 * NUM_MODULUS_LIMBS):
        if pending or have == 0:                      # buffered inputs or no outputs left -> duplexing
            state = perm(state)
            buf, have, pending = state[:, :8].copy(), 8, 0
        have -= 1
        out.append(buf[:, have])                      # Vec::pop takes from the end
    out = np.stack(out, axis=1)                       # [n, 32]
    res = []
    for row in out:
        vals = []
        for half in range(2):
            v = 0
            for i, c in enumerate(row[16 * half:16 * half + 16]):
                v += (int(c) & 0xFFFFFFFF) << (32 * i)      # f_slice_to_biguint: the low 32 bits of each challenge
            vals.append(v % BN254_P)
        res.append((vals[0], vals[1]))
    return res


# ---- map_to_g2 (RFC 9380 6.6.1, Shallue-van de Woestijne, Z = 1) -------------------------------------------------
def _g(x):
    return F2.add(F2.mul(F2.mul(x, x), x), I.G2_B)


def _neg(a):
    return F2.sub((0, 0), a)


def _fq_sgn(a: int) -> bool:
    return (a % BN254_P) & 1 == 1


def fq2_sgn(a) -> bool:
    """src/fields/sgn.rs:20-27."""
    return _fq_sgn(a[0]) or (a[0] % BN254_P == 0 and _fq_sgn(a[1]))


def _fq2_is_qr(a) -> bool:
    if a == (0, 0):
        return False
    norm = (a[0] * a[0] + a[1] * a[1]) % BN254_P      # a is a square in Fq2 iff its norm is a square in Fq
    return pow(norm, (BN254_P - 1) // 2, BN254_P) == 1


_Z = (1, 0)
_GZ = _g(_Z)
_NEG_Z_BY_TWO = F2.mul(_neg(_Z), F2.inv((2, 0)))
_TV4 = I.fq2_sqrt(F2.mul(F2.mul(_neg(_GZ), (3, 0)), F2.mul(_Z, _Z)))
_TV6 = F2.mul(F2.mul(_neg((4, 0)), _GZ), F2.inv(F2.mul((3, 0), F2.mul(_Z, _Z))))


def map_to_curve(u):
    """The point of the G2 CURVE (before cofactor clearing) of ``HashToG2::map_to_g2`` (hash_to_g2.rs:113-147).
    Square roots follow ark-ff's algorithms, which fix WHICH root is returned (tv4's choice decides which of x1, x2 is
    tried first): Fq by a^((p+1)/4) (p = 3 mod 4), Fq2 by the complex method with delta = (norm_sqrt + c0)/2, falling back
    to delta - norm_sqrt when delta is a non-residue (``inputs.fq2_sqrt``). y's sign is then fixed by sgn(u)."""
    return _map_with_tv4(u, _TV4)


def _map_with_tv4(u, tv4):
    one = (1, 0)
    tv1 = F2.mul(F2.mul(u, u), _GZ)
    tv2 = F2.add(one, tv1)
    tv1 = F2.sub(one, tv1)
    tv3 = F2.inv(F2.mul(tv1, tv2))
    tv5 = F2.mul(F2.mul(F2.mul(u, tv1), tv3), tv4)
    x1 = F2.sub(_NEG_Z_BY_TWO, tv5)
    x2 = F2.add(_NEG_Z_BY_TWO, tv5)
    t = F2.mul(F2.mul(tv2, tv2), tv3)
    x3 = F2.add(_Z, F2.mul(_TV6, F2.mul(t, t)))
    if _fq2_is_qr(_g(x1)):
        x = x1
    elif _fq2_is_qr(_g(x2)):
        x = x2
    else:
        x = x3
    y = I.fq2_sqrt(_g(x))
    assert y is not None
    if fq2_sgn(u) != fq2_sgn(y):
        y = _neg(y)
    assert F2.mul(y, y) == _g(x)
    return (x, y)


# ---- G2 arithmetic for the offsets -------------------------------------------------------------------------------
def g2_neg(P):
    return (P[0], _neg(P[1]))


def g2_add(P, Q):
    """Affine addition on the G2 curve; None is the point at infinity."""
    if P is None:
        return Q
    if Q is None:
        return P
    if P[0] == Q[0]:
        if F2.add(P[1], Q[1]) == (0, 0):
            return None
        lam = F2.mul(F2.mul((3, 0), F2.mul(P[0], P[0])), F2.inv(F2.mul((2, 0), P[1])))
    else:
        lam = F2.mul(F2.sub(Q[1], P[1]), F2.inv(F2.sub(Q[0], P[0])))
    x = F2.sub(F2.sub(F2.mul(lam, lam), P[0]), Q[0])
    return (x, F2.sub(F2.mul(lam, F2.sub(P[0], x)), P[1]))


def g2_mul(k: int, P):
    acc = None
    for bit in bin(k)[2:]:
        acc = g2_add(acc, acc)
        if bit == "1":
            acc = g2_add(acc, P)
    return acc


def _g2_words(P):
    return I._words(P[0][0]) + I._words(P[0][1]) + I._words(P[1][0]) + I._words(P[1][1])


def _g2_from_words(w):
    return ((_int256(w[0:4]), _int256(w[4:8])), (_int256(w[8:12]), _int256(w[12:16])))


def _g2_from_limbs16(l):
    return ((_from_limbs16(l[0:16]), _from_limbs16(l[16:32])), (_from_limbs16(l[32:48]), _from_limbs16(l[48:64])))


def _g2_limbs16(P):
    return [(c >> (16 * i)) & 0xFFFF for c in (P[0][0], P[0][1], P[1][0], P[1][1]) for i in range(16)]


def hash_to_g2_inputs(messages, permute, seed: int):
    """G2ScalarMulInput batch of the cofactor clearings of ``hash_to_g2`` over ``messages`` (hash_to_g2.rs:195-203):
    s = cofactor, x = map_to_curve(hash_to_fq2(message)), offset = a random subgroup point (``set_random_g2``).
    Returns (inputs[n, 36], timestamps[n], offsets) - keep ``offsets`` for ``hash_to_g2_outputs``."""
    us = hash_to_fq2(messages, permute)
    rng = I.SplitMix64(seed)
    rows, offsets = [], []
    for u in us:
        pt = map_to_curve(u)
        k = 0
        while k % BN254_R == 0:
            k = rng.bits256() & ((1 << 254) - 1)
        off = I.scalar_mul_gen(I.KIND_G2, k)
        offsets.append(off)
        rows.append(I._words(G2_COFACTOR) + _g2_words(pt) + _g2_words(off))
    return (np.array(rows, dtype=np.uint64).reshape(len(rows), 36), np.arange(len(rows), dtype=np.uint64), offsets)


def hash_to_g2_inputs_device(ctx, messages, seed: int):
    """``hash_to_g2_inputs`` built on the device (``Context.hash_to_g2``): the same rows whenever no drawn k is 0 mod r
    (the device fails with E_BAD_ARG where Python would draw again, probability about 2^-253 per message).
    Returns (inputs[n, 36], timestamps[n], offsets, hashes); offsets and hashes are affine points (x, y) of Fq2 pairs,
    so that ``hash_to_g2_outputs(results, offsets)`` applies unchanged, and hashes[i] is the hash_to_g2 output."""
    inputs, hashes = ctx.hash_to_g2(messages, seed)
    offsets = [_g2_from_words(r[20:36]) for r in inputs]
    return inputs, np.arange(inputs.shape[0], dtype=np.uint64), offsets, [_g2_from_words(h) for h in hashes]


def hash_to_g2_outputs(results, offsets):
    """``output_offset.add(neg_offset)`` (hash_to_g2.rs:204-208): the hash outputs from the native results
    ``cofactor * point + offset`` of a G2 proof (``Proof.results()``: x.c0, x.c1, y.c0, y.c1 as 16 limbs of 16 bits each
    per instance)."""
    res = np.asarray(results).reshape(-1, 64)
    return [g2_add(_g2_from_limbs16(r), g2_neg(off)) for r, off in zip(res, offsets)]


# ---- g1_msm (src/utils/g1_msm.rs:22-36) ----------------------------------------------------------------------------
def g1_neg(P):
    return None if P is None else (P[0], -P[1] % BN254_P)


def g1_add(P, Q):
    """Affine addition on G1; None is the point at infinity."""
    if P is None:
        return Q
    if Q is None:
        return P
    if P[0] == Q[0]:
        if (P[1] + Q[1]) % BN254_P == 0:
            return None
        lam = 3 * P[0] * P[0] * pow(2 * P[1], -1, BN254_P) % BN254_P
    else:
        lam = (Q[1] - P[1]) * pow(Q[0] - P[0], -1, BN254_P) % BN254_P
    x = (lam * lam - P[0] - Q[0]) % BN254_P
    return (x, (lam * (P[0] - x) - P[1]) % BN254_P)


def g1_mul(k: int, P):
    acc = None
    for bit in bin(k)[2:]:
        acc = g1_add(acc, acc)
        if bit == "1":
            acc = g1_add(acc, P)
    return acc


def g1_msm_inputs(ctx, scalars, points, seed: int):
    """The G1ScalarMulInput batch of ``g1_msm(scalars, points)``, built on the device: one chain that starts at a random
    subgroup point acc_0 (drawn from ``SplitMix64(seed)`` as ``hash_to_g2_inputs`` draws its offsets) and adds
    s_i * x_i term by term, so that row i is (s_i, x_i, acc_i) (``Context.scalar_mul_chains``).
    scalars: ints < 2^256; points: affine G1 points (x, y). Returns (inputs[n, 20], timestamps[n], msm) with
    msm = acc_n - acc_0 as an affine point, None for the point at infinity."""
    rng = I.SplitMix64(seed)
    k = 0
    while k % BN254_R == 0:
        k = rng.bits256() & ((1 << 254) - 1)
    off = I.scalar_mul_gen(I.KIND_G1, k)
    terms = np.array([I._words(int(s)) + I._words(p[0]) + I._words(p[1]) for s, p in zip(scalars, points)],
                     dtype=np.uint64).reshape(-1, 12)
    starts = np.array([0, terms.shape[0]], dtype=np.uint64)
    inputs, sums = ctx.scalar_mul_chains(I.KIND_G1, terms, starts, np.array(I._words(off[0]) + I._words(off[1]),
                                                                           dtype=np.uint64))
    total = (_int256(sums[0, :4]), _int256(sums[0, 4:]))
    return inputs, np.arange(inputs.shape[0], dtype=np.uint64), g1_add(total, g1_neg(off))
