"""CPU oracle for ark-serialize's compressed form (Compress::Yes) of BN254 points, proofs and keys.

TEST INFRASTRUCTURE ONLY, like zkp_oracle.py (whose uncompressed writer fixes the sign rule used here):
nothing under ``libzkp_b200/`` may import it.  Big-integer square roots in Fq and Fq2, compressed
encode / decode of G1 and G2, and the compressed Proof, VerifyingKey and ProvingKey encoders.
"""
from __future__ import annotations

from typing import Optional, Tuple

from .zkp_oracle import (F2_ONE, G1_B, G2_B, Q_MOD, ProvingKey, VerifyingKey, _f2_gt, _fq_bytes, _fq_from,
                         _vec, f2_add, f2_mul, f2_neg, f2_sqr)


# --------------------------------------------------------------------------
# ark-serialize compressed layout [UPSTREAM]: x only (G1 32 B, G2 x.c0 || x.c1 64 B), flags in the top
# two bits of the last byte: 0x40 infinity, 0x80 y is the larger of y and -y (the same order as the
# uncompressed writer's sign bit above), both set invalid.  Decoding takes a square root and checks no
# subgroup membership (deserialize_compressed_unchecked).
# --------------------------------------------------------------------------
def fq_sqrt(a: int) -> Optional[int]:
    """A square root in Fq (q = 3 mod 4: a^((q+1)/4)), None for a non-square."""
    a %= Q_MOD
    r = pow(a, (Q_MOD + 1) // 4, Q_MOD)
    return r if r * r % Q_MOD == a else None


def f2_pow(a, e: int):
    r = F2_ONE
    for bit in bin(e)[2:]:
        r = f2_sqr(r)
        if bit == '1':
            r = f2_mul(r, a)
    return r


def f2_sqrt(a) -> Optional[Tuple[int, int]]:
    """A square root in Fq2 by Adj and Rodriguez-Henriquez 2012, Algorithm 9 (q = 3 mod 4), None for a
    non-square.  (The device uses the norm method: a different algorithm, the same square.)"""
    minus_one = (Q_MOD - 1, 0)
    a1 = f2_pow(a, (Q_MOD - 3) // 4)
    alpha = f2_mul(f2_sqr(a1), a)
    a0 = f2_mul((alpha[0], (-alpha[1]) % Q_MOD), alpha)             # alpha^q * alpha (Frobenius = conjugation)
    if a0 == minus_one:
        return None
    x0 = f2_mul(a1, a)
    if alpha == minus_one:
        x = f2_mul((0, 1), x0)
    else:
        x = f2_mul(f2_pow(f2_add(F2_ONE, alpha), (Q_MOD - 1) // 2), x0)
    return x if f2_sqr(x) == (a[0] % Q_MOD, a[1] % Q_MOD) else None


def g1_to_bytes_compressed(P) -> bytes:
    if P is None:
        return _fq_bytes(0, 0x40)
    x, y = P
    return _fq_bytes(x, 0x80 if y > (Q_MOD - y) % Q_MOD else 0)


def g2_to_bytes_compressed(P) -> bytes:
    if P is None:
        return bytes(32) + _fq_bytes(0, 0x40)
    x, y = P
    return _fq_bytes(x[0]) + _fq_bytes(x[1], 0x80 if _f2_gt(y, f2_neg(y)) else 0)


def g1_from_bytes_compressed(b: bytes):
    x, fl = _fq_from(b[0:32], True)
    if fl == 0xC0:
        raise ValueError("both flags set")
    if fl & 0x40:
        return None
    y = fq_sqrt(x * x * x + G1_B)
    if y is None:
        raise ValueError("no G1 point with this x")
    if (y > (Q_MOD - y) % Q_MOD) != bool(fl & 0x80):
        y = (Q_MOD - y) % Q_MOD
    return (x, y)


def g2_from_bytes_compressed(b: bytes):
    x0, _ = _fq_from(b[0:32], False)
    x1, fl = _fq_from(b[32:64], True)
    if fl == 0xC0:
        raise ValueError("both flags set")
    if fl & 0x40:
        return None
    x = (x0, x1)
    y = f2_sqrt(f2_add(f2_mul(f2_sqr(x), x), G2_B))
    if y is None:
        raise ValueError("no twist point with this x")
    if _f2_gt(y, f2_neg(y)) != bool(fl & 0x80):
        y = f2_neg(y)
    return (x, y)


def proof_to_bytes_compressed(proof) -> bytes:
    """Proof<Bn254> compressed = A(32) || B(64) || C(32) = 128 B."""
    a, b, c = proof
    return g1_to_bytes_compressed(a) + g2_to_bytes_compressed(b) + g1_to_bytes_compressed(c)


def proof_from_bytes_compressed(b: bytes):
    if len(b) != 128:
        raise ValueError("bad compressed proof length")
    return (g1_from_bytes_compressed(b[0:32]), g2_from_bytes_compressed(b[32:96]),
            g1_from_bytes_compressed(b[96:128]))


def vk_to_bytes_compressed(vk: VerifyingKey) -> bytes:
    """232 + 32 (n_pub + 1) B."""
    return (g1_to_bytes_compressed(vk.alpha_g1) + g2_to_bytes_compressed(vk.beta_g2)
            + g2_to_bytes_compressed(vk.gamma_g2) + g2_to_bytes_compressed(vk.delta_g2)
            + _vec(vk.gamma_abc_g1, g1_to_bytes_compressed))


def pk_to_bytes_compressed(pk: ProvingKey) -> bytes:
    return (vk_to_bytes_compressed(pk.vk) + g1_to_bytes_compressed(pk.beta_g1)
            + g1_to_bytes_compressed(pk.delta_g1) + _vec(pk.a_query, g1_to_bytes_compressed)
            + _vec(pk.b_g1_query, g1_to_bytes_compressed) + _vec(pk.b_g2_query, g2_to_bytes_compressed)
            + _vec(pk.h_query, g1_to_bytes_compressed) + _vec(pk.l_query, g1_to_bytes_compressed))
