"""Checker for proof rerandomization (ark-groth16's rerandomize_proof; BKSV20, ePrint 2020/811, Thm. 3), beside the
oracle in zkp_oracle.py, which it uses unchanged.  Plain double-and-add (Curve.mul), no endomorphism: a different
algorithm from the engine's GLV / psi-split ladders.  Also the psi endomorphism of G2 and its eigenvalue, so that the
identity the engine's G2 ladder rests on, psi(Q) = [6 x^2] Q on the r-torsion, is checked here by big integers."""
from . import zkp_oracle as po

LAMBDA_PSI = 6 * po.BN_X * po.BN_X          # 127 bits, below r
XI = (9, 1)


def _f2_pow(a, e: int):
    r = po.F2_ONE
    for bit in bin(e)[2:]:
        r = po.f2_sqr(r)
        if bit == "1":
            r = po.f2_mul(r, a)
    return r


_TW_X = _f2_pow(XI, (po.Q_MOD - 1) // 3)
_TW_Y = _f2_pow(XI, (po.Q_MOD - 1) // 2)


def _conj(a):
    return (a[0], (-a[1]) % po.Q_MOD)


def psi(Q):
    """untwist - Frobenius - twist on the sextic twist: (conj(x) xi^((q-1)/3), conj(y) xi^((q-1)/2))."""
    if Q is None:
        return None
    return (po.f2_mul(_conj(Q[0]), _TW_X), po.f2_mul(_conj(Q[1]), _TW_Y))


def rerandomize(delta_g2, proof, r1: int, r2: int):
    """(A, B, C) -> (r1^-1 A, r1 B + (r1 r2) delta, C + r2 A) for non-zero r1, r2 mod r."""
    a, b, c = proof
    r1, r2 = r1 % po.R_MOD, r2 % po.R_MOD
    if r1 == 0 or r2 == 0:
        raise ValueError("factors must be non-zero")
    a2 = po.G1.mul(a, po.inv_mod(r1, po.R_MOD))
    b2 = po.G2.add(po.G2.mul(b, r1), po.G2.mul(delta_g2, r1 * r2 % po.R_MOD))
    c2 = po.G1.add(c, po.G1.mul(a, r2))
    return a2, b2, c2


def rerandomize_bytes(delta_g2, proof_bytes: bytes, r1: int, r2: int) -> bytes:
    """What the engine writes for one row: the rerandomized proof, ark-serialize uncompressed, or 256 B of 0xFF when
    the proof does not deserialize (validating) or a factor is 0 or >= r."""
    if not (0 < r1 < po.R_MOD and 0 < r2 < po.R_MOD):
        return b"\xff" * 256
    # both flags on a y coordinate are illegal in ark-serialize; the oracle's reader takes them for infinity
    if any(proof_bytes[i] & 0xC0 == 0xC0 for i in (63, 191, 255)):
        return b"\xff" * 256
    try:
        proof = po.proof_from_bytes(proof_bytes, validate=True)
    except ValueError:
        return b"\xff" * 256
    return po.proof_to_bytes(rerandomize(delta_g2, proof, r1, r2))
