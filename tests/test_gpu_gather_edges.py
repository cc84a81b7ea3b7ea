"""The batched table-gather MSMs (msm_batch.cu: k_msm_batch, then k_msm_reduce_tree or k_msm_reduce1 / k_msm_fold) on
proving keys whose query points are crafted rather than drawn from a setup, bit-exact against the Python oracle's
prove_with_assignment at sampled proofs.

The key's A, B1, L, H (G1) and B2 (G2) queries repeat one point X by variable j: X, X, -X, the identity, 2^c X, and an
unrelated Y.  The assignment z gives X and its repeat the same value v and -X the value v too, and 2^c X the value
(v - d_0(v)) / 2^c, whose digit in window w equals v's in window w + 1: those units gather the same table point.  Units
are laid out base-major and an item accumulates a running sum, so the equal and opposite terms meet mostly in the
reductions of the items' partial sums (P + P, P + (-P), sums at infinity), and only where an item's running sum happens
to equal the next gathered point inside k_msm_batch's madd.  v runs over random values, r - 1 and values whose every
window digit is -2^(c-1) (the table's last row) or 2^(c-1) - 1.  Each key runs at c = 16 (2-byte digits) and c = 17
(4-byte digits), with 384 / 385 proofs (the latency form and the batch form) and 513 (the large gather grid).

Two more keys put ONE point in every B2 entry, with z equal across the variables of a proof, so that the partial sums of
the items are equal and the fold and tree reductions double; or with z alternating v, r - v, so that they cancel."""
import random

import numpy as np
import pytest

from libzkp_b200 import engine
from test_curve_prims_host import R_MOD, digit_extremes
from test_gpu_msm_edges import recode
from test_gpu_prove_less import _csr

pytestmark = pytest.mark.gpu


def _circuit(po, n_wit=14):
    """a chain of products over n_wit witnesses (unsatisfied assignments are proved as they are)"""
    cs = po.ConstraintSystem()
    w = [cs.new_witness(i + 2) for i in range(n_wit)]
    for i in range(0, n_wit - 1, 2):
        cs.enforce(w[i].lc, w[i + 1].lc, w[(i + 2) % n_wit].lc)
    return cs


def _crafted(C, X, Y, c, j):
    """the point of class j % 6: X, X, -X, identity, 2^c X, Y"""
    return [X, X, C.neg(X), None, C.mul(X, 1 << c), Y][j % 6]


def _z_value(v, c, j):
    """the assignment of class j % 6 against the crafted point"""
    d0 = recode(v, c)[0]
    return [v, v, v, (v * 7 + 3) % R_MOD, (v - d0) >> c, digit_extremes(c)[(j // 6) % 2]][j % 6]


def _key(po, cs, seed, c, b2=None):
    opk = po.setup(cs, po.Trapdoor.from_seed(seed))
    rng = random.Random(seed)
    g1 = lambda: po.G1.mul(po.G1_GEN, rng.randrange(1, R_MOD))
    g2 = lambda: po.G2.mul(po.G2_GEN, rng.randrange(1, R_MOD))
    X, Y, X2, Y2 = g1(), g1(), g2(), g2()
    nv = len(opk.a_query)
    opk.a_query = [_crafted(po.G1, X, Y, c, j) for j in range(nv)]
    opk.b_g1_query = [_crafted(po.G1, X if j % 12 < 6 else Y, X, c, j) for j in range(nv)]   # shared A/B1 terms too
    opk.l_query = [_crafted(po.G1, Y, X, c, j + 1) for j in range(len(opk.l_query))]
    opk.h_query = [_crafted(po.G1, X, Y, c, j) for j in range(len(opk.h_query))]
    opk.b_g2_query = b2(nv, X2) if b2 else [_crafted(po.G2, X2, Y2, c, j) for j in range(nv)]
    return opk


def _prove_and_check(po, cs, opk, c, sizes, zfn, seed, sample=(0, 1, 2)):
    A, B, C = cs.matrices()
    ni, nw = cs.num_instance(), cs.num_witness()
    pk = engine.ProvingKey(po.pk_to_bytes(opk), window_bits=c)
    try:
        assert pk.window_bits == c
        pk.circuit_load(len(A), ni, nw, [_csr(po, M) for M in (A, B, C)])
        rng = random.Random(seed)
        for n in sizes:
            zs = [[1] + [zfn(i, j) for j in range(1, ni + nw)] for i in range(n)]
            z = np.stack([np.frombuffer(b"".join(v.to_bytes(32, "little") for v in zz), np.uint8) for zz in zs])
            rs = [(rng.randrange(1, R_MOD), rng.randrange(1, R_MOD)) for _ in range(n)]
            r = np.stack([np.frombuffer(x.to_bytes(32, "little"), np.uint8) for x, _ in rs])
            s = np.stack([np.frombuffer(y.to_bytes(32, "little"), np.uint8) for _, y in rs])
            proofs, status = pk.prove_batch(z, r, s)
            assert not status.any()
            for i in sorted({*sample, n // 2, n - 1}):
                h = po.witness_map(A, B, C, ni, zs[i])
                want = po.proof_to_bytes(po.prove_with_assignment(opk, rs[i][0], rs[i][1], h, zs[i], ni))
                assert proofs[i].tobytes() == want, (c, n, i)
    finally:
        pk.close()


def _v(c, i):
    """the per-proof value: digit extremes, r - 1, small values and random ones"""
    fixed = digit_extremes(c) + [R_MOD - 1, 1, (1 << (c - 1)) - 1, 1 << (c - 1)]
    return fixed[i] if i < len(fixed) else random.Random(i).randrange(R_MOD)


@pytest.mark.parametrize("c", [16, 17])
def test_gather_crafted_key_bit_exact(po, c):
    cs = _circuit(po)
    opk = _key(po, cs, 70 + c, c)
    _prove_and_check(po, cs, opk, c, (384, 385, 513), lambda i, j: _z_value(_v(c, i), c, j), 80 + c,
                     sample=(0, 1, 2, 3, 5))


@pytest.mark.parametrize("alternate", [False, True], ids=["equal", "cancel"])
def test_gather_g2_equal_partial_sums(po, alternate):
    """every B2 point the same: equal z makes every item's partial sum equal (the reductions double); z alternating
    v, r - v makes them cancel"""
    c = 16
    cs = _circuit(po, 30)
    opk = _key(po, cs, 90, c, b2=lambda nv, X2: [X2] * nv)

    def zfn(i, j):
        v = _v(c, i)
        return (R_MOD - v) % R_MOD if alternate and j % 2 else v
    _prove_and_check(po, cs, opk, c, (100, 600), zfn, 95)
