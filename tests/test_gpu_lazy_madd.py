"""The G1 gather kernel accumulates in the redundant form (madd_lazy, coordinates in [0, 2p)) and stores canonical
partial sums.  Its doubling and infinity branches test residues, not bit patterns: a circuit whose first two L-query
bases are the same point drives the accumulator through P + P (equal small scalars: one nonzero digit each) and
P + (-P) (scalars v and r - v: the last nonzero digit of the second base cancels the sum), and the proofs must stay
bit-exact against the Python oracle.  The builtin circuits' bit-exactness at every batch form is checked in
test_gpu_prove_less.py."""
import numpy as np
import pytest

from libzkp_b200 import engine
from test_gpu_prove_less import _csr

pytestmark = pytest.mark.gpu


def _twin_bases(po):
    """(w1 + w2) * w3 = w4 and w3 * w3 = w5: w1 and w2 have identical columns, so their L-query points are equal,
    and they are the first two bases of the L MSM."""
    cs = po.ConstraintSystem()
    w1, w2, w3 = cs.new_witness(1), cs.new_witness(1), cs.new_witness(2)
    cs.enforce(w1.lc + w2.lc, w3.lc, cs.new_witness(4).lc)
    cs.mul(w3, w3)
    return cs


def test_doubling_and_infinity_branches_bit_exact_vs_python_oracle(po):
    cs = _twin_bases(po)
    A, B, C = cs.matrices()
    ni, nw = cs.num_instance(), cs.num_witness()
    opk = po.setup(cs, po.Trapdoor.from_seed(11))
    assert opk.l_query[0] is not None and opk.l_query[0] == opk.l_query[1]
    pk = engine.ProvingKey(po.pk_to_bytes(opk), window_bits=8)
    try:
        pk.circuit_load(len(A), ni, nw, [_csr(po, M) for M in (A, B, C)])
        rng = po.SplitMix64(123)
        n = 600                                        # the batch form's large grid
        zs = []
        for i in range(n):
            v = 1 + rng.next_u64() % 127               # below 2^(c-1): one nonzero signed digit
            twin = (v, po.R_MOD - v, rng.next_fr())[i % 3]
            zs.append([1, v, twin] + [rng.next_fr() for _ in range(ni + nw - 3)])
        z = np.stack([np.frombuffer(b"".join(x.to_bytes(32, "little") for x in zz), np.uint8) for zz in zs])
        rs = [(rng.next_fr(), rng.next_fr()) for _ in range(n)]
        r = np.stack([np.frombuffer(x.to_bytes(32, "little"), np.uint8) for x, _ in rs])
        s = np.stack([np.frombuffer(y.to_bytes(32, "little"), np.uint8) for _, y in rs])
        proofs, status = pk.prove_batch(z, r, s)
        assert not status.any()
        for i in (0, 1, 2, 3, 4, 5, 298, 299, n - 1):
            h = po.witness_map(A, B, C, ni, zs[i])
            want = po.proof_to_bytes(po.prove_with_assignment(opk, rs[i][0], rs[i][1], h, zs[i], ni))
            assert proofs[i].tobytes() == want, f"proof {i}"
    finally:
        pk.close()
