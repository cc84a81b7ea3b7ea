"""The batched prover computes a term shared by the A and B1 sums once (variables whose A and B1 query points are the
same point, as in every MiMC-5 round of libzkp's circuits) and sizes its G1 gather grid from the unit count.  The
proof bytes do not change: proofs stay bit-exact against the oracles across the latency / batch boundaries, on both
builtin circuits and on caller-supplied R1CS with all, none or some of such pairs."""
import numpy as np
import pytest

from libzkp_b200 import engine

pytestmark = pytest.mark.gpu

WINDOW_BITS = 12


@pytest.fixture(scope="module")
def eq_pk_less(eq_keys):
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=WINDOW_BITS)
    pk.circuit_builtin(engine.EQUALITY, 110)
    yield pk
    pk.close()


@pytest.fixture(scope="module")
def mb_pk_less(mb_keys):
    pk = engine.ProvingKey(mb_keys.pk_bytes, window_bits=WINDOW_BITS)
    pk.circuit_builtin(engine.MEMBERSHIP, 64)
    yield pk
    pk.close()


def shared_pairs(opk):
    """Indices j >= 1 of the variables whose A and B1 query points are the same non-identity point."""
    return [j for j in range(1, len(opk.a_query)) if opk.a_query[j] is not None and opk.a_query[j] == opk.b_g1_query[j]]


def g1_units_expected(opk, W):
    nz = lambda pts: sum(p is not None for p in pts)
    a, b1 = nz(opk.a_query[1:]), nz(opk.b_g1_query[1:])
    delta = 3 if opk.delta_g1 is not None else 0          # r*delta into A, s*delta into B1, -rs*delta into L
    return W * (a + b1 - len(shared_pairs(opk)) + nz(opk.l_query) + nz(opk.h_query) + delta)


def test_equality_and_membership_keys_share_110_terms(eq_keys, mb_keys, eq_pk_less, mb_pk_less, po):
    for keys, pk in ((eq_keys, eq_pk_less), (mb_keys, mb_pk_less)):
        opk = po.pk_from_bytes(keys.pk_bytes)
        assert len(shared_pairs(opk)) == 110
        g1_units, _, _, _ = pk.work()
        assert g1_units == g1_units_expected(opk, pk.windows)
    # the equality key walked 1399 bases per window before the shared terms: 110 fewer now
    assert eq_pk_less.work()[0] == (1399 - 110) * eq_pk_less.windows


@pytest.mark.parametrize("n", [1, 64, 384, 385, 1024, 4096])     # 384 | 385: latency | batch form; 1024 on: large-batch grid
def test_equality_bit_exact_vs_c_oracle(eq_pk_less, eq_keys, co, po, frs, n):
    rng = po.SplitMix64(700 + n)
    a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
    r, s = frs(710 + n, n), frs(720 + n, n)
    proofs, _, status = eq_pk_less.prove_equality_batch(a, a, r, s)
    want, wstat = co.prove_batch(eq_keys.circuit, eq_keys.opk, a, a, None, None, r, s)
    assert not status.any() and not wstat.any()
    assert np.array_equal(proofs, want)


@pytest.mark.parametrize("n", [1, 64, 384, 385, 1024, 4096])
def test_membership_bit_exact_vs_c_oracle(mb_pk_less, mb_keys, co, po, frs, n):
    rng = po.SplitMix64(800 + n)
    sets = np.zeros((n, 64), np.uint64)
    lens = np.zeros(n, np.uint32)
    vals = np.zeros(n, np.uint64)
    for i in range(n):
        L = 1 + (i * 7) % 64
        lens[i] = L
        sets[i, :L] = [rng.next_u64() for _ in range(L)]
        vals[i] = sets[i, (i * 3) % L]
    r, s = frs(810 + n, n), frs(820 + n, n)
    proofs, _, status = mb_pk_less.prove_membership_batch(vals, sets, lens, r, s)
    want, wstat = co.prove_batch(mb_keys.circuit, mb_keys.opk, vals, None, sets, lens, r, s)
    assert not status.any() and not wstat.any()
    assert np.array_equal(proofs, want)


# ---- caller-supplied R1CS (lzkp_circuit_load) against the pure-Python oracle
def _square_chain(po):
    """t_{i+1} = t_i * t_i: every variable's A column equals its B column."""
    cs = po.ConstraintSystem()
    t = cs.new_witness(3)
    for _ in range(6):
        t = cs.mul(t, t)
    return cs


def _no_pairs(po):
    """No variable has equal A and B columns."""
    cs = po.ConstraintSystem()
    w = [cs.new_witness(v) for v in (2, 5, 7)]
    p = cs.mul(w[0], w[1])
    q = cs.mul(p, w[2])
    cs.enforce(w[0].lc + w[2].lc, w[1].lc + po.lc_const(1), cs.new_witness(0).lc)
    cs.mul(q, w[0])
    return cs


def _instance_in_c(po):
    """Public inputs in C (x * y = out, out public) beside one shared pair (u * u)."""
    cs = po.ConstraintSystem()
    out = cs.new_input(77)
    x, y, u = cs.new_witness(7), cs.new_witness(11), cs.new_witness(4)
    cs.enforce(x.lc, y.lc, out.lc)
    v = cs.mul(u, u)
    cs.enforce(v.lc, x.lc, cs.new_input(112).lc)
    return cs


def _csr(po, rows):
    rowptr, col, val = [0], [], []
    for row in rows:
        for v, c in row:
            col.append(c)
            val.append(np.frombuffer((v % po.R_MOD).to_bytes(32, "little"), np.uint8))
        rowptr.append(len(col))
    return (np.array(rowptr, np.uint32), np.array(col, np.uint32),
            np.stack(val) if val else np.zeros((0, 32), np.uint8))


@pytest.mark.parametrize("build, n_shared", [(_square_chain, 6), (_no_pairs, 0), (_instance_in_c, 1)])
def test_custom_r1cs_bit_exact_vs_python_oracle(po, build, n_shared):
    cs = build(po)
    A, B, C = cs.matrices()
    ni, nw = cs.num_instance(), cs.num_witness()
    opk = po.setup(cs, po.Trapdoor.from_seed(9))
    assert len(shared_pairs(opk)) == n_shared
    pk = engine.ProvingKey(po.pk_to_bytes(opk), window_bits=8)
    try:
        pk.circuit_load(len(A), ni, nw, [_csr(po, M) for M in (A, B, C)])
        assert pk.work()[0] == g1_units_expected(opk, pk.windows)
        rng = po.SplitMix64(90 + n_shared)
        n = 600                                        # above the latency and small-grid limits
        zs = [[1] + [rng.next_fr() for _ in range(ni + nw - 1)] for _ in range(n)]   # unsatisfied assignments
        z = np.stack([np.frombuffer(b"".join(v.to_bytes(32, "little") for v in zz), np.uint8) for zz in zs])
        rs = [(rng.next_fr(), rng.next_fr()) for _ in range(n)]
        r = np.stack([np.frombuffer(x.to_bytes(32, "little"), np.uint8) for x, _ in rs])
        s = np.stack([np.frombuffer(y.to_bytes(32, "little"), np.uint8) for _, y in rs])
        proofs, status = pk.prove_batch(z, r, s)
        assert not status.any()
        for i in (0, 1, 2, 300, n - 1):
            h = po.witness_map(A, B, C, ni, zs[i])
            want = po.proof_to_bytes(po.prove_with_assignment(opk, rs[i][0], rs[i][1], h, zs[i], ni))
            assert proofs[i].tobytes() == want, f"proof {i}"
        # the batch form (600 proofs) and the latency form (the same inputs in calls of 1 and 300) agree byte for byte
        p1, _ = pk.prove_batch(z[:1], r[:1], s[:1])
        p300, _ = pk.prove_batch(z[300:600], r[300:600], s[300:600])
        assert np.array_equal(p1[0], proofs[0]) and np.array_equal(p300, proofs[300:600])
    finally:
        pk.close()
