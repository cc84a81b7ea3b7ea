"""pairing.cuh's tower and pairing, coop.cuh's warp-cooperative products and r-torsion ladder, and the G2 subgroup check
of the verifier, on the device:
- the serial tower / pairing code against the oracle (cases of test_prim_host.py), bit-identical to the host build;
- coop::f12_mul (dense and line operands, aliased results, the squaring path, the extra product of lanes >= 18),
  coop::f12_frob and coop::f12_conj against the serial code, bit for bit;
- the r-torsion test of B in its device forms (scalar_mul_window + g2_subgroup_from_xp per lane, and
  coop::g2_in_subgroup) against [r] T == O on points of every prime order dividing the twist's cofactor, the special
  branches of the cooperative ladder from crafted states, and VerifyingKey.verify_batch / verify_batch_device rejecting
  such a B in every form without touching the other proofs of the call;
- the cooperative verifier's self-test (LZKP_COOP_SELFTEST=1) at key load."""
import random

import numpy as np
import pytest

import prim_shim as ps
from prim_shim import Mont, fq12_flat, ints, words
from test_prim_host import g2_points, pairing_cases, tower_cases

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev(tmp_path_factory):
    return ps.device(tmp_path_factory)


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return ps.host(tmp_path_factory)


def both(dev, host, fam, code, rec):
    d, h = dev.run(fam, code, rec), host.run(fam, code, rec)
    bad = np.flatnonzero((d != h).any(axis=1))
    assert bad.size == 0, (fam, code, "device != host build", bad[:5].tolist())
    return d


def test_tower_ops(dev, host, po):
    for name, code, rec, check in tower_cases(po, 2402):
        check(both(dev, host, ps.FAM_TOWER, code, rec))


def test_pairing_value_and_multi_miller_loop(dev, host, po):
    """e(P, Q) on the device is the oracle's pairing to pairing_power (test_prim_host.py pins the relation); N = 1..4
    pairs with skip flags, bilinearity, and a skipped pair giving 1."""
    names, rec, want = pairing_cases(po, 88)
    out = both(dev, host, ps.FAM_PAIRING, 1, rec)
    for name, row, w in zip(names, out, want):
        assert fq12_flat(po, row) == w, name
    both(dev, host, ps.FAM_PAIRING, 0, rec)              # the Miller values alone, bit for bit


# ---------------------------------------------------------------- coop.cuh products
def rand_fq2s(rng, q, n):
    mq = Mont(q)
    return words([mq.to(rng.randrange(q)) for _ in range(2 * n)]).reshape(n, 16)


def test_coop_f12_mul(dev, host, po):
    q = po.Q_MOD
    rng = random.Random(31)
    n = 512
    a = rand_fq2s(rng, q, 6 * n).reshape(n, 96)
    b = rand_fq2s(rng, q, 6 * n).reshape(n, 96)
    a[0] = 0
    b[1] = 0
    a[2] = ps.fq12_words(po, list(po._F12_ONE))
    sa, sb = rand_fq2s(rng, q, n), rand_fq2s(rng, q, n)
    rec = np.concatenate([a, b, sa, sb], axis=1)
    tw = lambda x, y: np.concatenate([x, y], axis=1)
    prod = host.run(ps.FAM_FQ2, 0, tw(sa, sb))
    dense = host.run(ps.FAM_TOWER, 3, tw(a, b))          # serial f12_mul
    square = host.run(ps.FAM_TOWER, 3, tw(a, a))
    line = b.copy()
    line[:, 48:] = 0
    sparse = host.run(ps.FAM_TOWER, 10, tw(a, line))     # serial f12_mul_by_034 with (c0, c3, c4) = (l0, l1, l2)
    for mode, want in ((0, dense), (1, dense), (2, dense), (3, square)):
        out = dev.coop_f12_mul(False, mode, rec)
        assert np.array_equal(out[:, :96], want), ("dense", mode, np.flatnonzero((out[:, :96] != want).any(1))[:5])
        assert np.array_equal(out[:, 96:], prod), ("extra product", mode)
    lrec = rec.copy()
    lrec[:, 96 + 48:192] = 0
    for mode in (0, 1):
        out = dev.coop_f12_mul(True, mode, lrec)
        assert np.array_equal(out[:, :96], sparse), ("sparse", mode, np.flatnonzero((out[:, :96] != sparse).any(1))[:5])
        assert np.array_equal(out[:, 96:], prod), ("extra product, sparse", mode)


def test_coop_frobenius_and_conjugate(dev, host, po):
    rng = random.Random(32)
    n = 256
    a = rand_fq2s(rng, po.Q_MOD, 6 * n).reshape(n, 96)
    rec = np.concatenate([a, np.zeros_like(a)], axis=1)
    for k, code in ((0, 6), (1, 8), (2, 7), (3, 9)):
        want = host.run(ps.FAM_TOWER, code, rec)
        assert np.array_equal(dev.coop_f12_map(k, a), want), k


# ---------------------------------------------------------------- the r-torsion test of B
def test_g2_subgroup_device_forms(dev, host, po):
    B = po.G2.mul(po.G2_GEN, 0xfeedface12345)
    pts = g2_points(po, B, seed=9)
    rec = np.stack([ps.g2_words(po, U) for _, U, _ in pts])
    truth = np.array([ok for _, _, ok in pts])
    lanes = both(dev, host, ps.FAM_G2, 0, rec)          # scalar_mul_window<Fq2, 2> + g2_subgroup_from_xp (verify.cu)
    for (name, U, _), row in zip(pts, lanes):
        assert ps.g2_from_words(po, row) == po.G2.mul(U, po.BN_X), name
    assert np.array_equal(lanes[:, 32].astype(bool), truth), [p[0] for p, g in zip(pts, lanes[:, 32]) if bool(g) != p[2]]
    coop = dev.coop_subgroup(rec)
    assert np.array_equal(coop.astype(bool), truth), [p[0] for p, g in zip(pts, coop) if bool(g) != p[2]]


def _fq2_words(po, v):
    mq = Mont(po.Q_MOD)
    return words([mq.to(v[0]), mq.to(v[1])]).reshape(16)


def _xyzz(po, A, z):
    """XYZZ words of affine A scaled by z (X = x z^2, Y = y z^3, ZZ = z^2, ZZZ = z^3); None: infinity"""
    if A is None:
        one = (1, 0)
        return np.concatenate([_fq2_words(po, one), _fq2_words(po, one), np.zeros(32, np.uint32)])
    z2 = po.f2_mul(z, z)
    z3 = po.f2_mul(z2, z)
    return np.concatenate([_fq2_words(po, po.f2_mul(A[0], z2)), _fq2_words(po, po.f2_mul(A[1], z3)),
                           _fq2_words(po, z2), _fq2_words(po, z3)])


def _affine(po, row):
    mq = Mont(po.Q_MOD)
    v = [mq.frm(x) for x in ints(np.asarray(row[:64], np.uint32).reshape(8, 8))]
    X, Y, ZZ, ZZZ = (v[0], v[1]), (v[2], v[3]), (v[4], v[5]), (v[6], v[7])
    if ZZ == (0, 0):
        return None
    return (po.f2_mul(X, po.f2_inv(ZZ)), po.f2_mul(Y, po.f2_inv(ZZZ)))


def test_coop_ladder_special_branches(dev, po):
    """coop::ladder_step and coop::ladder_madd from crafted states: the accumulator at infinity, and accumulators whose
    double is +-B, where ladder_madd must decline (acc == +-B) and the serial formulas give 2B or O."""
    r = po.R_MOD
    rng = random.Random(33)
    B = po.G2.mul(po.G2_GEN, 0xabcdef987)
    inv2 = pow(2, -1, r)
    rz = lambda: (rng.randrange(1, po.Q_MOD), rng.randrange(po.Q_MOD))
    G = po.G2.mul(B, 12345)
    cases = [  # (mode, accumulator, add, expected)
        (0, None, 1, B), (0, None, 0, None),
        (0, G, 1, po.G2.add(po.G2.mul(G, 2), B)), (0, G, 0, po.G2.mul(G, 2)),
        (0, po.G2.mul(B, inv2), 1, po.G2.mul(B, 2)),                # 2 acc == B: the addition is a doubling
        (0, po.G2.mul(B, r - inv2), 1, None),                       # 2 acc == -B: the sum is infinity
        (1, G, 1, po.G2.add(G, B)),
    ]
    rec = np.zeros((len(cases) + 2, 97), np.uint32)
    for i, (mode, A, add, _) in enumerate(cases):
        rec[i, :64] = _xyzz(po, A, rz())
        rec[i, 64:96] = ps.g2_words(po, B)
        rec[i, 96] = add
    for i, A in enumerate((B, po.G2.neg(B))):                   # ladder_madd on acc == +-B: declines, state untouched
        rec[len(cases) + i, :64] = _xyzz(po, A, rz())
        rec[len(cases) + i, 64:96] = ps.g2_words(po, B)
    out0, out1 = dev.coop_ladder(0, rec), dev.coop_ladder(1, rec)
    for i, (mode, A, add, want) in enumerate(cases):
        out = out0 if mode == 0 else out1
        assert _affine(po, out[i]) == want, i
        assert out[i, 64] == 1, i
    for i in range(2):
        row = out1[len(cases) + i]
        assert row[64] == 0, i
        assert np.array_equal(row[:64], rec[len(cases) + i, :64]), i


# ---------------------------------------------------------------- the verifier
@pytest.fixture(scope="module")
def eq_proofs(eq_keys, po, frs):
    from libzkp_b200 import engine
    pk = engine.ProvingKey(eq_keys.pk_bytes, window_bits=10)
    try:
        pk.circuit_builtin(engine.EQUALITY, 110)
        n = 160
        rng = po.SplitMix64(5150)
        a = np.array([rng.next_u64() for _ in range(n)], np.uint64)
        proofs, cms, st = pk.prove_equality_batch(a, a, frs(5151, n), frs(5152, n))
    finally:
        pk.close()
    assert not st.any()
    return proofs, cms


@pytest.mark.parametrize("form", ["latency", "lanes", "combined"])
def test_off_subgroup_b_rejected(eq_keys, eq_proofs, po, form, monkeypatch):
    """B replaced by points outside the r-torsion (each prime order dividing h2, B + T_l for the proof's own B, a
    full-cofactor point, a raw twist point): exactly those proofs fail, through both the host-buffer and device calls."""
    from libzkp_b200 import engine
    from test_gpu_verify_device import _forms, dev_verify
    _forms(monkeypatch, form)
    proofs, cms = eq_proofs
    bad = proofs.copy()
    want = np.ones(len(proofs), bool)
    B0 = po.g2_from_bytes(bytes(proofs[0, 64:192]), False)
    off = [(name, U) for name, U, ok in g2_points(po, B0, seed=21) if not ok]
    assert len(off) == 10
    for j, (name, U) in enumerate(off):
        i = 13 * j + 5
        if name.startswith("B+"):                                  # the proof's own B shifted by T_l
            T = [V for n2, V in off if n2 == name[2:]][0]
            U = po.G2.add(po.g2_from_bytes(bytes(proofs[i, 64:192]), False), T)
        assert po.G2.on_curve(U) and po.G2.mul(U, po.R_MOD) is not None
        bad[i, 64:192] = np.frombuffer(po.g2_to_bytes(U), np.uint8)
        want[i] = False
    vk = engine.VerifyingKey(eq_keys.vk_bytes)
    try:
        host = vk.verify_batch(bad, cms)
        assert np.array_equal(host, want), (form, np.flatnonzero(host != want))
        dev = dev_verify(vk, bad, cms)
        assert np.array_equal(dev, want), (form, np.flatnonzero(dev != want))
    finally:
        vk.close()


def test_coop_selftest_at_key_load(eq_keys, po, trapdoor, frs, monkeypatch):
    """LZKP_COOP_SELFTEST=1 makes the key load compare the cooperative Miller loops (scaled and prepared lines), final
    exponentiation and subgroup ladder with the serial code on the key's points; a mismatch fails the load."""
    from libzkp_b200 import engine
    from test_gpu_verify_many_inputs import _squares_key_and_proofs
    monkeypatch.setenv("LZKP_COOP_SELFTEST", "1")
    vk_many, _, _ = _squares_key_and_proofs(po, trapdoor, frs, 300, 2, 3100)
    for vk_bytes in (eq_keys.vk_bytes, vk_many):
        vk = engine.VerifyingKey(vk_bytes)
        try:
            assert vk.info()[2], "latency form (and its self-test) not set up"
        finally:
            vk.close()
