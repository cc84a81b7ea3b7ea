"""pairing.cuh's tower, pairing and G2 r-torsion test, built for the host from tests/device_shim/prim_ops.h, against the
big-integer oracle; and the device build of the same shim compiles for sm_100a.  The case builders here are shared with
test_gpu_pairing_prims.py, which runs them on the device and requires its outputs to equal this build's bit for bit.

The pairing value is pinned: pairing.cuh's e(P, Q) = final_exponentiation(multi_miller_loop(P, Q)) is the oracle's
final_exp(miller_loop(Q, P)) raised to 2x(6x^2 + 3x + 1) (x the BN parameter), the constant its hard-part addition chain
multiplies the exponent (p^12 - 1)/r by.  That constant is coprime to r, so it is still a non-degenerate bilinear
pairing."""
import os
import random
import sys

import numpy as np
import pytest

import prim_shim as ps
from conftest import ROOT
from prim_shim import Mont, fq12_flat, fq12_words, tower_to_flat

sys.path.insert(0, os.path.join(ROOT, "tools"))


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return ps.host(tmp_path_factory)


# ---------------------------------------------------------------- tower
_FROB = {}


def frob(po, f, k):
    """f^(p^k) in the oracle's Fq12 (w^(p^k) cached)"""
    if k not in _FROB:
        _FROB[k] = po.f12_pow([0, 1] + [0] * 10, po.Q_MOD ** k)
    acc, pw = [0] * 12, list(po._F12_ONE)
    for c in f:
        acc = [(x + c * y) % po.Q_MOD for x, y in zip(acc, pw)]
        pw = po.f12_mul(pw, _FROB[k])
    return acc


def cyclotomic(po, g):
    """g^((p^6 - 1)(p^2 + 1))"""
    t = po.f12_mul(frob(po, g, 6), po._f12_inv_deg(g))
    return po.f12_mul(frob(po, t, 2), t)


def tower_cases(po, seed, n=6):
    """(name, code, records, check(out rows)) for every tower_op of prim_ops.h"""
    q = po.Q_MOD
    rng = random.Random(seed)
    rf = lambda: [rng.randrange(q) for _ in range(12)]
    one = list(po._F12_ONE)
    dense = [rf() for _ in range(n)] + [one, [0, 1] + [0] * 10, [5] + [0] * 5 + [q - 1] + [0] * 5]
    others = [rf() for _ in range(len(dense))]

    def rec(xs, ys):
        return np.stack([np.concatenate([fq12_words(po, x), fq12_words(po, y)]) for x, y in zip(xs, ys)])

    def f6(f):      # keep the c0 half (v^0, v^1, v^2 of c0): tower slots 0..2
        t = ps.flat_to_tower(po, f)
        return tower_to_flat(po, t[:3] + [(0, 0)] * 3)

    six = [f6(f) for f in dense]
    six_b = [f6(f) for f in others]
    cases = []

    def case(name, code, xs, ys, want):
        def check(out):
            for i, row in enumerate(out):
                got = fq12_flat(po, row)
                assert got == want(i), (name, i)
        cases.append((name, code, rec(xs, ys), check))

    v = [0, 0, 1] + [0] * 9           # v = w^2
    case("f6_mul", 0, six, six_b, lambda i: po.f12_mul(six[i], six_b[i]))
    case("f6_mul_v", 2, six, six_b, lambda i: po.f12_mul(six[i], v))
    case("f12_mul", 3, dense, others, lambda i: po.f12_mul(dense[i], others[i]))
    case("f12_sqr", 4, dense, others, lambda i: po.f12_mul(dense[i], dense[i]))
    case("f12_conj", 6, dense, others, lambda i: frob(po, dense[i], 6))
    case("f12_frob2", 7, dense, others, lambda i: frob(po, dense[i], 2))
    case("f12_frob_odd<1>", 8, dense, others, lambda i: frob(po, dense[i], 1))
    case("f12_frob_odd<3>", 9, dense, others, lambda i: frob(po, dense[i], 3))
    # inverses: the product with the input is one
    case("f6_inv", 1, six, six_b, lambda i: po._f12_inv_deg(six[i]))
    case("f12_inv", 5, dense, others, lambda i: po._f12_inv_deg(dense[i]))
    # f * (c0 + c3 w + c4 v w): the line's coefficients are the first three Fq2 of the second operand
    lines = []
    for y in others:
        t = ps.flat_to_tower(po, y)
        lines.append(tower_to_flat(po, [t[0], (0, 0), (0, 0), t[1], t[2], (0, 0)]))
    case("f12_mul_by_034", 10, dense, others, lambda i: po.f12_mul(dense[i], lines[i]))
    # the cyclotomic subgroup: squaring and the power by -x
    cyc = [cyclotomic(po, g) for g in dense[:n]] + [one]
    case("f12_cyclo_sqr", 11, cyc, cyc, lambda i: po.f12_mul(cyc[i], cyc[i]))
    case("f12_exp_neg_x", 12, cyc, cyc, lambda i: po._f12_inv_deg(po.f12_pow(cyc[i], po.BN_X)))
    # the final exponentiation: the (p^12 - 1)/r power times pairing_power
    fe = dense[:3] + [one]
    c = ps.pairing_power(po) % po.R_MOD
    case("final_exponentiation", 13, fe, fe, lambda i: po.f12_pow(po.final_exp(fe[i]), c))
    return cases


def test_tower_ops_host(host, po):
    for name, code, rec, check in tower_cases(po, 1201):
        check(host.run(ps.FAM_TOWER, code, rec))


# ---------------------------------------------------------------- pairing
class PairingRef:
    """The device's pairing of [a] G1 and [b] G2 is E^(a b), E = the oracle's e(G1, G2) to pairing_power."""

    def __init__(self, po):
        self.po = po
        self.E = po.f12_pow(po.final_exp(po.miller_loop(po.G2_GEN, po.G1_GEN)), ps.pairing_power(po) % po.R_MOD)

    def value(self, k):
        return self.po.f12_pow(self.E, k % self.po.R_MOD)


def pairing_rec(po, pairs, skip=0):
    """multi_miller_loop record: N, skip mask, then (P, Q) per pair"""
    rec = np.zeros(200, np.uint32)
    rec[0], rec[1] = len(pairs), skip
    for k, (P, Q) in enumerate(pairs):
        rec[8 + 48 * k:24 + 48 * k] = ps.g1_words(po, P)
        rec[24 + 48 * k:56 + 48 * k] = ps.g2_words(po, Q)
    return rec


def pairing_cases(po, seed):
    """(name, records of FAM_PAIRING code 1, expected oracle Fq12 per record).  Points are [a] G1 and [b] G2 so that
    every expected value is a power of one oracle pairing: bilinearity e([a]P, [b]Q) = e(P, Q)^(a b) is what is
    checked.  A skipped pair (what the verifier does for a point at infinity) contributes 1."""
    rng = random.Random(seed)
    ref = PairingRef(po)
    recs, want, names = [], [], []
    for n in (1, 2, 3, 4):
        for skip in sorted({0, 1 << (n - 1), (1 << n) - 1 if n > 1 else 0, 0b0101 & ((1 << n) - 1)}):
            ks = [(rng.randrange(1, po.R_MOD), rng.randrange(1, po.R_MOD)) for _ in range(n)]
            pairs = [(po.G1.mul(po.G1_GEN, a), po.G2.mul(po.G2_GEN, b)) for a, b in ks]
            recs.append(pairing_rec(po, pairs, skip))
            want.append(ref.value(sum(a * b for k, (a, b) in enumerate(ks) if not (skip >> k) & 1)))
            names.append((n, skip))
    # e(P, -Q) e(P, Q) = 1 and e([a]P, Q) e(P, [-a]Q) = 1 in one loop
    a = rng.randrange(1, po.R_MOD)
    P, Q = po.G1.mul(po.G1_GEN, 7), po.G2.mul(po.G2_GEN, 11)
    recs.append(pairing_rec(po, [(P, Q), (P, po.G2.neg(Q))]))
    recs.append(pairing_rec(po, [(po.G1.mul(P, a), Q), (P, po.G2.mul(Q, po.R_MOD - a))]))
    want += [list(po._F12_ONE)] * 2
    names += ["cancel", "cancel_a"]
    # the generators themselves and one skipped pair alone (P or Q at infinity)
    recs.append(pairing_rec(po, [(po.G1_GEN, po.G2_GEN)]))
    recs.append(pairing_rec(po, [(po.G1_GEN, po.G2_GEN)], skip=1))
    want += [ref.E, list(po._F12_ONE)]
    names += ["generators", "skipped"]
    return names, np.stack(recs), want


def test_pairing_value_host(host, po):
    # the relation itself, at points that are not built from the generators by a known scalar on this side
    P, Q = po.G1.mul(po.G1_GEN, 12345), po.G2.mul(po.G2_GEN, 67890)
    got = fq12_flat(po, host.run(ps.FAM_PAIRING, 1, pairing_rec(po, [(P, Q)])[None])[0])
    oracle = po.final_exp(po.miller_loop(Q, P))
    assert got != oracle
    assert got == po.f12_pow(oracle, ps.pairing_power(po) % po.R_MOD)
    names, rec, want = pairing_cases(po, 77)
    out = host.run(ps.FAM_PAIRING, 1, rec)
    for name, row, w in zip(names, out, want):
        assert fq12_flat(po, row) == w, name


# ---------------------------------------------------------------- G2 r-torsion
def h2_primes(po):
    """the twist's cofactor h2 = 2p - r = 10069 * 5864401 * 1875725156269 * (a 179-bit prime)"""
    h2 = 2 * po.Q_MOD - po.R_MOD
    small = [10069, 5864401, 1875725156269]
    big = h2 // (small[0] * small[1] * small[2])
    assert small[0] * small[1] * small[2] * big == h2 and big.bit_length() == 178
    return small + [big]


def twist_points(po, start):
    """points of the twist y^2 = x^3 + 3/(9 + u) at x = (t, 1), t = start, start + 1, ... (tools/subgroup_test_proto.py)"""
    import subgroup_test_proto as sp
    t = start
    while True:
        xx = (t, 1)
        y = sp.f2sqrt(sp.f2add(sp.f2mul(sp.f2sqr(xx), xx), sp.B_TWIST))
        if y is not None:
            assert po.G2.on_curve((xx, y))
            yield (xx, y)
        t += 1


def g2_points(po, B, seed=5):
    """(name, point, in the r-torsion) for: T_l of order exactly l for each prime l | h2, B + T_l, a full-cofactor point
    [r] T, a raw twist point, and subgroup points (B, [k] B, -B).  Truth: [r] U == O."""
    r = po.R_MOD
    order = (2 * po.Q_MOD - r) * r                      # #E'
    pts = twist_points(po, 1000 + seed)
    out = []
    for ell in h2_primes(po):
        while True:
            T = po.G2.mul(next(pts), order // ell)
            if T is not None:
                break
        assert po.G2.mul(T, ell) is None
        out.append((f"T_{ell}", T))
        out.append((f"B+T_{ell}", po.G2.add(B, T)))
    raw = next(pts)
    out.append(("full_cofactor", po.G2.mul(raw, r)))
    out.append(("raw", raw))
    out += [("B", B), ("3B", po.G2.mul(B, 3)), ("-B", po.G2.neg(B)), ("[x]B", po.G2.mul(B, po.BN_X))]
    return [(name, U, po.G2.mul(U, r) is None) for name, U in out]


def test_g2_subgroup_host(host, po):
    B = po.G2.mul(po.G2_GEN, 0x1234567890abcdef)
    pts = g2_points(po, B)
    assert sum(ok for _, _, ok in pts) == 4 and len(pts) == 14
    rec = np.stack([np.concatenate([ps.g2_words(po, U), np.zeros(0, np.uint32)]) for _, U, _ in pts])
    out = host.run(ps.FAM_G2, 0, rec)
    for (name, U, truth), row in zip(pts, out):
        assert row[32] == truth, name
        assert ps.g2_from_words(po, row) == po.G2.mul(U, po.BN_X), name


def test_no_ladder_prefix_reaches_infinity_on_small_order_points(po):
    """The accumulator of the [x] ladder (coop::g2_in_subgroup, scalar_mul_window) is [k] T for the prefixes k of x,
    doubled or incremented.  For T of order l | h2 it reaches infinity only when l | k, and it equals +-T only when
    l | k -+ 1: neither happens for any prime factor of h2, so the special branches of the ladder are reached only from
    crafted states (test_gpu_pairing_prims.py drives them that way)."""
    x, k, ks = po.BN_X, 1, []
    for i in range(61, -1, -1):
        k *= 2
        ks.append(k)
        if (x >> i) & 1:
            ks.append(k)                 # the accumulator the addition sees
            k += 1
            ks.append(k)
    assert k == x
    for ell in h2_primes(po):
        assert all(v % ell not in (0, 1, ell - 1) for v in ks), ell


@pytest.mark.skipif(ps.nvcc() is None, reason="nvcc not available")
def test_device_shim_compiles(tmp_path):
    """The device build of the shim (prim_kernels.cu) compiles for sm_100a with the library's flags."""
    out = ps.compile_device(tmp_path)
    assert os.path.getsize(out) > 0
