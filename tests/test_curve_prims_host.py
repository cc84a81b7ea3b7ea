"""ec.cuh's group law, ladders, scalar splits and window recoding, built for the host from tests/device_shim/prim_ops.h,
against the big-integer oracle.  The case builders here are shared with test_gpu_curve_prims.py, which runs them on the
device and requires its outputs to equal this build's bit for bit.

Random points almost never reach the branches that make a group law correct, so every case here is built to reach
one: an accumulator at infinity (zz stored as 0, and as p for the redundant form), P + P and P + (-P) with the
accumulator in the representation (l^2 x, l^3 y, l^2, l^3) for a random l (equality must be detected across
representations, not by bit pattern), adding the identity, redundant-form accumulators lifted into [p, 2p) under every
component mask, and chains of a few hundred additions that pass through infinity and continue.  The ladders and splits
run on the scalars where window code goes wrong: 0, 1, 2, r - 1, (r - 1) / 2, the endomorphism eigenvalues, the GLV
lattice basis and the rounding boundaries of glv_split, every window digit at -2^(c-1) or at 2^(c-1) - 1, and 2^k - 1,
2^k at the window and limb boundaries."""
import random

import numpy as np
import pytest

import prim_shim as ps
from prim_shim import R, Mont, ints, words

R_MOD = 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001
# eigenvalue of phi(x, y) = (beta x, y) on G1 (ec.cuh glv_lambda_mont) and of psi on G2 (6 x^2, ec.cuh psi_split)
LAMBDA = 0x30644E72E131A029048B6E193FD84104CC37A73FEC2BC5E9B8CA0B2D36636F23
LAMBDA_PSI = 0x6F4D8248EEB859FBF83E9682E87CFD46
# glv_split's reduced lattice basis (a1, b1), (a2, b2) of {(x, y): x + y lambda = 0 mod r}
A1, B1 = 0x6F4D8248EEB859FC8211BBEB7D4F1128, -0x89D3256894D213E3
A2, B2 = 0x89D3256894D213E3, 0x6F4D8248EEB859FD0BE4E1541221250B
# records: acc (XYZZ) | P (affine) | Q (XYZZ) | s | aux, in words of one coordinate (E = 8 for G1, 16 for G2)
(MADD, ADD, ADD_COLD, DBL, DBL_AFFINE, FROM_AFFINE, TO_AFFINE, NEG, MADD_LAZY, ON_CURVE, MUL254, MUL128, JOINT, GLV64,
 GATHER) = range(15)
GLV_SPLIT, PSI_SPLIT, GLV64_COEFF, RECODE = range(4)


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return ps.host(tmp_path_factory)


# ---------------------------------------------------------------- the two groups
class Group:
    """One of G1 / G2: the oracle's curve, the shim family, and the word layout of prim_ops.h's curve_op."""

    def __init__(self, po, g):
        self.po, self.g = po, g
        self.curve = po.G1 if g == 1 else po.G2
        self.F = self.curve.F
        self.fam = ps.FAM_G1_CURVE if g == 1 else ps.FAM_G2_CURVE
        self.E = 8 if g == 1 else 16
        self.in_words, self.out_words = 10 * self.E + 16, 8 * self.E + 1
        self.q = po.Q_MOD
        self.mq = Mont(self.q)
        self.gen = po.G1_GEN if g == 1 else po.G2_GEN

    # field elements <-> Montgomery words
    def comps(self, v):
        return [v] if self.g == 1 else list(v)

    def fwords(self, vals):
        return [self.mq.to(c) for v in vals for c in self.comps(v)]

    def fvals(self, row, k):
        """k field elements from Montgomery words (the raw residues, not reduced: a redundant form stays visible)"""
        raw = ints(np.asarray(row[:k * self.E], np.uint32).reshape(-1, 8))
        v = [self.mq.frm(x) for x in raw]
        return v if self.g == 1 else [(v[2 * i], v[2 * i + 1]) for i in range(k)]

    def raw(self, row, k):
        return ints(np.asarray(row[:k * self.E], np.uint32).reshape(-1, 8))

    def rand_f(self, rng):
        return rng.randrange(1, self.q) if self.g == 1 else (rng.randrange(self.q), rng.randrange(1, self.q))

    def point(self, k):
        return self.curve.mul(self.gen, k % R_MOD)

    # XYZZ: (l^2 x, l^3 y, l^2, l^3); infinity: zz = zzz = 0 with any x, y
    def xyzz(self, P, lam=None, inf_xy=None):
        F = self.F
        if P is None:
            x, y = inf_xy if inf_xy else (F.one, F.one)
            return [x, y, F.zero, F.zero]
        lam = lam if lam is not None else F.one
        l2 = F.sqr(lam)
        l3 = F.mul(l2, lam)
        return [F.mul(l2, P[0]), F.mul(l3, P[1]), l2, l3]

    def affine(self, P):
        return [self.F.zero, self.F.zero] if P is None else [P[0], P[1]]

    def record(self, acc=None, P=None, Q=None, s=0, aux=(), acc_words=None):
        """acc / Q: XYZZ coordinate lists (field values); P: affine point or None; s: a 256-bit integer"""
        F = self.F
        acc = acc if acc is not None else self.xyzz(None)
        Q = Q if Q is not None else self.xyzz(None)
        w = (acc_words if acc_words is not None else self.fwords(acc)) + self.fwords(self.affine(P)) + self.fwords(Q)
        rec = np.zeros(self.in_words, np.uint32)
        rec[:10 * self.E] = words(w).reshape(-1)
        rec[10 * self.E:10 * self.E + 8] = words([s]).reshape(-1)
        for i, a in enumerate(aux):
            rec[10 * self.E + 8 + i] = a & 0xffffffff
        return rec

    def decode(self, row, name):
        """an XYZZ output -> affine point or None, after checking that it is a valid XYZZ (zz^3 = zzz^2) and that
        infinity is stored with zz = zzz = 0 bit for bit"""
        F = self.F
        x, y, zz, zzz = self.fvals(row, 4)
        if F.is_zero(zz):
            assert not any(self.raw(row, 4)[2 * len(self.comps(zz)):]), (name, "infinity with non-zero zz / zzz bits")
            return None
        assert F.mul(F.sqr(zz), zz) == F.sqr(zzz), (name, "zz^3 != zzz^2")
        return (F.mul(x, F.inv(zz)), F.mul(y, F.inv(zzz)))

    def decode_affine(self, row):
        x, y = self.fvals(row, 2)
        return None if self.F.is_zero(x) and self.F.is_zero(y) else (x, y)


def groups(po):
    return [Group(po, 1), Group(po, 2)]


# ---------------------------------------------------------------- special scalars
def digit_extremes(c, top=254):
    """integers below 2^top whose signed c-bit digits (as recode_offset / the 4-bit ladders produce them) are all
    -2^(c-1), or all 2^(c-1) - 1, below the top window"""
    W = (top + c - 1) // c
    lo = sum(-(1 << (c - 1)) << (c * w) for w in range(W - 1))
    hi = sum(((1 << (c - 1)) - 1) << (c * w) for w in range(W - 1))
    out = []
    for base in (lo, hi):
        for t in range(1, 1 << 3):
            v = base + (t << (c * (W - 1)))
            if 0 <= v < R_MOD:
                out.append(v)
                break
    return out


def glv_hard_scalars():
    """the worst cases of glv_split's rounding: multiples of the lattice basis and the points next to them, and the
    scalars where floor(k * b2 / r), floor(k * |b1| / r) step (the estimate c_i is then off by the most)"""
    out = set()
    for m in (1, 2, 3, 7, 1 << 20, (1 << 64) - 1):
        for v in (A1, A2, B2, -B1, A1 + A2, B2 - B1):
            for d in (-1, 0, 1):
                out.add((m * v + d) % R_MOD)
    for bnd in (B2, -B1):
        for j in (1, 2, 3, bnd // 2, bnd - 1):
            k = -(-j * R_MOD // bnd)                       # the first k with floor(k bnd / r) = j
            for d in (-2, -1, 0, 1):
                out.add((k + d) % R_MOD)
    return sorted(out)


def special_scalars():
    """scalars in [0, r)"""
    r = R_MOD
    s = {0, 1, 2, 3, r - 1, r - 2, (r - 1) // 2, (r + 1) // 2, LAMBDA, r - LAMBDA, LAMBDA_PSI, r - LAMBDA_PSI,
         LAMBDA * LAMBDA % r}
    for k in (4, 8, 16, 31, 32, 63, 64, 96, 127, 128, 129, 160, 191, 192, 224, 252, 253):
        s |= {(1 << k) - 1, 1 << k, (1 << k) + 1}
    for c in (4, 8, 13, 16, 17):
        s |= set(digit_extremes(c))
    s |= {int("78" * 31 + "7", 16), int("87" * 31 + "8", 16)}
    return sorted(v % r for v in s | set(glv_hard_scalars()))


def mul128_scalars():
    """128-bit magnitudes for the u128 ladders"""
    s = {0, 1, 2, 8, 15, 16, 17, (1 << 128) - 1, 1 << 127, (1 << 127) - 1, (1 << 64) - 1, 1 << 64,
         int("8" * 32, 16), int("7" * 32, 16), int("78" * 16, 16), int("87" * 16, 16), LAMBDA_PSI - 1}
    for c in (4, 8, 16):
        s |= {v for v in digit_extremes(c, 128) if v < 1 << 128}
    return sorted(s)


# ---------------------------------------------------------------- group-law cases
def law_cases(grp, seed):
    """(name, code, records, check(out rows)) for the group law of one group"""
    po, F, C = grp.po, grp.F, grp.curve
    rng = random.Random(seed)
    pts = [grp.point(rng.randrange(1, R_MOD)) for _ in range(4)]
    lam = lambda: grp.rand_f(rng)
    cases = []

    def case(name, code, recs, want, exact=None):
        """want[i]: the expected affine point (None: infinity); exact[i]: words the output must equal bit for bit"""
        rec = np.stack(recs)

        def check(out):
            for i, row in enumerate(out):
                if exact is not None and exact[i] is not None:
                    assert np.array_equal(row[:4 * grp.E], exact[i]), (name, i, "changed")
                assert grp.decode(row, (name, i)) == want[i], (name, i)
        cases.append((name, code, rec, check))

    A, B = pts[0], pts[1]
    # madd and its lazy form on the same records (madd_lazy is G1's, checked below)
    recs, want = [], []
    for P in pts:
        for X in pts:
            if X is not P:
                recs.append(grp.record(acc=grp.xyzz(X, lam()), P=P)); want.append(C.add(X, P))
        recs.append(grp.record(acc=grp.xyzz(P, lam()), P=P)); want.append(C.add(P, P))              # P + P
        recs.append(grp.record(acc=grp.xyzz(C.neg(P), lam()), P=P)); want.append(None)               # P + (-P)
        recs.append(grp.record(acc=grp.xyzz(None), P=P)); want.append(P)                             # inf + P
        recs.append(grp.record(acc=grp.xyzz(None, inf_xy=(lam(), lam())), P=P)); want.append(P)      # other inf x, y
    madd_recs, madd_want = list(recs), list(want)
    ident = [grp.record(acc=grp.xyzz(X, lam()), P=None) for X in pts] + [grp.record(P=None)]
    ident_want = pts + [None]
    case("madd", MADD, recs + ident, want + ident_want,
         exact=[None] * len(recs) + [r[:4 * grp.E] for r in ident])                                 # X + O = X, unchanged
    # add / add_cold: the second operand in XYZZ form with its own l
    recs, want = [], []
    for X in pts:
        for Y in pts:
            recs.append(grp.record(acc=grp.xyzz(X, lam()), Q=grp.xyzz(Y, lam()))); want.append(C.add(X, Y))
        recs.append(grp.record(acc=grp.xyzz(X, lam()), Q=grp.xyzz(C.neg(X), lam()))); want.append(None)
        recs.append(grp.record(acc=grp.xyzz(None), Q=grp.xyzz(X, lam()))); want.append(X)
        recs.append(grp.record(acc=grp.xyzz(X, lam()), Q=grp.xyzz(None, inf_xy=(lam(), lam())))); want.append(X)
    recs.append(grp.record()); want.append(None)
    case("add", ADD, recs, want)
    case("add_cold", ADD_COLD, recs, want)
    # dbl: infinity stays, y = 0 gives infinity (no point of order 2 is on either curve: a crafted state)
    recs = [grp.record(acc=grp.xyzz(X, lam())) for X in pts] + [grp.record()]
    want = [C.add(X, X) for X in pts] + [None]
    recs.append(grp.record(acc=[lam(), F.zero, lam(), lam()])); want.append(None)
    case("dbl", DBL, recs, want)
    recs = [grp.record(P=X) for X in pts] + [grp.record(P=(lam(), F.zero))]
    case("dbl_affine", DBL_AFFINE, recs, [C.add(X, X) for X in pts] + [None])
    one = grp.fwords([F.one, F.one])
    case("from_affine", FROM_AFFINE, [grp.record(P=X) for X in pts] + [grp.record(P=None)], pts + [None],
         exact=[np.array(words(grp.fwords([X[0], X[1]]) + one).reshape(-1)) for X in pts] + [None])
    recs = [grp.record(acc=grp.xyzz(X, lam())) for X in pts] + [grp.record(acc=grp.xyzz(None, inf_xy=(lam(), lam())))]

    def check_affine(out, want=pts + [None]):
        for i, row in enumerate(out):
            assert grp.decode_affine(row) == want[i], ("to_affine", i)
            if want[i] is None:
                assert not row[:2 * grp.E].any()
    cases.append(("to_affine", TO_AFFINE, np.stack(recs), check_affine))
    case("neg", NEG, [grp.record(acc=grp.xyzz(X, lam())) for X in pts], [C.neg(X) for X in pts])
    # on_curve: points, identity, and off-curve (x, y + 1)
    recs = [grp.record(P=X) for X in pts] + [grp.record(P=None)]
    bad = [(X[0], F.add(X[1], F.one)) for X in pts]
    recs += [grp.record(P=X) for X in bad]
    flags = [1] * (len(pts) + 1) + [0] * len(bad)

    def check_on_curve(out):
        assert out[:, 8 * grp.E].tolist() == flags
    cases.append(("on_curve", ON_CURVE, np.stack(recs), check_on_curve))
    if grp.g == 1:
        # madd_lazy on the madd records with the accumulator lifted into [p, 2p) under every component mask; an
        # accumulator at infinity also with zz (and zzz) stored as p
        recs, want = [], []
        for mask in range(16):
            for rec_m, w in zip(madd_recs, madd_want):
                r = rec_m.copy()
                acc = ints(r[:32].reshape(4, 8))
                acc = [v + grp.q if (mask >> j) & 1 else v for j, v in enumerate(acc)]
                r[:32] = words(acc).reshape(-1)
                recs.append(r); want.append(w)
        for zzz in (0, grp.q):
            for P in pts:
                acc_w = [grp.mq.to(lam()), grp.mq.to(lam()), grp.q, zzz]
                recs.append(grp.record(acc_words=acc_w, P=P)); want.append(P)

        def check_lazy(out, recs=recs, want=want):
            for i, row in enumerate(out):
                assert grp.decode(row, ("madd_lazy", i)) == want[i], ("madd_lazy", i)
                lazy = ints(row[32:64].reshape(4, 8))
                assert max(lazy) < 2 * grp.q, ("madd_lazy", i, "left [0, 2p)")
                assert [v % grp.q for v in lazy] == ints(row[:32].reshape(4, 8)), ("madd_lazy", i)
        cases.append(("madd_lazy", MADD_LAZY, np.stack(recs), check_lazy))
    return cases


def gather_cases(grp, seed):
    """gather_point on a 2-row table of two units read from the record itself: every row at both signs.  The host build
    runs prim_ops.h's restatement of gather_point (the library's is device code), so these cases test the library only
    in test_gpu_curve_prims.py."""
    rng = random.Random(seed)
    pts = [grp.point(rng.randrange(1, R_MOD)) for _ in range(3)] + [None]
    tbl = pts + [grp.point(5)]                           # five affine points: acc (two) | P | Q (two)
    acc_w = grp.fwords(grp.affine(tbl[0]) + grp.affine(tbl[1]))
    Q = grp.affine(tbl[3]) + grp.affine(tbl[4])
    recs, want = [], []
    for unit in (0, 1):
        for d in (1, 2, -1, -2):
            recs.append(grp.record(acc_words=acc_w, P=tbl[2], Q=Q, aux=(0, 2, unit, d)))
            p = tbl[2 * unit + abs(d) - 1]
            want.append(grp.curve.neg(p) if d < 0 else p)

    def check(out):
        for i, row in enumerate(out):
            got = grp.decode_affine(row)
            assert got == want[i], ("gather_point", i)
            if want[i] is not None:                      # the y of the table, or its negation, exactly
                assert np.array_equal(row[:2 * grp.E], words(grp.fwords(grp.affine(want[i]))).reshape(-1)), i
    return [("gather_point", GATHER, np.stack(recs), check)]


def ladder_cases(grp, seed):
    """scalar_mul_window<F, 8> / <F, 4>, joint_mul_u128<F, 2> (phi on G1, psi on G2, every sign mask) and, on G1,
    scalar_mul_glv64 against [k] P"""
    rng = random.Random(seed)
    C = grp.curve
    P = grp.point(rng.randrange(1, R_MOD))
    lam = lambda: grp.rand_f(rng)
    cases = []

    def case(name, code, ks, want_k, aux=lambda k: ()):
        recs = [grp.record(acc=grp.xyzz(P, lam()), s=k, aux=aux(k)) for k in ks]

        def check(out):
            for i, row in enumerate(out):
                assert grp.decode(row, (name, hex(ks[i]))) == C.mul(P, want_k(ks[i]) % R_MOD), (name, hex(ks[i]))
        cases.append((name, code, np.stack(recs), check))

    s254 = special_scalars() + [(1 << 254) - 1, (1 << 255), (1 << 256) - 1, R_MOD, 2 * R_MOD - 1]
    case("scalar_mul_window<8>", MUL254, s254, lambda k: k)
    s128 = mul128_scalars()
    case("scalar_mul_window<4>", MUL128, s128, lambda k: k)
    eig = LAMBDA if grp.g == 1 else LAMBDA_PSI
    pairs = [(a, b) for a in (0, 1, (1 << 128) - 1, int("78" * 16, 16)) for b in (0, 1, (1 << 127) - 1, int("87" * 16, 16))]
    pairs += [(rng.getrandbits(128), rng.getrandbits(128)) for _ in range(6)]
    ks, negs = [], []
    for i, (a, b) in enumerate(pairs):
        for neg in range(4):
            ks.append(a | b << 128)
            negs.append(neg)
    joint = dict(zip(range(len(ks)), negs))
    recs = [grp.record(acc=grp.xyzz(P, lam()), s=k, aux=(joint[i],)) for i, k in enumerate(ks)]

    def check_joint(out):
        for i, row in enumerate(out):
            a, b, neg = ks[i] & ((1 << 128) - 1), ks[i] >> 128, joint[i]
            want = (-a if neg & 1 else a) + (-b if neg & 2 else b) * eig
            assert grp.decode(row, ("joint_mul", i)) == C.mul(P, want % R_MOD), ("joint_mul_u128", i, hex(a), hex(b), neg)
    cases.append(("joint_mul_u128", JOINT, np.stack(recs), check_joint))
    if grp.g == 1:
        k64 = [(a, b) for a in (0, 1, 8, (1 << 64) - 1, int("78" * 8, 16), 1 << 63) for b in (0, 1, (1 << 64) - 1, int("87" * 8, 16))]
        case("scalar_mul_glv64", GLV64, [a | b << 64 for a, b in k64], lambda k: (k & ((1 << 64) - 1)) + (k >> 64) * LAMBDA)
    return cases


def chain_check(grp, run, seed, steps=300, chains=6, lazy=False):
    """`chains` accumulators, each fed `steps` madds (or madd_lazy, the redundant form carried from step to step) whose
    partial sums return to infinity and continue: blocks of random points followed by their negations in reverse
    order, P, P, -P, O, -P (a doubling, then back) and P, -P, O.  The running sum is checked against the oracle after every step."""
    rng = random.Random(seed)
    C = grp.curve
    pool = [grp.point(rng.randrange(1, R_MOD)) for _ in range(8)]
    seqs = []
    for _ in range(chains):
        seq = []
        while len(seq) < steps:
            fw = [rng.choice(pool) for _ in range(rng.randrange(1, 12))]
            seq += fw + [C.neg(p) for p in reversed(fw)]
            p = rng.choice(pool)
            seq += [p, p, C.neg(p), None, C.neg(p)] if rng.random() < 0.5 else [p, C.neg(p), None]
        seqs.append(seq[:steps])
    code = MADD_LAZY if lazy else MADD
    accw = [grp.fwords(grp.xyzz(None))] * chains
    want = [None] * chains
    infs = 0
    for t in range(steps):
        rec = np.stack([grp.record(acc_words=accw[j], P=seqs[j][t]) for j in range(chains)])
        out = run(grp.fam, code, rec)
        for j in range(chains):
            want[j] = C.add(want[j], seqs[j][t])
            infs += want[j] is None
            assert grp.decode(out[j], ("chain", t)) == want[j], ("chain", j, t)
            accw[j] = ints(out[j, 4 * grp.E:8 * grp.E].reshape(-1, 8)) if lazy else ints(out[j, :4 * grp.E].reshape(-1, 8))
    assert infs > chains * steps // 20                   # the chains did pass through infinity


def all_curve_cases(po, seed):
    out = []
    for grp in groups(po):
        for name, code, rec, check in law_cases(grp, seed) + gather_cases(grp, seed) + ladder_cases(grp, seed):
            out.append((f"G{grp.g} {name}", grp.fam, code, rec, check))
    return out


# ---------------------------------------------------------------- splits and recoding
def scalar_rec(vals, c=0, W=0):
    rec = np.zeros((len(vals), 16), np.uint32)
    rec[:, :8] = words(vals)
    rec[:, 8], rec[:, 9] = c, W
    return rec


def signed(v, neg):
    return -v if neg else v


def check_glv_split(ks, out):
    for k, row in zip(ks, out):
        k1, k2 = ints(row[0:4][None])[0], ints(row[4:8][None])[0]
        assert row[10] == 1, ("glv_split not ok", hex(k))
        assert k1 < 1 << 128 and k2 < 1 << 128, hex(k)
        assert (signed(k1, row[8]) + signed(k2, row[9]) * LAMBDA - k) % R_MOD == 0, hex(k)


def check_psi_split(ks, out):
    for k, row in zip(ks, out):
        k0, k1 = ints(row[0:4][None])[0], ints(row[4:8][None])[0]
        assert k0 + k1 * LAMBDA_PSI == k and k0 < LAMBDA_PSI and k1 < 1 << 127, hex(k)


def check_recode(ks, c, W, out):
    lo, hi = -(1 << (c - 1)), 1 << (c - 1)
    for k, row in zip(ks, out):
        d = row[:W].view(np.int32).tolist()
        assert all(lo <= x < hi for x in d), (c, hex(k))
        assert sum(x << (c * w) for w, x in enumerate(d)) == k, (c, W, hex(k))
        assert not row[W:].any()


def recode_windows(c):
    """the window counts the library recodes with: 254-bit scalars (engine.cu window_count) and GLV halves below
    2^129 (msm_large.cu)"""
    return sorted({(255 + c - 1) // c, (130 + c - 1) // c})


def recode_scalars(c, W):
    """the special scalars (and the digit extremes of this c) that W windows can hold: s + K < 2^(c W).  With
    c W >= 255 that is every scalar below r, r - 1 included, also where the bound is tight (c W = 255 at c = 15 and
    17).  The GLV window counts (c W >= 130) must hold every magnitude below 2^(c W - 2), the bound that
    k_msm_digits_glv checks."""
    K = sum(1 << (c * w + c - 1) for w in range(W))
    cand = {k for k in special_scalars() + digit_extremes(c) + digit_extremes(c, c * W - 1) if k < R_MOD}
    if c * W < 255:
        cand.add((1 << (c * W - 2)) - 1)                 # the largest magnitude k_msm_digits_glv lets through
    ks = sorted({k for k in cand if k + K < 1 << (c * W)})
    if c * W >= 255:
        assert len(ks) == len(cand) and R_MOD - 1 in ks
    else:
        assert (1 << 128) + 1 in ks and (1 << (c * W - 2)) - 1 in ks
    return ks


def scalar_cases():
    """(name, code, records, check(out rows)) for the scalar family"""
    ks = special_scalars()
    cases = [("glv_split", GLV_SPLIT, scalar_rec(ks), lambda out: check_glv_split(ks, out)),
             ("psi_split", PSI_SPLIT, scalar_rec(ks), lambda out: check_psi_split(ks, out))]
    k64 = [a | b << 64 for a in (0, 1, (1 << 64) - 1, 1 << 63) for b in (0, 1, (1 << 64) - 1, 1 << 63)]

    def check_coeff(out):
        for k, got in zip(k64, ints(out[:, :8])):
            assert got == ((k & ((1 << 64) - 1)) + (k >> 64) * LAMBDA) % R_MOD, hex(k)
    cases.append(("glv64_coefficient", GLV64_COEFF, scalar_rec(k64), check_coeff))
    for c in range(8, 18):
        for W in recode_windows(c):
            kc = recode_scalars(c, W)
            cases.append((f"recode c={c} W={W}", RECODE, scalar_rec(kc, c, W),
                          lambda out, kc=kc, c=c, W=W: check_recode(kc, c, W, out)))
    return cases


# ---------------------------------------------------------------- tests
def test_reference_constants(po):
    """the eigenvalues and the lattice basis the checks rely on"""
    G = po.G1_GEN
    phi = po.G1.mul(G, LAMBDA)
    assert phi[1] == G[1] and phi[0] != G[0]                      # [lambda] G = (beta x, y)
    assert pow(LAMBDA, 3, R_MOD) == 1 and LAMBDA_PSI == 6 * po.BN_X ** 2
    assert (A1 + B1 * LAMBDA) % R_MOD == 0 and (A2 + B2 * LAMBDA) % R_MOD == 0
    assert A1 * B2 - A2 * B1 == R_MOD


def test_group_law_host(host, po):
    for name, fam, code, rec, check in all_curve_cases(po, 31):
        check(host.run(fam, code, rec))


@pytest.mark.parametrize("g, lazy", [(1, False), (1, True), (2, False)], ids=["g1", "g1_lazy", "g2"])
def test_madd_chains_through_infinity_host(host, po, g, lazy):
    chain_check(Group(po, g), host.run, 7 + g, steps=300 if g == 1 else 120, chains=6 if g == 1 else 3, lazy=lazy)


def test_splits_and_recoding_host(host):
    for name, code, rec, check in scalar_cases():
        check(host.run(ps.FAM_SCALAR, code, rec))


def test_glv_split_worst_case_magnitudes(host):
    """glv_split's magnitudes at the rounding boundaries stay below 2^128 (its ok flag); msm_large.cu's k_msm_digits_glv
    sizes its windows for magnitudes below 2^129, with the same constants"""
    ks = glv_hard_scalars()
    out = host.run(ps.FAM_SCALAR, GLV_SPLIT, scalar_rec(ks))
    check_glv_split(ks, out)
    assert max(ints(out[:, 0:4]) + ints(out[:, 4:8])).bit_length() <= 128
