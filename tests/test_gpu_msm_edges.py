"""The Pippenger MSMs (msm_large.cu) in every form on crafted bases and scalars, against the C oracle (or a known
discrete logarithm): generic G1 with the GLV split, generic G1 without it (LZKP_MSM_NO_GLV=1, read when the bases are
loaded), resident G1, and generic and resident G2, at several window sizes c.

Random inputs almost never put equal or opposite points in one bucket, or a partial sum of a bucket at infinity.  These
cases do:
- bases [P, P] with scalars [1, 2]: adjacent buckets hold equal sums;
- bases [P, -P] with equal scalars: the result is infinity (and its 0x40 encoding);
- identity bases mixed in; all scalars zero;
- bases P and 2^c P (and -2^c P) with the second scalar (s - d_0) / 2^c, so that its digit in window w equals the
  first's in window w + 1: in the resident form (one bucket set holding 2^(c w) P_i for every window) the two land in
  one bucket as equal points, or as opposite ones, whose sum is then d_0 P;
- scalars whose every window digit is -2^(c-1) or 2^(c-1) - 1, and the GLV worst cases of test_curve_prims_host.py;
- in G2, long runs (half of the scalars 1, a quarter r - 1) that reach k_long_run."""
import random

import numpy as np
import pytest

from libzkp_b200 import engine
from test_curve_prims_host import LAMBDA, R_MOD, digit_extremes, glv_hard_scalars, special_scalars

pytestmark = pytest.mark.gpu

# (name, group, resident, glv, c)
FORMS = ([("g1_glv", 1, False, True, c) for c in (8, 13, 16)] + [("g1_no_glv", 1, False, False, c) for c in (13, 16)]
         + [("g1_resident", 1, True, False, c) for c in (8, 13, 16)]
         + [("g2_generic", 2, False, False, c) for c in (8, 13, 16)] + [("g2_resident", 2, True, False, c) for c in (8, 13, 16)])


def fr_bytes(vals):
    return np.frombuffer(b"".join(int(v % R_MOD).to_bytes(32, "little") for v in vals), np.uint8).reshape(len(vals), 32).copy()


def recode(s, c):
    """the signed c-bit digits of recode_offset (W = ceil(255 / c))"""
    W = (255 + c - 1) // c
    v = s + sum(1 << (c * w + c - 1) for w in range(W))
    return [((v >> (c * w)) & ((1 << c) - 1)) - (1 << (c - 1)) for w in range(W)]


class Form:
    def __init__(self, po, co, group, resident, glv, c, monkeypatch):
        self.po, self.co, self.group, self.resident, self.c = po, co, group, resident, c
        self.curve = po.G1 if group == 1 else po.G2
        self.gen = po.G1_GEN if group == 1 else po.G2_GEN
        self.to_bytes = po.g1_to_bytes if group == 1 else po.g2_to_bytes
        self.oracle = co.msm_g1 if group == 1 else co.msm_g2
        self.size = 64 if group == 1 else 128
        if glv:
            monkeypatch.delenv("LZKP_MSM_NO_GLV", raising=False)
        else:
            monkeypatch.setenv("LZKP_MSM_NO_GLV", "1")

    def bases(self, pts):
        return np.frombuffer(b"".join(self.to_bytes(p) for p in pts), np.uint8).reshape(len(pts), self.size).copy()

    def msm(self, pts, scalars):
        B = engine.MsmBases(self.group, self.bases(pts), window_bits=self.c, resident_windows=self.resident)
        try:
            return B.msm(fr_bytes(scalars))
        finally:
            B.close()

    def check(self, name, pts, scalars, want=None):
        got = self.msm(pts, scalars)
        ora = self.oracle(self.bases(pts), fr_bytes(scalars))
        assert got == ora, name
        if want is not None:
            assert got == self.to_bytes(want), name
        return got


def infinity_bytes(size):
    return bytes(size - 1) + b"\x40"


@pytest.mark.parametrize("name, group, resident, glv, c", FORMS, ids=[f"{f[0]}_c{f[4]}" for f in FORMS])
def test_msm_special_cases(po, co, monkeypatch, name, group, resident, glv, c):
    f = Form(po, co, group, resident, glv, c, monkeypatch)
    C = f.curve
    rng = random.Random(1000 * group + c)
    P, Q = f.curve.mul(f.gen, rng.randrange(1, R_MOD)), f.curve.mul(f.gen, rng.randrange(1, R_MOD))
    # equal sums in adjacent buckets, and P + (-P)
    f.check("[P, P] * [1, 2]", [P, P], [1, 2], C.mul(P, 3))
    for s in (1, 2, (1 << (c - 1)) - 1, 1 << (c - 1), R_MOD - 1, rng.randrange(R_MOD)):
        assert f.check(f"[P, -P] * {s}", [P, C.neg(P)], [s, s]) == infinity_bytes(f.size)
    assert f.check("[P, -P, P, -P, Q, -Q]", [P, C.neg(P), P, C.neg(P), Q, C.neg(Q)], [5, 5, 7, 7, 9, 9]) == infinity_bytes(f.size)
    # identity bases mixed in, and all scalars zero
    pts = [P, None, Q, None, C.neg(P), P, None]
    f.check("identities", pts, [rng.randrange(R_MOD) for _ in pts])
    f.check("identities, equal scalars", pts, [3] * len(pts), C.mul(C.add(P, Q), 3))
    assert f.check("all zero", [P, Q, P], [0, 0, 0]) == infinity_bytes(f.size)
    assert f.check("identity only", [None, None], [1, R_MOD - 1]) == infinity_bytes(f.size)
    # P and +-2^c P: window w of the second base meets window w + 1 of the first
    Pc = C.mul(P, 1 << c)
    for s in (rng.randrange(R_MOD), R_MOD - 1, (R_MOD - 1) // 2) + tuple(digit_extremes(c)):
        d0 = recode(s, c)[0]
        s2 = (s - d0) >> c
        assert recode(s2, c)[:-1] == recode(s, c)[1:]
        f.check("P, 2^c P", [P, Pc], [s, s2], C.mul(P, (s + (s2 << c)) % R_MOD))
        f.check("P, -2^c P", [P, C.neg(Pc)], [s, s2], C.mul(P, d0 % R_MOD))
    # digit extremes and the GLV worst cases, on a handful of bases (repeated ones included)
    ks = digit_extremes(c) + digit_extremes(c, 128) + glv_hard_scalars()[::4] + [1, R_MOD - 1, LAMBDA]
    pts = [P, Q, C.neg(P)] * ((len(ks) + 2) // 3)
    f.check("digit extremes", pts[:len(ks)], ks)
    for k in special_scalars()[::7]:
        f.check(f"[k] P, k = {k:#x}", [P], [k], C.mul(P, k))


@pytest.mark.parametrize("resident", [False, True], ids=["generic", "resident"])
def test_msm_g2_long_runs(co, po, frs, resident):
    """half of the scalars equal 1 and a quarter r - 1 (giant buckets: k_long_run, G2 with 32 KB of shared memory), on
    bases k_i G2 with known k_i: the result is (sum k_i s_i) G2"""
    n, m = 1 << 16, 512
    ks = frs(91, m)
    pts = engine.generator_mul(2, ks)
    bases = np.concatenate([pts] * (n // m))
    sc = frs(92, n)
    sc[0::2] = np.frombuffer((1).to_bytes(32, "little"), np.uint8)
    sc[1::4] = np.frombuffer((R_MOD - 1).to_bytes(32, "little"), np.uint8)
    kl, sl = co.fr_list(ks), co.fr_list(sc)
    want = po.g2_to_bytes(po.G2.mul(po.G2_GEN, sum(kl[i % m] * s for i, s in enumerate(sl)) % R_MOD))
    assert np.array_equal(pts[:8], co.g2_gen_mul(ks[:8]))
    B = engine.MsmBases(2, bases, resident_windows=resident)
    try:
        assert B.msm(sc) == want
        # the same with the long runs cancelling: every base once with 1 and once with r - 1
        sc2 = sc.copy()
        sc2[1::2] = np.frombuffer((R_MOD - 1).to_bytes(32, "little"), np.uint8)
        sc2[0::2] = np.frombuffer((1).to_bytes(32, "little"), np.uint8)
        bases2 = np.repeat(pts, 2, axis=0)
        B2 = engine.MsmBases(2, np.concatenate([bases2] * (n // (2 * m))), resident_windows=resident)
        try:
            assert B2.msm(sc2) == infinity_bytes(128)
        finally:
            B2.close()
    finally:
        B.close()
