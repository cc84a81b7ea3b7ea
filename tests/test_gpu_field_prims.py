"""field.cuh on the device (sm_100a build: the inline-PTX carry chains and the out-of-line Fq2 product fq2_mul_call /
fq2_sqr_call) against Python integers, at the edges of every operation's input range and on 10^5 seeded random inputs
per operation.  Every device output must also be bit-identical to the host build's (the portable C++ bodies) on the same
input: for the redundant-form operations the representative in [0, 2p) is deterministic, so this is stronger than
checking the residue."""
import random

import numpy as np
import pytest

import prim_shim as ps
from prim_shim import R, ints, records

pytestmark = pytest.mark.gpu
N_RANDOM = 100_000
LIMB_EDGES = (0, 1, 0x80000000, 0xffffffff)


@pytest.fixture(scope="module")
def dev(tmp_path_factory):
    return ps.device(tmp_path_factory)


@pytest.fixture(scope="module")
def host(tmp_path_factory):
    return ps.host(tmp_path_factory)


def both(dev, host, fam, code, rec):
    """device output, after requiring it to equal the host build's bit for bit"""
    d, h = dev.run(fam, code, rec), host.run(fam, code, rec)
    bad = np.flatnonzero((d != h).any(axis=1))
    assert bad.size == 0, (fam, code, "device != host build", bad[:5].tolist(), rec[bad[0]].tolist())
    return d


def check(name, got, want, inputs):
    bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
    assert not bad, (name, len(bad), "first:", [hex(v) for v in inputs[bad[0]]], hex(got[bad[0]]), hex(want[bad[0]]))


def edges(m):
    """0, 1, 2, m-1, m-2, (m +- 1)/2, R, R^2 and R^-1 mod m, 2^k at the limb boundaries, one limb all ones, m - 2^(32k)"""
    e = [0, 1, 2, m - 1, m - 2, (m - 1) // 2, (m + 1) // 2, R % m, R * R % m, pow(R, -1, m)]
    e += [1 << k for k in sorted({31, 32, 63, 64, 95, 96, 127, 128, 159, 160, 191, 192, 223, 224, 252, 253})]
    e += [0xffffffff << (32 * k) for k in range(8)] + [m - (1 << (32 * k)) for k in range(8)]
    return sorted({v for v in e if v < m})


def lazy_edges(q):
    return sorted(set(edges(q)) | {q, q + 1, 2 * q - 2, 2 * q - 1})


def random_below(rng, bound, n):
    """half uniform, half built from limbs that are 0, 1, 2^31, 2^32 - 1 or random (where rare carries live)"""
    out = []
    for i in range(n):
        if i & 1:
            v = rng.getrandbits(256)
        else:
            v = 0
            for j in range(8):
                v |= (rng.choice(LIMB_EDGES) if rng.random() < 0.6 else rng.getrandbits(32)) << (32 * j)
        out.append(v % bound if v >= bound else v)
    return out


def operands(rng, edge, bound, k, n=N_RANDOM):
    """k operand columns: every edge against every edge (k = 1: each edge), then n random rows"""
    if k == 1:
        cols = [list(edge)]
    else:
        cols = [[a for a in edge for _ in edge], [b for _ in edge for b in edge]]
        cols += [[edge[(i * 7 + 3 * j) % len(edge)] for i in range(len(edge) ** 2)] for j in range(k - 2)]
    return [c + random_below(rng, bound, n) for c in cols]


def field_rec(*cols):
    return records(32, *[(8 * j, c) for j, c in enumerate(cols)])


FIELDS = [("fr", ps.FAM_FR, 0x30644E72E131A029B85045B68181585D2833E84879B9709143E1F593F0000001),
          ("fq", ps.FAM_FQ, 0x30644E72E131A029B85045B68181585D97816A916871CA8D3C208C16D87CFD47)]


@pytest.mark.parametrize("name, fam, m", FIELDS, ids=[f[0] for f in FIELDS])
def test_canonical_field_ops(dev, host, name, fam, m):
    rng = random.Random(0x5eed ^ fam)
    ri = pow(R, -1, m)
    e = edges(m)
    a, b = operands(rng, e, m, 2)
    rec = field_rec(a, b)
    run = lambda code: ints(both(dev, host, fam, code, rec)[:, :8])
    inp = list(zip(a, b))
    check("mul", run(0), [x * y * ri % m for x, y in inp], inp)
    check("add", run(2), [(x + y) % m for x, y in inp], inp)
    check("sub", run(3), [(x - y) % m for x, y in inp], inp)
    check("gt_canonical", run(10), [int(x > y) for x, y in inp], inp)
    check("==", run(12), [int(x == y) for x, y in inp], inp)
    (u,) = operands(rng, e, m, 1)
    rec = field_rec(u)
    run = lambda code: ints(both(dev, host, fam, code, rec)[:, :8])
    inp = [(x,) for x in u]
    check("sqr", run(1), [x * x * ri % m for x in u], inp)
    check("neg", run(4), [(-x) % m for x in u], inp)
    check("dbl", run(5), [2 * x % m for x in u], inp)
    check("from_canonical", run(7), [x * R % m for x in u], inp)
    check("to_canonical", run(8), [x * ri % m for x in u], inp)
    check("is_zero", run(11), [int(x == 0) for x in u], inp)
    # the inverse of the element x R^-1 is stored as (x R^-1)^-1 R = R^2 / x;  0 -> 0
    v = u[:len(e) + 20_000]
    got = ints(both(dev, host, fam, 6, field_rec(v))[:, :8])
    check("inverse", got, [R * R * pow(x, -1, m) % m if x else 0 for x in v], [(x,) for x in v])
    # a b - c d with one reduction; a b == c d and a b == c d +- 1 (the borrow at wide_fix_negative's boundary)
    a, b, c, d = operands(rng, e, m, 4, n=N_RANDOM // 2)
    for i in range(400):
        x, y = rng.getrandbits(126) + 1, rng.getrandbits(126) + 1
        for s in (-1, 0, 1):
            a.append(1), b.append(x * y + s), c.append(x), d.append(y)
        a.append(y), b.append(x), c.append(x), d.append(y)
    a.append(m - 1), b.append(m - 1), c.append(m - 1), d.append(m - 1)
    inp = list(zip(a, b, c, d))
    got = ints(both(dev, host, fam, 9, field_rec(a, b, c, d))[:, :8])
    check("msub", got, [(w * x - y * z) * ri % m for w, x, y, z in inp], inp)


def test_redundant_form_ops(dev, host):
    """The [0, 2p) operations of the G1 gather kernel, each against the bound written beside it in field.cuh."""
    q = FIELDS[1][2]
    fam, ri = ps.FAM_FQ, pow(R, -1, q)
    rng = random.Random(0x1a2f)
    le = lazy_edges(q)
    # mul_lazy: a < R - p, b < R;  (a b + m p) / R < a b / R + p
    ea = sorted(set(le) | {R - q - 1, (1 << 255) - 1, 4 * q - 1, 3 * q})
    eb = sorted(set(ea) | {R - 1, R - 2})
    a = [x for x in ea for _ in eb] + random_below(rng, R - q, N_RANDOM)
    b = [y for _ in ea for y in eb] + random_below(rng, R, N_RANDOM)
    r = ints(both(dev, host, fam, 13, field_rec(a, b))[:, :8])
    inp = list(zip(a, b))
    check("mul_lazy residue", [v % q for v in r], [x * y * ri % q for x, y in inp], inp)
    check("mul_lazy bound", [int(v * R < x * y + q * R) for v, (x, y) in zip(r, inp)], [1] * len(r), inp)
    # operands below 2p: below 2p (and below 1.76p)
    small = [i for i, (x, y) in enumerate(inp) if x < 2 * q and y < 2 * q]
    assert len(small) > 1000 and all(r[i] < 2 * q for i in small)
    # sqr_lazy: a < 2^255, result < a^2 / R + p
    u = sorted(set(le) | {(1 << 255) - 1, (1 << 255) - q}) + random_below(rng, 1 << 255, N_RANDOM)
    r = ints(both(dev, host, fam, 14, field_rec(u))[:, :8])
    inp = [(x,) for x in u]
    check("sqr_lazy residue", [v % q for v in r], [x * x * ri % q for x in u], inp)
    check("sqr_lazy bound", [int(v * R < x * x + q * R) for v, x in zip(r, u)], [1] * len(r), inp)
    # add_2p / sub_2p / is_zero_2p / canonical on [0, 2p): exact representatives
    a, b = operands(rng, le, 2 * q, 2)
    rec = field_rec(a, b)
    inp = list(zip(a, b))
    p2 = 2 * q
    check("add_2p", ints(both(dev, host, fam, 16, rec)[:, :8]), [x + y - p2 if x + y >= p2 else x + y for x, y in inp], inp)
    check("sub_2p", ints(both(dev, host, fam, 17, rec)[:, :8]), [x - y + p2 if x < y else x - y for x, y in inp], inp)
    check("is_zero_2p", ints(both(dev, host, fam, 18, rec)[:, :8]), [int(x in (0, q)) for x in a], inp)
    check("canonical", ints(both(dev, host, fam, 19, rec)[:, :8]), [x % q for x in a], inp)
    # msub_lazy: all four below 2p -> below 2p
    a, b, c, d = operands(rng, le, 2 * q, 4, n=N_RANDOM // 2)
    for i in range(400):
        x, y = rng.getrandbits(127) + 1, rng.getrandbits(127) + 1
        for s in (-1, 0, 1):
            a.append(1), b.append(x * y + s), c.append(x), d.append(y)
    t = 2 * q - 1
    for row in ((t, t, 0, 0), (0, 0, t, t), (t, t, t, t), (1, 0, t, t), (q, t, t, q), (t, t, t, t - 1), (t, t - 1, t, t)):
        for col, v in zip((a, b, c, d), row):
            col.append(v)
    inp = list(zip(a, b, c, d))
    r = ints(both(dev, host, fam, 15, field_rec(a, b, c, d))[:, :8])
    check("msub_lazy residue", [v % q for v in r], [(w * x - y * z) * ri % q for w, x, y, z in inp], inp)
    check("msub_lazy bound", [int(v < 2 * q) for v in r], [1] * len(r), inp)


@pytest.mark.parametrize("name, fam, m", FIELDS, ids=[f[0] for f in FIELDS])
def test_wide_ops(dev, host, name, fam, m):
    rng = random.Random(0x3dee ^ fam)
    ri = pow(R, -1, m)
    # reduce_wide / reduce_wide_lazy: T < p 2^256.  p 2^256 - 1, T_lo = 0, T_hi = p - 1, and random
    ts = [0, 1, m * R - 1, m * R - m, (m - 1) * R, (m - 1) * R + R - 1, (2 * m - 1) ** 2, R - 1, R, (m - 1) ** 2]
    ts += [hi * R for hi in edges(m)] + [(m - 1) * R + lo for lo in edges(m)] + [k * R + (R - 1) for k in edges(m)]
    ts += [rng.getrandbits(512) % (m * R) for _ in range(N_RANDOM)]
    ts += [(rng.getrandbits(256) % m) * (rng.getrandbits(256) % m) for _ in range(N_RANDOM // 4)]
    rec = records(32, (0, ps.words(ts, 16)))
    inp = [(t,) for t in ts]
    check("reduce_wide", ints(both(dev, host, fam, 20, rec)[:, :8]), [t * ri % m for t in ts], inp)
    r = ints(both(dev, host, fam, 21, rec)[:, :8])
    check("reduce_wide_lazy residue", [v % m for v in r], [t * ri % m for t in ts], inp)
    check("reduce_wide_lazy bound", [int(v <= (t >> 256) + m and v < 2 * m) for v, t in zip(r, ts)], [1] * len(r), inp)
    # mul_wide: any 256-bit operands, the exact 512-bit product
    e = sorted(set(edges(m)) | {R - 1, R - 2, R >> 1, (R >> 1) - 1})
    a, b = operands(rng, e, R, 2)
    inp = list(zip(a, b))
    check("mul_wide", ints(both(dev, host, fam, 22, field_rec(a, b))), [x * y for x, y in inp], inp)
    # add16 / sub16: carry and borrow out of 512 bits
    W = 1 << 512
    we = [0, 1, W - 1, W - 2, R - 1, R, W >> 1, (W >> 1) - 1] + [0xffffffff << (32 * k) for k in range(16)]
    x = [s for s in we for _ in we] + [rng.getrandbits(512) for _ in range(N_RANDOM // 2)] + \
        [rng.getrandbits(512) | (W - R) for _ in range(N_RANDOM // 2)]
    y = [t for _ in we for t in we] + [rng.getrandbits(512) for _ in range(N_RANDOM // 2)] + \
        [rng.getrandbits(512) | (W - 1 - ((1 << 64) - 1)) for _ in range(N_RANDOM // 2)]
    rec = records(32, (0, ps.words(x, 16)), (16, ps.words(y, 16)))
    inp = list(zip(x, y))
    out = both(dev, host, fam, 23, rec)
    check("add16", ints(out[:, :16]), [(s + t) % W for s, t in inp], inp)
    check("add16 carry", out[:, 16].tolist(), [int(s + t >= W) for s, t in inp], inp)
    out = both(dev, host, fam, 24, rec)
    check("sub16", ints(out[:, :16]), [(s - t) % W for s, t in inp], inp)
    check("sub16 borrow", out[:, 16].tolist(), [int(s < t) for s, t in inp], inp)


def test_fq2_ops(dev, host):
    """The device's Fq2 product and square are the out-of-line fq2_mul_call / fq2_sqr_call (fq2_mul_lazy and the
    two-product square); the host build's are the inline Karatsuba forms."""
    q = FIELDS[1][2]
    ri = pow(R, -1, q)
    rng = random.Random(0xf2)
    e = [v for v in edges(q)]
    n = N_RANDOM
    a0, a1 = [x for x in e for _ in e], [y for _ in e for y in e]
    b0, b1 = list(reversed(a0)), list(a1)
    a0 += random_below(rng, q, n); a1 += random_below(rng, q, n); b0 += random_below(rng, q, n); b1 += random_below(rng, q, n)
    # a0 b0 - a1 b1 exactly 0, and -1 (as integers: the borrow of the c0 difference)
    for _ in range(500):
        x, y, k = rng.randrange(1, q), rng.randrange(1, q), rng.randrange(2, q)
        a0 += [x, 1, x]; a1 += [y, 1, 1]; b0 += [y, k - 1, 1]; b1 += [x, k, x - 1]
    rec = records(32, (0, a0), (8, a1), (16, b0), (24, b1))
    inp = list(zip(a0, a1, b0, b1))

    def fq2(out):
        v = ints(out.reshape(-1, 8))
        return list(zip(v[0::2], v[1::2]))

    want_mul = [((x0 * y0 - x1 * y1) * ri % q, (x0 * y1 + x1 * y0) * ri % q) for x0, x1, y0, y1 in inp]
    check("fq2 *", fq2(both(dev, host, ps.FAM_FQ2, 0, rec)), want_mul, inp)
    check("fq2_mul_lazy", fq2(both(dev, host, ps.FAM_FQ2, 5, rec)), want_mul, inp)
    check("fq2 sqr", fq2(both(dev, host, ps.FAM_FQ2, 1, rec)),
          [((x0 * x0 - x1 * x1) * ri % q, 2 * x0 * x1 * ri % q) for x0, x1, _, _ in inp], inp)
    check("fq2_mul_xi", fq2(both(dev, host, ps.FAM_FQ2, 3, rec)),
          [((9 * x0 - x1) % q, (9 * x1 + x0) % q) for x0, x1, _, _ in inp], inp)
    check("fq2_conj", fq2(both(dev, host, ps.FAM_FQ2, 4, rec)), [(x0, (-x1) % q) for x0, x1, _, _ in inp], inp)
    check("fq2 +", fq2(both(dev, host, ps.FAM_FQ2, 6, rec)),
          [((x0 + y0) % q, (x1 + y1) % q) for x0, x1, y0, y1 in inp], inp)
    check("fq2 -", fq2(both(dev, host, ps.FAM_FQ2, 7, rec)),
          [((x0 - y0) % q, (x1 - y1) % q) for x0, x1, y0, y1 in inp], inp)
    # inverse of the element (x0 + x1 u) R^-1, stored times R; 0 -> 0
    m = len(e) ** 2 + 20_000
    rec = rec[:m]
    want = []
    for x0, x1, _, _ in inp[:m]:
        nrm = (x0 * x0 + x1 * x1) % q
        if nrm == 0:
            want.append((0, 0))
            continue
        k = R * R * pow(nrm, -1, q)          # (x R^-1)^-1 R = conj(x) R^2 / |x|^2
        want.append((x0 * k % q, (-x1) * k % q))
    check("fq2 inverse", fq2(both(dev, host, ps.FAM_FQ2, 2, rec)), want, inp[:m])


def test_fq_half(dev):
    """coop::fq_half on [0, 2p), odd and even: (a + p [a odd]) / 2 exactly, which is a / 2 mod p."""
    q = FIELDS[1][2]
    rng = random.Random(0x4a1f)
    u = lazy_edges(q) + [q - 3, q + 2, q + 3] + random_below(rng, 2 * q, N_RANDOM)
    got = ints(dev.fq_half(ps.words(u)))
    inp = [(x,) for x in u]
    check("fq_half", got, [(x + q) >> 1 if x & 1 else x >> 1 for x in u], inp)
    inv2 = pow(2, -1, q)
    assert all(g % q == x * inv2 % q for g, x in zip(got[:5000], u[:5000]))
