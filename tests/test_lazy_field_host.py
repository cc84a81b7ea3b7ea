"""field.cuh's redundant-form field operations (values in [0, 2p)) and ec.cuh's madd_lazy, built for the host:
every result is congruent to the exact value and inside its stated bound, and the lazy mixed addition lands on the
canonical madd's residues through every special case."""
import ctypes as C
import os
import subprocess

import pytest

from conftest import ROOT

R = 1 << 256


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    out = tmp_path_factory.mktemp("lazy") / "lazy_host.so"
    subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-o", str(out),
                    os.path.join(ROOT, "tests", "host_shim", "lazy_host.cpp")], check=True)
    return C.CDLL(str(out))


def buf(*vals, n=32):
    return (C.c_uint8 * (n * len(vals)))(*b"".join(v.to_bytes(n, "little") for v in vals))


def limbs(o, n=32):
    raw = bytes(o)
    return [int.from_bytes(raw[i:i + n], "little") for i in range(0, len(raw), n)]


def fq_op(shim, op, a, b=0):
    o = (C.c_uint8 * 32)()
    shim.fq_lazy_op(op, buf(a), buf(b), o)
    return limbs(o)[0]


def edge_and_random(po, q, n, seed):
    rng = po.SplitMix64(seed)
    edge = [0, 1, q - 1, q, q + 1, 2 * q - 2, 2 * q - 1, R % q, (R % q) + q]
    return edge + [(rng.next_fr() * 7 + rng.next_fr()) % (2 * q) for _ in range(n)]


def test_fq_redundant_ops(shim, po):
    q = po.Q_MOD
    rinv = pow(R, -1, q)
    vals = edge_and_random(po, q, 150, 5)
    for i, a in enumerate(vals):
        for b in (vals[(i * 7 + 3) % len(vals)], 2 * q - 1, q, 0):
            r = fq_op(shim, 0, a, b)
            assert r % q == a * b * rinv % q and r < 2 * q and r < a * b // R + q + 1
            r = fq_op(shim, 2, a, b)
            assert r % q == (a - b) % q and r < 2 * q
            r = fq_op(shim, 3, a, b)
            assert r % q == (a + b) % q and r < 2 * q
        r = fq_op(shim, 1, a)
        assert r % q == a * a * rinv % q and r < 2 * q
        assert fq_op(shim, 4, a) == a % q
        assert fq_op(shim, 5, a) == (a % q == 0)
    # the product's wider contract: first operand below R - p, second any 256-bit value
    for a in (4 * q - 1, R - q - 1, 3 * q):
        for b in (2 * q - 1, 4 * q - 1, R - 1, q - 1, 0):
            r = fq_op(shim, 0, a, b)
            assert r % q == a * b * rinv % q and r < a * b // R + q + 1
    for a in ((1 << 255) - 1, 2 * q - 1, 5 * q // 2):      # squaring: below 2^255
        r = fq_op(shim, 1, a)
        assert r % q == a * a * rinv % q and r < a * a // R + q + 1
    # reduction of any T < p R, and a b - c d with all four operands below 2p
    rng = po.SplitMix64(6)
    for t in [0, 1, q * R - 1, q * R - q, (2 * q - 1) ** 2, R - 1] + [rng.next_fr() * rng.next_fr() * 9 % (q * R) for _ in range(100)]:
        o = (C.c_uint8 * 32)()
        shim.fq_reduce_wide_lazy_host(buf(t, n=64), o)
        r = limbs(o)[0]
        assert r % q == t * rinv % q and r < 2 * q
    top = 2 * q - 1
    cases = [(top, top, 0, 0), (0, 0, top, top), (top, top, top, top), (1, 0, top, top), (q, top, top, q)] + \
            [tuple(vals[(i * k + k) % len(vals)] for k in (1, 3, 7, 11)) for i in range(len(vals))]
    for a, b, c, d in cases:
        o = (C.c_uint8 * 32)()
        shim.fq_msub_lazy_host(buf(a), buf(b), buf(c), buf(d), o)
        r = limbs(o)[0]
        assert r % q == (a * b - c * d) * rinv % q and r < 2 * q


class G1:
    """XYZZ / affine byte packing; field elements are 1-tuples."""

    def __init__(self, shim, po):
        self.q, self.k = po.Q_MOD, 1
        self.rinv = pow(R, -1, self.q)
        self.madd_fn, self.canon_fn = shim.g1_madd_host, shim.g1_canonical_host

    def mul(self, a, b):                       # Montgomery product
        return (a[0] * b[0] * self.rinv % self.q,)

    def madd(self, lazy, acc, pt):
        a = buf(*[v for c in acc for v in c])
        self.madd_fn(lazy, a, buf(*[v for c in pt for v in c]))
        v = limbs(a)
        return [tuple(v[i * self.k:(i + 1) * self.k]) for i in range(4)]

    def canonical(self, acc):
        a = buf(*[v for c in acc for v in c])
        self.canon_fn(a)
        v = limbs(a)
        return [tuple(v[i * self.k:(i + 1) * self.k]) for i in range(4)]


def lift(acc, q, mask):                        # add p to the components that mask selects: same residues in [p, 2p)
    return [tuple(v + q if (mask >> (2 * i + j)) & 1 else v for j, v in enumerate(c)) for i, c in enumerate(acc)]


def test_madd_lazy_equals_madd(shim, po):
    """madd_lazy against the canonical madd on the same residues.  The formula's identities do not need the points
    on the curve, so the operands are random field elements; the special cases are built from their definitions."""
    g = G1(shim, po)
    q, k = g.q, g.k
    rng = po.SplitMix64(41)
    rand = lambda: tuple(rng.next_fr() % q for _ in range(k))
    one, zero = tuple([R % q] + [0] * (k - 1)), tuple([0] * k)
    inf = [one, one, zero, zero]

    def check(acc_canon, acc_lazy, pt):
        want = g.madd(0, acc_canon, pt)
        got = g.madd(1, acc_lazy, pt)
        assert max(v for c in got for v in c) < 2 * q
        assert g.canonical(got) == want
        return want, got

    # a chain from infinity: 200 additions, the lazy accumulator never made canonical in between
    canon, lazy = inf, inf
    for i in range(200):
        pt = (rand(), rand())
        canon = g.madd(0, canon, pt)
        lazy = g.madd(1, lazy, pt)
        assert max(v for c in lazy for v in c) < 2 * q
        assert g.canonical(lazy) == canon, i
    for mask in (0, 0xff, 0x55, 0xaa, 0x0f, 0xf0):
        acc = [rand(), rand(), rand(), rand()]
        px, py = rand(), rand()
        # plain addition, accumulator coordinates in [p, 2p)
        check(acc, lift(acc, q, mask), (px, py))
        # P + P: U2 = x, S2 = y -> the doubling branch
        zz, zzz = acc[2], acc[3]
        dbl = [g.mul(px, zz), g.mul(py, zzz), zz, zzz]
        want, _ = check(dbl, lift(dbl, q, mask), (px, py))
        assert want[2] != zero
        # P + (-P): U2 = x, S2 = -y -> infinity
        neg = [g.mul(px, zz), g.mul(tuple((q - v) % q for v in py), zzz), zz, zzz]
        want, got = check(neg, lift(neg, q, mask), (px, py))
        assert want[2] == zero and got[2] == zero
        # accumulator at infinity, zz stored as 0 or as p
        check([acc[0], acc[1], zero, zero], lift([acc[0], acc[1], zero, zero], q, mask), (px, py))
        # adding the identity (0, 0) changes nothing
        _, got = check(acc, lift(acc, q, mask), (zero, zero))
        assert got == lift(acc, q, mask)
