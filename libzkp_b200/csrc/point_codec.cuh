// point_codec.cuh — ark-serialize compressed points: square roots in Fq and Fq2, decoding a compressed G1 / G2 point
// into the uncompressed layout, and encoding an uncompressed point into the compressed one.
//
// Compressed G1 = x (32 B canonical LE), compressed G2 = x.c0 || x.c1 (64 B); the flags sit in the top two bits of the
// last byte: 0x40 = point at infinity, 0x80 = y is the larger of y and -y (canonical integers; in Fq2 c1 decides, then
// c0 - the order write_g1 / write_g2 of dev_util.cuh use for the uncompressed form), both = invalid.
// Decoding checks no subgroup membership (ark's deserialize_compressed_unchecked): the key loaders with validation and
// every verifier form check it on the decoded bytes, as they do for uncompressed input.
#pragma once
#include <string.h>
#include "field.cuh"

namespace lzkp {

// (q + 1) / 4: BN254's q = 3 mod 4, so a^((q+1)/4) is a square root of a whenever a has one
LZ_CONST_ARRAY(kSqrtExp, 0xb61f3f52u, 0x4f082305u, 0x5a1c72a3u, 0x65e05aa4u, 0xa0605617u, 0x6e14116du, 0xb84c680au,
               0x0c19139cu)

// a^((q+1)/4), left to right over the 252 exponent bits: 251 squarings and 108 products.  Every thread runs the same
// exponent, so the branch on a bit never diverges.
LZ_HD Fq fq_pow_sqrt(const Fq &a) {
    Fq r = a;                                                   // bit 251, the top one
#pragma unroll
    for (int limb = 7; limb >= 0; limb--) {
        const uint32_t e = kSqrtExp(limb);
#pragma unroll 1
        for (int b = limb == 7 ? 26 : 31; b >= 0; b--) {
            r = r.sqr();
            if ((e >> b) & 1u) r = r * a;
        }
    }
    return r;
}
// Root of a Montgomery element; false when a is not a square.
LZ_HD bool fq_sqrt(const Fq &a, Fq &root) {
    root = fq_pow_sqrt(a);
    return root.sqr() == a;
}
// x / 2 mod q (any representation: halving commutes with the Montgomery map)
LZ_HD Fq fq_halve(const Fq &x) {
    uint32_t t[8];
    const Fq m = Fq::modulus(), z = Fq::zero();
    add8(t, x.l, (x.l[0] & 1u) ? m.l : z.l);                  // x + q < 2^255: no carry out
    Fq r;
#pragma unroll
    for (int i = 0; i < 7; i++) r.l[i] = (t[i] >> 1) | (t[i + 1] << 31);
    r.l[7] = t[7] >> 1;
    return r;
}
// Root in Fq2 by the norm method: a = a0 + a1 u is a square iff N(a) = a0^2 + a1^2 is one in Fq; then with s = sqrt(N(a))
// and t = (a0 + s) / 2, x0 = t^((q+1)/4) satisfies x0^2 = +-t, and the root is x0 + a1 / (2 x0) u (x0^2 = t) or
// a1 / (2 x0) + x0 u (x0^2 = -t, since -1 is a non-square and t (a0 - s) / 2 = -a1^2 / 4).  t = 0 only when a1 = 0 and a0
// is a non-square; then t = a0 - t = a0 instead, which lands in the second case.  Two exponentiations and one inversion;
// the result is squared and compared with a, so a non-square is rejected whatever the intermediate values were.
LZ_HD bool fq2_sqrt(const Fq2 &a, Fq2 &root) {
    const Fq n = a.c0.sqr() + a.c1.sqr();
    const Fq s = fq_pow_sqrt(n);
    Fq t = fq_halve(a.c0 + s);
    if (t.is_zero()) t = a.c0 - t;
    const Fq x0 = fq_pow_sqrt(t);
    const Fq w = a.c1 * x0.dbl().inverse();
    if (x0.sqr() == t) root = Fq2{x0, w};
    else root = Fq2{w, x0};
    const Fq2 sq{(root.c0 + root.c1) * (root.c0 - root.c1), (root.c0 * root.c1).dbl()};
    return sq == a;
}

// ---- byte helpers (canonical limbs; the flags are the top two bits of limb 7) ----------------------------------------
LZ_HD void fq_load(const uint8_t *b, Fq &c) { memcpy(c.l, b, 32); }
LZ_HD void fq_store(uint8_t *b, const Fq &c, uint32_t flags) {
    memcpy(b, c.l, 32);
    b[31] |= (uint8_t)flags;
}
LZ_HD uint32_t take_flags(Fq &c) {                           // 2 = 0x80 (larger y), 1 = 0x40 (infinity)
    const uint32_t f = c.l[7] >> 30;
    c.l[7] &= 0x3FFFFFFFu;
    return f;
}
LZ_HD bool fq_lt_modulus(const Fq &c) {
    uint32_t d[8];
    const Fq m = Fq::modulus();
    return sub8(d, c.l, m.l) != 0;
}
// canonical y is the larger of y, -y
LZ_HD bool fq_larger(const Fq &y) { return Fq::gt_canonical(y, y.neg()); }
LZ_HD bool fq2_larger(const Fq &y0, const Fq &y1) {
    const Fq n0 = y0.neg(), n1 = y1.neg();
    return y1 == n1 ? Fq::gt_canonical(y0, n0) : Fq::gt_canonical(y1, n1);
}

// ---- compression of uncompressed bytes: format work only (no curve check); the 0x80 bit of the input is not read,
// the sign comes from y.  false for a non-canonical coordinate, flags outside the last byte or both flags set.
LZ_HD bool compress_g1(const uint8_t *in, uint8_t *out) {
    Fq x, y;
    fq_load(in, x);
    fq_load(in + 32, y);
    const uint32_t f = take_flags(y);
    if (!fq_lt_modulus(x) || !fq_lt_modulus(y) || f == 3) return false;     // flags on x make it >= 2^254 > q
    if (f & 1u) { fq_store(out, Fq::zero(), 0x40); return true; }
    fq_store(out, x, fq_larger(y) ? 0x80 : 0);
    return true;
}
LZ_HD bool compress_g2(const uint8_t *in, uint8_t *out) {
    Fq x0, x1, y0, y1;
    fq_load(in, x0);
    fq_load(in + 32, x1);
    fq_load(in + 64, y0);
    fq_load(in + 96, y1);
    const uint32_t f = take_flags(y1);
    if (!fq_lt_modulus(x0) || !fq_lt_modulus(x1) || !fq_lt_modulus(y0) || !fq_lt_modulus(y1) || f == 3) return false;
    if (f & 1u) { fq_store(out, Fq::zero(), 0); fq_store(out + 32, Fq::zero(), 0x40); return true; }
    fq_store(out, x0, 0);
    fq_store(out + 32, x1, fq2_larger(y0, y1) ? 0x80 : 0);
    return true;
}

// ---- decompression into the uncompressed layout (what write_g1 / write_g2 produce for the same point).  false for a
// non-canonical x, flags on x.c0, both flags set, or an x with no point on the curve (G1: y^2 = x^3 + 3; G2, the twist:
// y^2 = x^3 + 3 / (9 + u)).  The infinity flag decodes to the point at infinity whatever the (canonical) x, as the
// uncompressed readers do.
LZ_HD bool decompress_g1(const uint8_t *in, uint8_t *out) {
    Fq x;
    fq_load(in, x);
    const uint32_t f = take_flags(x);
    if (!fq_lt_modulus(x) || f == 3) return false;
    if (f & 1u) {
        fq_store(out, Fq::zero(), 0);
        fq_store(out + 32, Fq::zero(), 0x40);
        return true;
    }
    Fq b;
#pragma unroll
    for (int i = 0; i < 8; i++) b.l[i] = FqParams::B3(i);
    const Fq xm = Fq::from_canonical(x), rhs = xm.sqr() * xm + b;
    Fq y;
    if (!fq_sqrt(rhs, y)) return false;
    Fq yc = y.to_canonical();                                   // y != 0: G1 has odd order, no 2-torsion point
    if (fq_larger(yc) != ((f & 2u) != 0)) yc = yc.neg();
    fq_store(out, x, 0);
    fq_store(out + 32, yc, f & 2u ? 0x80 : 0);
    return true;
}
LZ_HD bool decompress_g2(const uint8_t *in, uint8_t *out) {
    Fq x0, x1;
    fq_load(in, x0);
    fq_load(in + 32, x1);
    const uint32_t f0 = take_flags(x0), f = take_flags(x1);
    if (f0 || !fq_lt_modulus(x0) || !fq_lt_modulus(x1) || f == 3) return false;
    if (f & 1u) {
        fq_store(out, Fq::zero(), 0); fq_store(out + 32, Fq::zero(), 0); fq_store(out + 64, Fq::zero(), 0);
        fq_store(out + 96, Fq::zero(), 0x40);
        return true;
    }
    Fq2 b;
#pragma unroll
    for (int i = 0; i < 8; i++) { b.c0.l[i] = FqParams::G2B_C0(i); b.c1.l[i] = FqParams::G2B_C1(i); }
    const Fq2 xm{Fq::from_canonical(x0), Fq::from_canonical(x1)};
    const Fq2 rhs = xm.sqr() * xm + b;
    Fq2 y;
    if (!fq2_sqrt(rhs, y)) return false;
    Fq y0 = y.c0.to_canonical(), y1 = y.c1.to_canonical();     // y != 0: the twist has odd order as well
    if (fq2_larger(y0, y1) != ((f & 2u) != 0)) { y0 = y0.neg(); y1 = y1.neg(); }
    fq_store(out, x0, 0);
    fq_store(out + 32, x1, 0);
    fq_store(out + 64, y0, 0);
    fq_store(out + 96, y1, f & 2u ? 0x80 : 0);
    return true;
}

}  // namespace lzkp
