// ec.cuh — BN254 G1 / G2 group law for sm_100a in extended Jacobian ("XYZZ") coordinates.
//
// Replaces ark-ec's short_weierstrass::Projective arithmetic used inside the five
// MSMs and the proof assembly of ark-groth16's create_proof_with_assignment
// (reached from the reference at src/backend/snark.rs:364 and :442).  Group
// elements are unique, so any correct law yields the same affine results; XYZZ is
// chosen because the mixed addition that dominates bucket / table accumulation costs
// 8M + 2S with no inversion.
//
// Affine points use (0, 0) for the point at infinity ((0,0) is on neither curve);
// XYZZ points use zz == 0.  All special cases (infinity, P + P, P + (-P)) are
// handled, because proving-key queries legitimately contain identity points and
// repeated points (SURVEY.md §7 hard part 5).
#pragma once
#include "field.cuh"

namespace lzkp {

template <class F>
struct Affine {
    F x, y;
    LZ_HD bool is_inf() const { return x.is_zero() && y.is_zero(); }
    LZ_HD static Affine inf() { return Affine{F::zero(), F::zero()}; }
    LZ_HD Affine neg() const { return Affine{x, y.neg()}; }
};

template <class F>
struct XYZZ {
    F x, y, zz, zzz;
    LZ_HD bool is_inf() const { return zz.is_zero(); }
    LZ_HD static XYZZ inf() { return XYZZ{F::one(), F::one(), F::zero(), F::zero()}; }
    LZ_HD static XYZZ from_affine(const Affine<F> &p) {
        if (p.is_inf()) return inf();
        return XYZZ{p.x, p.y, F::one(), F::one()};
    }
    LZ_HD XYZZ neg() const { return XYZZ{x, y.neg(), zz, zzz}; }

    // 2 * (affine p), p != inf   (mdbl-2008-s-1, a = 0).  Rare branch of madd: not inlined.
    LZ_COLD static XYZZ dbl_affine(const Affine<F> &p) {
        if (p.y.is_zero()) return inf();
        F U = p.y.dbl(), V = U.sqr(), W = U * V, S = p.x * V;
        F xx = p.x.sqr(), M = xx.dbl() + xx;
        XYZZ r;
        r.x = M.sqr() - S.dbl();
        r.y = F::msub(M, S - r.x, W, p.y);
        r.zz = V;
        r.zzz = W;
        return r;
    }
    // *this = 2 * *this   (dbl-2008-s-1, a = 0): 6M + 3S
    LZ_HD void dbl() {
        if (is_inf()) return;
        if (y.is_zero()) { *this = inf(); return; }
        F U = y.dbl(), V = U.sqr(), W = U * V, S = x * V;
        F xx = x.sqr(), M = xx.dbl() + xx;
        F X3 = M.sqr() - S.dbl();
        F Y3 = F::msub(M, S - X3, W, y);
        x = X3; y = Y3;
        zz = V * zz;
        zzz = W * zzz;
    }
    LZ_COLD void dbl_cold() { dbl(); }
    LZ_COLD void add_cold(const XYZZ &q) { add(q); }
    LZ_COLD void madd_cold(const Affine<F> &p) { madd(p); }
    // *this += affine p   (madd-2008-s): 8M + 2S
    LZ_HD void madd(const Affine<F> &p) {
        if (p.is_inf()) return;
        if (is_inf()) { *this = from_affine(p); return; }
        F U2 = p.x * zz, S2 = p.y * zzz;
        F Pp = U2 - x, R = S2 - y;
        if (Pp.is_zero()) {
            if (R.is_zero()) *this = dbl_affine(p);
            else *this = inf();
            return;
        }
        F PP = Pp.sqr(), PPP = Pp * PP, Q = x * PP;
        F X3 = R.sqr() - PPP - Q.dbl();
        F Y3 = F::msub(R, Q - X3, y, PPP);
        x = X3; y = Y3;
        zz = zz * PP;
        zzz = zzz * PPP;
    }
    // madd with the accumulator in field.cuh's redundant form (F = Fq): x, y, zz, zzz in [0, 2p), p canonical.  The
    // same formula and residues as madd without the final subtraction of each product; canonical() brings the result
    // back.  The zero tests compare residues (0 or p), not bit patterns.
    // Bounds in multiples of p (R = 2^256 = 5.29p; a lazy product is < a b / R + p):
    LZ_HD void madd_lazy(const Affine<F> &p) {
        if (p.is_inf()) return;
        if (zz.is_zero_2p()) { *this = from_affine(p); return; }
        F U2 = F::mul_lazy(p.x, zz), S2 = F::mul_lazy(p.y, zzz);     // 1 x 2: < 1.38
        F Pp = F::sub_2p(U2, x), R = F::sub_2p(S2, y);               // [0, 2)
        if (Pp.is_zero_2p()) {
            if (R.is_zero_2p()) *this = dbl_affine(p);
            else *this = inf();
            return;
        }
        F PP = Pp.sqr_lazy();                                        // 2 x 2: < 1.76
        F PPP = F::mul_lazy(Pp, PP), Q = F::mul_lazy(x, PP);         // 2 x 1.76: < 1.67
        F RR = R.sqr_lazy();                                         // < 1.76
        F X3 = F::sub_2p(F::sub_2p(RR, PPP), F::add_2p(Q, Q));       // [0, 2) from operands < 2
        F Y3 = F::msub_lazy(R, F::sub_2p(Q, X3), y, PPP);            // all four < 2: < 2
        x = X3; y = Y3;
        zz = F::mul_lazy(zz, PP);                                    // 2 x 1.76: < 1.67
        zzz = F::mul_lazy(zzz, PPP);                                 // 2 x 1.67: < 1.63
    }
    // [0, 2p) coordinates -> canonical
    LZ_HD XYZZ canonical() const { return XYZZ{x.canonical(), y.canonical(), zz.canonical(), zzz.canonical()}; }
    // *this += q   (add-2008-s): 12M + 2S
    LZ_HD void add(const XYZZ &q) {
        if (q.is_inf()) return;
        if (is_inf()) { *this = q; return; }
        F U1 = x * q.zz, U2 = q.x * zz, S1 = y * q.zzz, S2 = q.y * zzz;
        F Pp = U2 - U1, R = S2 - S1;
        if (Pp.is_zero()) {
            if (R.is_zero()) dbl_cold();
            else *this = inf();
            return;
        }
        F PP = Pp.sqr(), PPP = Pp * PP, Q = U1 * PP;
        F X3 = R.sqr() - PPP - Q.dbl();
        F Y3 = F::msub(R, Q - X3, S1, PPP);
        x = X3; y = Y3;
        zz = zz * q.zz * PP;
        zzz = zzz * q.zzz * PPP;
    }
    // x/zz, y/zzz with one inversion:  t = 1/(zz*zzz); 1/zz = t*zzz; 1/zzz = t*zz
    LZ_COLD Affine<F> to_affine() const {
        if (is_inf()) return Affine<F>::inf();
        F t = (zz * zzz).inverse();
        return Affine<F>{x * (t * zzz), y * (t * zz)};
    }
};

// k * p by signed 4-bit windows: digits d_i in [-8, 8] with k = sum d_i 16^i (carries resolved LSB-first into a
// bitmask), one table of p .. 8p, then per window four doublings and at most one addition.  Against bit-by-bit
// double-and-add this does a quarter of the additions, and the lanes of a warp (different scalars) stay on the same
// instruction except where a digit is zero - a divergent `if (bit)` made every lane pay for every addition.
template <class F, int LIMBS>
LZ_COLD XYZZ<F> scalar_mul_window(const XYZZ<F> &p, const uint32_t (&k)[LIMBS]) {
    constexpr int NW = LIMBS * 8;
    static_assert(NW <= 64, "carry mask is 64 bits");
    XYZZ<F> T[8];
    T[0] = p;
    T[1] = p;
    T[1].dbl_cold();
#pragma unroll 1
    for (int i = 2; i < 8; i++) {
        T[i] = T[i - 1];
        T[i].add_cold(p);
    }
    uint64_t carries = 0;
    uint32_t c = 0;
#pragma unroll 1
    for (int i = 0; i < NW; i++) {
        const uint32_t v = ((k[i >> 3] >> ((i & 7) * 4)) & 15u) + c;
        c = v >= 8u ? 1u : 0u;
        carries |= (uint64_t)c << i;
    }
    XYZZ<F> acc = XYZZ<F>::inf();
#pragma unroll 1
    for (int i = NW; i >= 0; i--) {
        acc.dbl_cold(); acc.dbl_cold(); acc.dbl_cold(); acc.dbl_cold();
        int d;
        if (i == NW) d = (int)c;
        else {
            const uint32_t cin = i ? (uint32_t)(carries >> (i - 1)) & 1u : 0u, cout = (uint32_t)(carries >> i) & 1u;
            d = (int)(((k[i >> 3] >> ((i & 7) * 4)) & 15u) + cin) - (int)(16u * cout);
        }
        if (d != 0) {                        // one addition for both signs: lanes with opposite signs do not serialise
            XYZZ<F> q = T[(d < 0 ? -d : d) - 1];
            if (d < 0) q.y = q.y.neg();
            acc.add_cold(q);
        }
    }
    return acc;
}
// k * p for a canonical 254-bit scalar (limbs little-endian)
template <class F>
LZ_COLD XYZZ<F> scalar_mul(const XYZZ<F> &p, const Fr &k_canonical) {
    return scalar_mul_window<F, 8>(p, k_canonical.l);
}

// ---- GLV split of a BN254 scalar: k = +-k1 +- k2 * lambda (mod r) with k1, k2 < 2^128, where lambda is the
// eigenvalue of the G1 endomorphism phi(x, y) = (beta * x, y).  Halves the serial doubling chain of a
// variable-base scalar multiplication (proof assembly: s * A and r * B1).  Lattice basis (a1, b1), (a2, b2)
// from the extended Euclidean algorithm on (r, lambda); c_i = floor(k * g_i / 2^256) with g_i = floor(2^256 *
// {b2, -b1} / r) (checked against exact rounding over 2 * 10^5 scalars: |k1|, |k2| <= 2^127).
struct GlvSplit {
    uint32_t k1[4], k2[4];
    bool neg1, neg2, ok;      // ok == false: magnitudes did not fit 128 bits (never observed) -> caller uses the plain ladder
};
// out (no limbs) = low limbs of a (na limbs) * b (nb limbs)
template <int NO, int NA, int NB>
LZ_HD void mul_limbs(uint32_t (&out)[NO], const uint32_t (&a)[NA], const uint32_t (&b)[NB]) {
    uint64_t acc = 0, hi = 0;
#pragma unroll
    for (int k = 0; k < NO; k++) {
#pragma unroll
        for (int i = 0; i < NA; i++) {
            int j = k - i;
            if (j < 0 || j >= NB) continue;
            uint64_t p = (uint64_t)a[i] * b[j];
            acc += (uint32_t)p;
            hi += p >> 32;
        }
        out[k] = (uint32_t)acc;
        acc = (acc >> 32) + hi;
        hi = 0;
    }
}
LZ_HD GlvSplit glv_split(const Fr &k) {
    const uint32_t G1C[5] = {0x00ff6565u, 0x5398fd03u, 0xa773d2d2u, 0x4ccef014u, 0x00000002u};
    const uint32_t G2C[3] = {0xc7e0b3d7u, 0xd91d232eu, 0x00000002u};
    const uint32_t A1[4] = {0x7d4f1128u, 0x8211bbebu, 0xeeb859fcu, 0x6f4d8248u};
    const uint32_t A2[2] = {0x94d213e3u, 0x89d32568u};          // a2 = -b1
    const uint32_t B2[4] = {0x1221250bu, 0x0be4e154u, 0xeeb859fdu, 0x6f4d8248u};
    uint32_t t13[13], t11[11], c1[5], c2[3];
    mul_limbs<13, 8, 5>(t13, k.l, G1C);
#pragma unroll
    for (int i = 0; i < 5; i++) c1[i] = t13[8 + i];
    mul_limbs<11, 8, 3>(t11, k.l, G2C);
#pragma unroll
    for (int i = 0; i < 3; i++) c2[i] = t11[8 + i];
    // k1 = k - c1 a1 - c2 a2,  k2 = c1 |b1| - c2 b2   (mod 2^256, two's complement)
    uint32_t p1[8], p2[8], p3[8], p4[8], k1[8], k2[8], t[8];
    mul_limbs<8, 5, 4>(p1, c1, A1);
    mul_limbs<8, 3, 2>(p2, c2, A2);
    mul_limbs<8, 5, 2>(p3, c1, A2);       // |b1| == a2
    mul_limbs<8, 3, 4>(p4, c2, B2);
    sub8(t, k.l, p1);
    sub8(k1, t, p2);
    sub8(k2, p3, p4);
    GlvSplit o;
    o.neg1 = (k1[7] >> 31) != 0;
    o.neg2 = (k2[7] >> 31) != 0;
    uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (o.neg1) { sub8(t, zero, k1);
#pragma unroll
        for (int i = 0; i < 8; i++) k1[i] = t[i]; }
    if (o.neg2) { sub8(t, zero, k2);
#pragma unroll
        for (int i = 0; i < 8; i++) k2[i] = t[i]; }
    o.ok = (k1[4] | k1[5] | k1[6] | k1[7] | k2[4] | k2[5] | k2[6] | k2[7]) == 0;
#pragma unroll
    for (int i = 0; i < 4; i++) { o.k1[i] = k1[i]; o.k2[i] = k2[i]; }
    return o;
}
// k * p for a 128-bit magnitude
template <class F>
LZ_COLD XYZZ<F> scalar_mul_u128(const XYZZ<F> &p, const uint32_t (&k)[4]) {
    return scalar_mul_window<F, 4>(p, k);
}

// k1 * p + k2 * phi(p) for 64-bit k1 = (k[0], k[1]) and k2 = (k[2], k[3]), phi(x, y) = (beta x, y) = [lambda] (x, y):
// the two signed 4-bit window ladders share their doublings (17 windows: 68 doublings and at most 34 additions, where a
// 128-bit scalar needs 132 and 33).  Used with RANDOM (k1, k2): the coefficient is k1 + lambda k2 mod r, and
// (k1, k2) -> k1 + lambda k2 is injective on [0, 2^64)^2 (the GLV lattice of lambda has no non-zero point in that box:
// its reduced basis, glv_split's A1 / A2 / B2, has entries of 127 bits), so the coefficient still takes 2^128 values.
static LZ_COLD XYZZ<Fq> scalar_mul_glv64(const XYZZ<Fq> &p, const uint32_t (&k)[4]) {
    XYZZ<Fq> T[8];
    T[0] = p;
    T[1] = p;
    T[1].dbl_cold();
#pragma unroll 1
    for (int i = 2; i < 8; i++) {
        T[i] = T[i - 1];
        T[i].add_cold(p);
    }
    Fq beta;
#pragma unroll
    for (int i = 0; i < 8; i++) beta.l[i] = FqParams::BETA(i);
    uint32_t carries[2] = {0, 0}, top[2] = {0, 0};
#pragma unroll 1
    for (int h = 0; h < 2; h++) {
        uint32_t c = 0;
#pragma unroll 1
        for (int i = 0; i < 16; i++) {
            const uint32_t v = ((k[2 * h + (i >> 3)] >> ((i & 7) * 4)) & 15u) + c;
            c = v >= 8u ? 1u : 0u;
            carries[h] |= c << i;
        }
        top[h] = c;
    }
    XYZZ<Fq> acc = XYZZ<Fq>::inf();
#pragma unroll 1
    for (int i = 16; i >= 0; i--) {
        acc.dbl_cold(); acc.dbl_cold(); acc.dbl_cold(); acc.dbl_cold();
#pragma unroll 1
        for (int h = 0; h < 2; h++) {
            int d;
            if (i == 16) d = (int)top[h];
            else {
                const uint32_t cin = i ? (carries[h] >> (i - 1)) & 1u : 0u, cout = (carries[h] >> i) & 1u;
                d = (int)(((k[2 * h + (i >> 3)] >> ((i & 7) * 4)) & 15u) + cin) - (int)(16u * cout);
            }
            if (d != 0) {
                XYZZ<Fq> q = T[(d < 0 ? -d : d) - 1];
                if (h) q.x = q.x * beta;
                if (d < 0) q.y = q.y.neg();
                acc.add_cold(q);
            }
        }
    }
    return acc;
}
// lambda (the eigenvalue of phi on G1: phi(P) = [lambda] P for FqParams::BETA), Montgomery form mod r
// lambda = 0x30644e72e131a029048b6e193fd84104cc37a73fec2bc5e9b8ca0b2d36636f23 (checked with the big-integer oracle)
LZ_HD Fr glv_lambda_mont() {
    const uint32_t v[8] = {0x55fcd653u, 0x0363f299u, 0x5fc1e200u, 0x73e7950bu, 0x576d9d24u, 0xc5fce83eu, 0xa1c3a4d4u, 0x059c805du};
    Fr r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.l[i] = v[i];
    return r;
}
// k1 + lambda k2 mod r as a canonical residue
LZ_HD Fr glv64_coefficient(const uint32_t (&k)[4]) {
    Fr k1 = Fr::zero(), k2 = Fr::zero();
    k1.l[0] = k[0]; k1.l[1] = k[1];
    k2.l[0] = k[2]; k2.l[1] = k[3];
    return k1 + k2 * glv_lambda_mont();          // (k2)(lambda R) R^-1 = k2 lambda, canonical
}

using G1Affine = Affine<Fq>;
using G2Affine = Affine<Fq2>;
using G1XYZZ = XYZZ<Fq>;
using G2XYZZ = XYZZ<Fq2>;

// y^2 == x^3 + b ?
static LZ_COLD bool g1_on_curve(const G1Affine &p) {
    if (p.is_inf()) return true;
    Fq b3;
#pragma unroll
    for (int i = 0; i < 8; i++) b3.l[i] = FqParams::B3(i);
    return p.y.sqr() == p.x.sqr() * p.x + b3;
}
static LZ_COLD bool g2_on_curve(const G2Affine &p) {
    if (p.is_inf()) return true;
    Fq2 b;
#pragma unroll
    for (int i = 0; i < 8; i++) { b.c0.l[i] = FqParams::G2B_C0(i); b.c1.l[i] = FqParams::G2B_C1(i); }
    return p.y.sqr() == p.x.sqr() * p.x + b;
}

}  // namespace lzkp
