// prim_ops.h — one dispatch function per family of field / tower / pairing / G2 operations of libzkp_b200/csrc, for
// tests that run the same inputs through a device build (prim_kernels.cu, nvcc for sm_100a: the PTX carry chains and
// the out-of-line Fq2 product) and a host build (tests/host_shim/prim_host.cpp, g++: the portable C++ bodies).
//
// Every family has the form  op(int code, const uint32_t *in, uint32_t *out)  on one fixed-size record per item.
// Field elements are 8 little-endian 32-bit limbs, in Montgomery form unless the operation says otherwise.  Fq2 is
// c0 || c1, Fq6 c0 || c1 || c2, Fq12 c0 || c1 (struct layouts, 32 / 64 / 192 / 384 bytes).
#pragma once
#include <stddef.h>

#include "../../libzkp_b200/csrc/pairing.cuh"

namespace prim {
using namespace lzkp;

enum Family { FAM_FR = 0, FAM_FQ = 1, FAM_FQ2 = 2, FAM_TOWER = 3, FAM_PAIRING = 4, FAM_G2 = 5, FAM_COUNT = 6 };
// words per input / output record of each family
LZ_HD constexpr int in_words(int f) { return f == FAM_TOWER ? 192 : f == FAM_PAIRING ? 200 : 32; }
LZ_HD constexpr int out_words(int f) { return f <= FAM_FQ ? 17 : f == FAM_FQ2 ? 16 : f == FAM_G2 ? 33 : 96; }

template <class T> LZ_HD T load(const uint32_t *p) {
    T v;
    uint32_t *d = reinterpret_cast<uint32_t *>(&v);
    for (int i = 0; i < (int)(sizeof(T) / 4); i++) d[i] = p[i];
    return v;
}
template <class T> LZ_HD void store(uint32_t *p, const T &v) {
    const uint32_t *s = reinterpret_cast<const uint32_t *>(&v);
    for (int i = 0; i < (int)(sizeof(T) / 4); i++) p[i] = s[i];
}

// Fr / Fq.  in = a | b | c | d (8 words each; the wide operations read T = in[0..15] and U = in[16..31]).
// out[0..7] = the result, out[0] = 0 / 1 for a predicate; the wide operations write 16 words and out[16] = carry.
//   0 a*b   1 a.sqr()   2 a+b   3 a-b   4 a.neg()   5 a.dbl()   6 a.inverse()   7 from_canonical(a)   8 a.to_canonical()
//   9 msub(a,b,c,d)   10 gt_canonical(a,b)   11 a.is_zero()   12 a == b
//   13 mul_lazy(a,b)   14 a.sqr_lazy()   15 msub_lazy(a,b,c,d)   16 add_2p(a,b)   17 sub_2p(a,b)   18 a.is_zero_2p()
//   19 a.canonical()   20 reduce_wide(T)   21 reduce_wide_lazy(T)   22 mul_wide(a,b)   23 add16(T,U)   24 sub16(T,U)
template <class F>
LZ_HD void field_op(int code, const uint32_t *in, uint32_t *out) {
    const F a = load<F>(in), b = load<F>(in + 8), c = load<F>(in + 16), d = load<F>(in + 24);
    uint32_t T[16], U[16], W[16];
    for (int i = 0; i < 16; i++) { T[i] = in[i]; U[i] = in[16 + i]; W[i] = 0; }
    for (int i = 0; i < 17; i++) out[i] = 0;
    F r = F::zero();
    switch (code) {
        case 0: r = a * b; break;
        case 1: r = a.sqr(); break;
        case 2: r = a + b; break;
        case 3: r = a - b; break;
        case 4: r = a.neg(); break;
        case 5: r = a.dbl(); break;
        case 6: r = a.inverse(); break;
        case 7: r = F::from_canonical(a); break;
        case 8: r = a.to_canonical(); break;
        case 9: r = F::msub(a, b, c, d); break;
        case 10: r.l[0] = F::gt_canonical(a, b) ? 1u : 0u; break;
        case 11: r.l[0] = a.is_zero() ? 1u : 0u; break;
        case 12: r.l[0] = a == b ? 1u : 0u; break;
        case 13: r = F::mul_lazy(a, b); break;
        case 14: r = a.sqr_lazy(); break;
        case 15: r = F::msub_lazy(a, b, c, d); break;
        case 16: r = F::add_2p(a, b); break;
        case 17: r = F::sub_2p(a, b); break;
        case 18: r.l[0] = a.is_zero_2p() ? 1u : 0u; break;
        case 19: r = a.canonical(); break;
        case 20: r = F::reduce_wide(T); break;
        case 21: r = F::reduce_wide_lazy(T); break;
        case 22: mul_wide(W, a.l, b.l); break;
        case 23: out[16] = add16(W, T, U); break;
        case 24: out[16] = sub16(W, T, U); break;
        default: break;
    }
    if (code >= 22) for (int i = 0; i < 16; i++) out[i] = W[i];
    else store(out, r);
}

// Fq2.  in = a | b (16 words each), out = 16 words.
//   0 a*b (device: fq2_mul_call)   1 a.sqr() (device: fq2_sqr_call)   2 a.inverse()   3 fq2_mul_xi(a)   4 fq2_conj(a)
//   5 fq2_mul_lazy(a,b)   6 a+b   7 a-b
LZ_HD void fq2_op(int code, const uint32_t *in, uint32_t *out) {
    const Fq2 a = load<Fq2>(in), b = load<Fq2>(in + 16);
    Fq2 r = Fq2::zero();
    switch (code) {
        case 0: r = a * b; break;
        case 1: r = a.sqr(); break;
        case 2: r = a.inverse(); break;
        case 3: r = fq2_mul_xi(a); break;
        case 4: r = fq2_conj(a); break;
        case 5: r = fq2_mul_lazy(a, b); break;
        case 6: r = a + b; break;
        default: r = a - b; break;
    }
    store(out, r);
}

// pairing.cuh's tower.  in = a | b (Fq12, 96 words each; the Fq6 operations read the c0 halves, f12_mul_by_034 reads
// (c0, c3, c4) = the first three Fq2 of b), out = 96 words (an Fq6 result in the first 48).
//   0 f6_mul   1 f6_inv   2 f6_mul_v   3 f12_mul   4 f12_sqr   5 f12_inv   6 f12_conj   7 f12_frob2   8 f12_frob_odd<1>
//   9 f12_frob_odd<3>   10 f12_mul_by_034   11 f12_cyclo_sqr   12 f12_exp_neg_x   13 final_exponentiation
LZ_HD void tower_op(int code, const uint32_t *in, uint32_t *out) {
    const Fq12 a = load<Fq12>(in), b = load<Fq12>(in + 96);
    Fq12 r;
    f12_one(r);
    switch (code) {
        case 0: f6_mul(r.c0, a.c0, b.c0); break;
        case 1: f6_inv(r.c0, a.c0); break;
        case 2: f6_mul_v(r.c0, a.c0); break;
        case 3: f12_mul(r, a, b); break;
        case 4: f12_sqr(r, a); break;
        case 5: f12_inv(r, a); break;
        case 6: f12_conj(r, a); break;
        case 7: f12_frob2(r, a); break;
        case 8: f12_frob_odd<1>(r, a); break;
        case 9: f12_frob_odd<3>(r, a); break;
        case 10: r = a; f12_mul_by_034(r, b.c0.c0, b.c0.c1, b.c0.c2); break;
        case 11: f12_cyclo_sqr(r, a); break;
        case 12: f12_exp_neg_x(r, a); break;
        default: final_exponentiation(r, a); break;
    }
    store(out, r);
}

// multi_miller_loop<N>.  in[0] = N (1..4), in[1] = skip mask (bit k: pair k skipped), in[8 + 48 k ..] = pair k: P (G1
// affine, 16 words) then Q (G2 affine, 32 words).  out = the Miller value (code 0) or its final exponentiation (code 1).
template <int N>
LZ_HD void miller_n(Fq12 &f, const uint32_t *in) {
    G1Affine P[N];
    G2Affine Q[N];
    bool skip[N];
    for (int k = 0; k < N; k++) {
        P[k] = load<G1Affine>(in + 8 + 48 * k);
        Q[k] = load<G2Affine>(in + 8 + 48 * k + 16);
        skip[k] = ((in[1] >> k) & 1u) != 0;
    }
    multi_miller_loop<N>(f, P, Q, skip);
}
LZ_HD void pairing_op(int code, const uint32_t *in, uint32_t *out) {
    Fq12 f;
    switch (in[0]) {
        case 1: miller_n<1>(f, in); break;
        case 2: miller_n<2>(f, in); break;
        case 3: miller_n<3>(f, in); break;
        default: miller_n<4>(f, in); break;
    }
    if (code == 1) { Fq12 e; final_exponentiation(e, f); f = e; }
    store(out, f);
}

// The r-torsion test of a twist point exactly as verify.cu's read_g2_checked runs it (lane per proof): [x] P by
// scalar_mul_window<Fq2, 2>, then g2_subgroup_from_xp.  in = P (G2 affine, not infinity), out[0..31] = [x] P in affine
// form (all zero: infinity), out[32] = 1 when P passes.
LZ_HD void g2_op(int, const uint32_t *in, uint32_t *out) {
    const G2Affine p = load<G2Affine>(in);
    const uint32_t x[2] = {kBnXLimbs[0], kBnXLimbs[1]};
    const G2XYZZ xp = scalar_mul_window<Fq2, 2>(G2XYZZ::from_affine(p), x);
    store(out, xp.to_affine());
    out[32] = g2_subgroup_from_xp(p, xp) ? 1u : 0u;
}

LZ_HD void run(int family, int code, const uint32_t *in, uint32_t *out) {
    switch (family) {
        case FAM_FR: field_op<Fr>(code, in, out); break;
        case FAM_FQ: field_op<Fq>(code, in, out); break;
        case FAM_FQ2: fq2_op(code, in, out); break;
        case FAM_TOWER: tower_op(code, in, out); break;
        case FAM_PAIRING: pairing_op(code, in, out); break;
        default: g2_op(code, in, out); break;
    }
}

}  // namespace prim
