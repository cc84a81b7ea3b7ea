// proof_read.cuh — validating readers of ark-serialize's uncompressed points, shared by the verifier (verify.cu) and
// proof rerandomization (rerandomize.cu): what Proof::deserialize_uncompressed (Validate::Yes) checks per point.
// The readers use 128-bit loads: a point's bytes must be 16-byte aligned.
#pragma once
#include "pairing.cuh"

namespace lzkp {
namespace {          // internal to each unit that includes it

__device__ __forceinline__ bool read_fq_canonical(const uint8_t *b, Fq &out, uint32_t &flags) {
    const uint4 *s = reinterpret_cast<const uint4 *>(b);
    uint4 lo = s[0], hi = s[1];
    flags = hi.w >> 30;
    hi.w &= 0x3FFFFFFFu;
    Fq c;
    c.l[0] = lo.x; c.l[1] = lo.y; c.l[2] = lo.z; c.l[3] = lo.w; c.l[4] = hi.x; c.l[5] = hi.y; c.l[6] = hi.z; c.l[7] = hi.w;
    uint32_t d[8];
    Fq m = Fq::modulus();
    bool ok = sub8(d, c.l, m.l) != 0;          // c < q
    out = Fq::from_canonical(c);
    return ok;
}
// ark-serialize uncompressed, validating: canonical coordinates, on the curve (infinity flag accepted)
__device__ __noinline__ bool read_g1_checked(const uint8_t *b, G1Affine &p) {
    uint32_t f0, f1;
    bool ok = read_fq_canonical(b, p.x, f0) & read_fq_canonical(b + 32, p.y, f1);
    if (f0) ok = false;
    if (f1 & 1u) { p = G1Affine::inf(); return ok; }        // infinity flag (bit 6 of the last byte)
    return ok && g1_on_curve(p);
}
__device__ __noinline__ bool read_g2_on_curve(const uint8_t *b, G2Affine &p) {
    uint32_t f0, f1, f2, f3;
    bool ok = read_fq_canonical(b, p.x.c0, f0) & read_fq_canonical(b + 32, p.x.c1, f1) &
              read_fq_canonical(b + 64, p.y.c0, f2) & read_fq_canonical(b + 96, p.y.c1, f3);
    if (f0 | f1 | f2) ok = false;
    if (f3 & 1u) { p = G2Affine::inf(); return ok; }
    return ok && g2_on_curve(p);
}
__device__ __noinline__ bool read_g2_checked(const uint8_t *b, G2Affine &p) {
    if (!read_g2_on_curve(b, p)) return false;
    if (p.is_inf()) return true;
    // subgroup check (deserialize_uncompressed validates it): pairing.cuh g2_subgroup_from_xp, one 63-bit ladder
    const uint32_t x[2] = {kBnXLimbs[0], kBnXLimbs[1]};
    return g2_subgroup_from_xp(p, scalar_mul_window<Fq2, 2>(G2XYZZ::from_affine(p), x));
}

}  // namespace
}  // namespace lzkp
