// dev_util.cuh — small device helpers shared by every translation unit of the engine.
#pragma once
#include "ec.cuh"

namespace lzkp {

// ---------------------------------------------------------------- load / store
template <class T>
__device__ __forceinline__ T ldg_vec(const T *p) {          // read-only path, 128-bit pieces
    static_assert(sizeof(T) % 16 == 0, "vector load");
    T r;
    const uint4 *s = reinterpret_cast<const uint4 *>(p);
    uint4 *d = reinterpret_cast<uint4 *>(&r);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = __ldg(s + i);
    return r;
}
template <class T>
__device__ __forceinline__ T ld_vec(const T *p) {
    T r;
    const uint4 *s = reinterpret_cast<const uint4 *>(p);
    uint4 *d = reinterpret_cast<uint4 *>(&r);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = s[i];
    return r;
}
template <class T>
__device__ __forceinline__ void st_vec(T *p, const T &v) {
    uint4 *d = reinterpret_cast<uint4 *>(p);
    const uint4 *s = reinterpret_cast<const uint4 *>(&v);
#pragma unroll
    for (int i = 0; i < (int)(sizeof(T) / 16); i++) d[i] = s[i];
}
__device__ __forceinline__ Fr fr_from_u64(uint64_t v) {
    Fr c = Fr::zero();
    c.l[0] = (uint32_t)v;
    c.l[1] = (uint32_t)(v >> 32);
    return c;
}
__device__ __forceinline__ bool fr_is_canonical(const Fr &a) {   // a < r ?
    uint32_t d[8];
    Fr m = Fr::modulus();
    return sub8(d, a.l, m.l) != 0;
}
__host__ __device__ __forceinline__ uint32_t bitrev(uint32_t x, uint32_t bits) {
#ifdef __CUDA_ARCH__
    return __brev(x) >> (32 - bits);
#else
    uint32_t r = 0;
    for (uint32_t i = 0; i < bits; i++) r |= ((x >> i) & 1u) << (bits - 1 - i);
    return r;
#endif
}


template <class F>
__device__ __forceinline__ Affine<F> gather_point(const Affine<F> *table, uint32_t N, uint32_t tbl_unit, int d) {
    int mag = d < 0 ? -d : d;
    Affine<F> pt = ldg_vec(table + (size_t)tbl_unit * N + (uint32_t)(mag - 1));
    if (d < 0) pt.y = pt.y.neg();
    return pt;
}

// ---------------------------------------------------------------- ark-serialize writers
__device__ __forceinline__ void put_fq(uint8_t *out, const Fq &canon, uint32_t flags) {
    uint4 *o = reinterpret_cast<uint4 *>(out);
    o[0] = make_uint4(canon.l[0], canon.l[1], canon.l[2], canon.l[3]);
    o[1] = make_uint4(canon.l[4], canon.l[5], canon.l[6], canon.l[7] | (flags << 24));
}
// ark-serialize SW-affine uncompressed: x || y, flags in the top bits of the last byte:
// 0x80 = y > -y (canonical integer order), 0x40 = infinity (then x = y = 0).
__device__ __forceinline__ void write_g1(uint8_t *out, const G1Affine &p) {
    if (p.is_inf()) { put_fq(out, Fq::zero(), 0); put_fq(out + 32, Fq::zero(), 0x40); return; }
    Fq y = p.y.to_canonical(), ny = p.y.neg().to_canonical();
    put_fq(out, p.x.to_canonical(), 0);
    put_fq(out + 32, y, Fq::gt_canonical(y, ny) ? 0x80u : 0u);
}
__device__ __forceinline__ void write_g2(uint8_t *out, const G2Affine &p) {
    if (p.is_inf()) {
        put_fq(out, Fq::zero(), 0); put_fq(out + 32, Fq::zero(), 0); put_fq(out + 64, Fq::zero(), 0);
        put_fq(out + 96, Fq::zero(), 0x40);
        return;
    }
    Fq y0 = p.y.c0.to_canonical(), y1 = p.y.c1.to_canonical();
    Fq n0 = p.y.c0.neg().to_canonical(), n1 = p.y.c1.neg().to_canonical();
    bool neg = (y1 == n1) ? Fq::gt_canonical(y0, n0) : Fq::gt_canonical(y1, n1);   // c1 first, then c0
    put_fq(out, p.x.c0.to_canonical(), 0);
    put_fq(out + 32, p.x.c1.to_canonical(), 0);
    put_fq(out + 64, y0, 0);
    put_fq(out + 96, y1, neg ? 0x80u : 0u);
}

}  // namespace lzkp
