// Host build of field.cuh's redundant-form operations ([0, 2p) values) and ec.cuh's madd_lazy, checked against
// Python big integers and the canonical madd by tests/test_lazy_field_host.py.  Field elements are 8 little-endian
// 32-bit limbs (32 B), XYZZ points x || y || zz || zzz (128 B), affine points x || y (64 B).
#include "../../libzkp_b200/csrc/ec.cuh"
#include <cstring>
using namespace lzkp;
template <class T> static T ld(const uint8_t *p) { T v; std::memcpy(&v, p, sizeof(T)); return v; }
template <class T> static void st(uint8_t *p, const T &v) { std::memcpy(p, &v, sizeof(T)); }
static_assert(sizeof(Fq) == 32 && sizeof(G1XYZZ) == 128 && sizeof(G1Affine) == 64, "packed layouts");
extern "C" {
// op: 0 mul_lazy, 1 sqr_lazy, 2 sub_2p, 3 add_2p, 4 canonical, 5 is_zero_2p (o[0] = 0 / 1)
void fq_lazy_op(int op, const uint8_t *a, const uint8_t *b, uint8_t *o) {
    const Fq x = ld<Fq>(a), y = ld<Fq>(b);
    Fq r = Fq::zero();
    switch (op) {
        case 0: r = Fq::mul_lazy(x, y); break;
        case 1: r = x.sqr_lazy(); break;
        case 2: r = Fq::sub_2p(x, y); break;
        case 3: r = Fq::add_2p(x, y); break;
        case 4: r = x.canonical(); break;
        default: r.l[0] = x.is_zero_2p() ? 1u : 0u;
    }
    st(o, r);
}
void fq_msub_lazy_host(const uint8_t *a, const uint8_t *b, const uint8_t *c, const uint8_t *d, uint8_t *o) {
    st(o, Fq::msub_lazy(ld<Fq>(a), ld<Fq>(b), ld<Fq>(c), ld<Fq>(d)));
}
void fq_reduce_wide_lazy_host(const uint8_t *t64, uint8_t *o) {
    uint32_t T[16];
    std::memcpy(T, t64, 64);
    st(o, Fq::reduce_wide_lazy(T));
}
// acc += p: lazy != 0 runs madd_lazy (result left in the redundant form), else the canonical madd
void g1_madd_host(int lazy, uint8_t *acc, const uint8_t *p) {
    G1XYZZ a = ld<G1XYZZ>(acc);
    if (lazy) a.madd_lazy(ld<G1Affine>(p)); else a.madd(ld<G1Affine>(p));
    st(acc, a);
}
void g1_canonical_host(uint8_t *acc) { st(acc, ld<G1XYZZ>(acc).canonical()); }
}
