// prim_kernels.cu — device build of prim_ops.h (one item per thread) and warp kernels for coop.cuh's entry points
// (one item per warp).  Built by the tests with the library's nvcc flags, without LZKP_FQ2_INLINE, so the Fq2 products
// are the out-of-line fq2_mul_call / fq2_sqr_call the engine runs.  Every launcher takes device pointers, an item count
// and a stream, and returns cudaGetLastError().
#include <cuda_runtime.h>

#include "../../libzkp_b200/csrc/coop.cuh"
#include "prim_ops.h"

using namespace lzkp;

namespace {

template <int FAM>
__device__ void run_family(int code, const uint32_t *in, uint32_t *out) {
    if (FAM == prim::FAM_FR) prim::field_op<Fr>(code, in, out);
    else if (FAM == prim::FAM_FQ) prim::field_op<Fq>(code, in, out);
    else if (FAM == prim::FAM_FQ2) prim::fq2_op(code, in, out);
    else if (FAM == prim::FAM_TOWER) prim::tower_op(code, in, out);
    else if (FAM == prim::FAM_PAIRING) prim::pairing_op(code, in, out);
    else if (FAM == prim::FAM_G1_CURVE) prim::curve_op<Fq>(code, in, out);
    else if (FAM == prim::FAM_G2_CURVE) prim::curve_op<Fq2>(code, in, out);
    else if (FAM == prim::FAM_SCALAR) prim::scalar_op(code, in, out);
    else prim::g2_op(code, in, out);
}
// one kernel per family, so that the field operations are not compiled beside the pairing
template <int FAM>
__global__ void k_prim(int code, const uint32_t *__restrict__ in, uint32_t *__restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    run_family<FAM>(code, in + (size_t)i * prim::in_words(FAM), out + (size_t)i * prim::out_words(FAM));
}

// coop::fq_half on one Fq per thread (a plain 8-word value in, a plain value out)
__global__ void k_fq_half(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, int n) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    prim::store(out + 8 * i, coop::fq_half(prim::load<Fq>(in + 8 * i)));
}

// coop::f12_mul<SPARSE> on one item per warp.  Item: a (96 words) | b (96; SPARSE: a line l0 | l1 | l2 in the first 48)
// | sa (16) | sb (16).  mode 0: r separate; 1: r aliases a; 2: r aliases b; 3: a squaring (b is a).  out: r (96) | so (16),
// so = sa * sb computed by the lanes >= 18 alongside the product.
constexpr int kMulIn = 96 + 96 + 16 + 16, kMulOut = 96 + 16;
struct MulSmem {
    Fq2 a[6], b[6], r[6], sa, sb, so;
    coop::Scratch s;
};
template <bool SPARSE>
__global__ void k_coop_f12_mul(int mode, const uint32_t *__restrict__ in, uint32_t *__restrict__ out, int n) {
    __shared__ MulSmem sm[4];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, item = blockIdx.x * 4 + w;
    if (item >= n) return;                                   // whole warps leave together
    MulSmem &m = sm[w];
    const uint32_t *src = in + (size_t)item * kMulIn;
    if (lane < 6) {
        m.a[lane] = prim::load<Fq2>(src + 16 * lane);
        m.b[lane] = prim::load<Fq2>(src + 96 + 16 * lane);
        m.r[lane] = Fq2::zero();
    }
    if (lane == 0) {
        m.sa = prim::load<Fq2>(src + 192);
        m.sb = prim::load<Fq2>(src + 208);
        m.so = Fq2::zero();
        m.s.P[18] = Fq2::zero();                             // the zero slot (scratch_init)
    }
    __syncwarp();
    const Fq2 *a = m.a, *b = mode == 3 ? m.a : m.b;
    Fq2 *r = mode == 1 ? m.a : mode == 2 ? m.b : m.r;
    coop::f12_mul<SPARSE>(r, a, b, &m.s, lane >= 18 ? &m.sa : nullptr, lane >= 18 ? &m.sb : nullptr,
                          lane >= 18 ? &m.so : nullptr);
    uint32_t *dst = out + (size_t)item * kMulOut;
    if (lane < 6) prim::store(dst + 16 * lane, r[lane]);
    if (lane == 0) prim::store(dst + 96, m.so);
}

// coop::f12_frob<K> (K = 1, 2, 3) and coop::f12_conj (K = 0) on one Fq12 per warp, in place
template <int K>
__global__ void k_coop_f12_map(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, int n) {
    __shared__ Fq2 sm[4][6];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, item = blockIdx.x * 4 + w;
    if (item >= n) return;
    if (lane < 6) sm[w][lane] = prim::load<Fq2>(in + (size_t)item * 96 + 16 * lane);
    __syncwarp();
    if (K == 0) coop::f12_conj(sm[w], sm[w]);
    else coop::f12_frob<K == 0 ? 1 : K>(sm[w], sm[w]);
    if (lane < 6) prim::store(out + (size_t)item * 96 + 16 * lane, sm[w][lane]);
}

// coop::g2_in_subgroup on one twist point (32 words, not infinity) per warp; out = 1 when it passes
__global__ void k_coop_subgroup(const uint32_t *__restrict__ in, uint32_t *__restrict__ out, int n) {
    __shared__ coop::LadderState sm[4];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, item = blockIdx.x * 4 + w;
    if (item >= n) return;
    const bool ok = coop::g2_in_subgroup(&sm[w], prim::load<G2Affine>(in + (size_t)item * 32));
    if (lane == 0) out[item] = ok ? 1u : 0u;
}

// The ladder of coop::g2_in_subgroup from a crafted state.  Item: X | Y | ZZ | ZZZ | bx | by (16 words each) | add.
// mode 0: one coop::ladder_step(st, add);  mode 1: coop::ladder_madd alone.  out: X | Y | ZZ | ZZZ (64) | madd's result.
constexpr int kLadIn = 97, kLadOut = 65;
__global__ void k_coop_ladder(int mode, const uint32_t *__restrict__ in, uint32_t *__restrict__ out, int n) {
    __shared__ coop::LadderState sm[4];
    const int w = threadIdx.x >> 5, lane = threadIdx.x & 31, item = blockIdx.x * 4 + w;
    if (item >= n) return;
    coop::LadderState *st = &sm[w];
    const uint32_t *src = in + (size_t)item * kLadIn;
    if (lane == 0) {
        st->X = prim::load<Fq2>(src); st->Y = prim::load<Fq2>(src + 16);
        st->ZZ = prim::load<Fq2>(src + 32); st->ZZZ = prim::load<Fq2>(src + 48);
        st->bx = prim::load<Fq2>(src + 64); st->by = prim::load<Fq2>(src + 80);
    }
    __syncwarp();
    bool done = true;
    if (mode == 0) coop::ladder_step(st, src[96] != 0);
    else done = coop::ladder_madd(st);
    uint32_t *dst = out + (size_t)item * kLadOut;
    if (lane == 0) {
        prim::store(dst, st->X); prim::store(dst + 16, st->Y); prim::store(dst + 32, st->ZZ); prim::store(dst + 48, st->ZZZ);
        dst[64] = done ? 1u : 0u;
    }
}

template <int FAM>
cudaError_t launch_prim(int code, const void *in, void *out, int n, cudaStream_t st) {
    k_prim<FAM><<<(n + 127) / 128, 128, 0, st>>>(code, static_cast<const uint32_t *>(in), static_cast<uint32_t *>(out), n);
    return cudaGetLastError();
}

}  // namespace

extern "C" {

int prim_words(int family, int *in_words, int *out_words) {
    if (family < 0 || family >= prim::FAM_COUNT) return -1;
    *in_words = prim::in_words(family);
    *out_words = prim::out_words(family);
    return 0;
}

// prim_ops.h family `family`, operation `code`, on n records
int prim_launch(int family, int code, const void *in, void *out, int n, cudaStream_t st) {
    if (n <= 0) return (int)cudaGetLastError();
    switch (family) {
        case prim::FAM_FR: return (int)launch_prim<prim::FAM_FR>(code, in, out, n, st);
        case prim::FAM_FQ: return (int)launch_prim<prim::FAM_FQ>(code, in, out, n, st);
        case prim::FAM_FQ2: return (int)launch_prim<prim::FAM_FQ2>(code, in, out, n, st);
        case prim::FAM_TOWER: return (int)launch_prim<prim::FAM_TOWER>(code, in, out, n, st);
        case prim::FAM_PAIRING: return (int)launch_prim<prim::FAM_PAIRING>(code, in, out, n, st);
        case prim::FAM_G2: return (int)launch_prim<prim::FAM_G2>(code, in, out, n, st);
        case prim::FAM_G1_CURVE: return (int)launch_prim<prim::FAM_G1_CURVE>(code, in, out, n, st);
        case prim::FAM_G2_CURVE: return (int)launch_prim<prim::FAM_G2_CURVE>(code, in, out, n, st);
        case prim::FAM_SCALAR: return (int)launch_prim<prim::FAM_SCALAR>(code, in, out, n, st);
        default: return (int)cudaErrorInvalidValue;
    }
}

int prim_fq_half(const void *in, void *out, int n, cudaStream_t st) {
    if (n > 0) k_fq_half<<<(n + 127) / 128, 128, 0, st>>>(static_cast<const uint32_t *>(in), static_cast<uint32_t *>(out), n);
    return (int)cudaGetLastError();
}

int prim_coop_f12_mul(int sparse, int mode, const void *in, void *out, int n, cudaStream_t st) {
    const dim3 grid((n + 3) / 4), block(128);
    if (n <= 0) return (int)cudaGetLastError();
    if (sparse) k_coop_f12_mul<true><<<grid, block, 0, st>>>(mode, static_cast<const uint32_t *>(in), static_cast<uint32_t *>(out), n);
    else k_coop_f12_mul<false><<<grid, block, 0, st>>>(mode, static_cast<const uint32_t *>(in), static_cast<uint32_t *>(out), n);
    return (int)cudaGetLastError();
}

// k = 0: f12_conj, 1 / 2 / 3: f12_frob<k>
int prim_coop_f12_map(int k, const void *in, void *out, int n, cudaStream_t st) {
    const dim3 grid((n + 3) / 4), block(128);
    const uint32_t *i = static_cast<const uint32_t *>(in);
    uint32_t *o = static_cast<uint32_t *>(out);
    if (n <= 0) return (int)cudaGetLastError();
    switch (k) {
        case 0: k_coop_f12_map<0><<<grid, block, 0, st>>>(i, o, n); break;
        case 1: k_coop_f12_map<1><<<grid, block, 0, st>>>(i, o, n); break;
        case 2: k_coop_f12_map<2><<<grid, block, 0, st>>>(i, o, n); break;
        case 3: k_coop_f12_map<3><<<grid, block, 0, st>>>(i, o, n); break;
        default: return (int)cudaErrorInvalidValue;
    }
    return (int)cudaGetLastError();
}

int prim_coop_subgroup(const void *in, void *out, int n, cudaStream_t st) {
    if (n > 0) k_coop_subgroup<<<(n + 3) / 4, 128, 0, st>>>(static_cast<const uint32_t *>(in), static_cast<uint32_t *>(out), n);
    return (int)cudaGetLastError();
}

int prim_coop_ladder(int mode, const void *in, void *out, int n, cudaStream_t st) {
    if (n > 0) k_coop_ladder<<<(n + 3) / 4, 128, 0, st>>>(mode, static_cast<const uint32_t *>(in), static_cast<uint32_t *>(out), n);
    return (int)cudaGetLastError();
}

}  // extern "C"
