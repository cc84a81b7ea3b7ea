// rerandomize.cu — Groth16::<Bn254>::rerandomize_proof (ark-groth16 prover.rs; BKSV20, ePrint 2020/811, Thm. 3), batched.
//
// A valid proof (A, B, C) of a statement becomes a fresh proof of the same statement, statistically indistinguishable
// from a newly generated one, with the verifying key's delta alone (no proving key, no witness):
//     A' = r1^-1 A,   B' = r1 B + (r1 r2) delta,   C' = C + r2 A        (r1, r2 non-zero, supplied by the caller)
// Input validation is Proof::deserialize_uncompressed's (validating): canonical coordinates, legal flags, A, B, C on
// their curves (infinity accepted), B in the r-torsion (proof_read.cuh).  The subgroup check is also what makes the psi
// split below correct: psi acts as [lambda_psi] only on the r-torsion.
//
// Three launches, one thread per proof each: the checks (k_rerandomize_check), B' (k_rerandomize_g2), A' and C'
// (k_rerandomize_g1).  One kernel doing all three kept values live across calls into G2 code that uses all 255
// registers, and ptxas spilled them; split, no kernel keeps anything but its row across a call and none spills.
// Per proof, in Fq products (estimated from the formulas; an Fq2 product is 3, an Fq2 squaring 2):
//   * B in the r-torsion: one 63-bit G2 ladder                                                            ~2.3 k
//   * r1 B + (r1 r2) delta: both scalars psi-split (ec.cuh psi_split) into 127-bit halves, ONE joint signed-window
//     ladder over B, psi(B), delta, psi(delta): 132 G2 doublings, <= 132 G2 additions, tables of B and delta  ~9.0 k
//   * r1^-1 A and r2 A: r1^-1 by the binary inversion in Fr, both scalars GLV-split (ec.cuh glv_split), two joint
//     ladders over A, phi(A) sharing one table                                                              ~2.6 k
//   * three conversions to affine (three inversions)                                                        ~0.3 k
// delta is read from the key (eng::vk_delta_neg, negated for free); nothing is built for it at key load, no per-key
// scratch is written, so concurrent calls on one key need no ordering.
#include <algorithm>
#include <string>

#include "common.h"
#include "dev_util.cuh"
#include "proof_read.cuh"
#include "verify.h"

namespace lzkp {
namespace {

constexpr int kThreads = 64;
constexpr size_t kChunk = size_t(1) << 20;       // proofs per pass of lzkp_proofs_rerandomize: 321 MB of device scratch

// k * P through the GLV split of k (the pattern of kernels_prove.cuh glv_half): T = tables of P and phi(P); when the
// split does not fit 128 bits (never observed) the plain 254-bit ladder.
__device__ __forceinline__ G1XYZZ glv_mul(const G1XYZZ (&T)[2][8], const Fr &k) {
    const GlvSplit sp = glv_split(k);
    if (!sp.ok) return scalar_mul(T[0][0], k);
    const uint32_t kk[2][4] = {{sp.k1[0], sp.k1[1], sp.k1[2], sp.k1[3]}, {sp.k2[0], sp.k2[1], sp.k2[2], sp.k2[3]}};
    return joint_mul_u128<Fq, 2>(T, kk, (sp.neg1 ? 1u : 0u) | (sp.neg2 ? 2u : 0u));
}

// B' = r1 B + (r1 r2) delta = k0(r1) B + k1(r1) psi(B) + k0(r1 r2) delta + k1(r1 r2) psi(delta), written to out.
// (Values live across calls are kept few: the factors are read here, not passed in registers.)
__device__ __noinline__ void g2_rerandomize(const G2Affine &B, const G2Affine *delta_neg, const Fr *r1p, const Fr *r2p, uint8_t *out) {
    uint32_t k[4][4];
    {
        const Fr r1 = ld_vec(r1p), r12 = Fr::from_canonical(r1) * ld_vec(r2p);     // (r1 R)(r2) R^-1 = r1 r2, canonical
        psi_split(r1.l, k[0], k[1]);
        psi_split(r12.l, k[2], k[3]);
    }
    G2XYZZ T[4][8];
    {
        G2Affine delta = ldg_vec(delta_neg);
        delta.y = delta.y.neg();
        window_table(T[2], G2XYZZ::from_affine(delta));
    }
    window_table(T[0], G2XYZZ::from_affine(B));
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        T[1][i] = g2_psi(T[0][i]);
        T[3][i] = g2_psi(T[2][i]);
    }
    write_g2(out, joint_mul_u128<Fq2, 4>(T, k, 0u).to_affine());
}

// A' = r1^-1 A and C' = C + r2 A, written to out and out + 192
__device__ __noinline__ void g1_rerandomize(const G1Affine &A, const G1Affine &C, const Fr *r1p, const Fr *r2p, uint8_t *out) {
    G1XYZZ T[2][8];
    window_table(T[0], G1XYZZ::from_affine(A));
    Fq beta;
#pragma unroll
    for (int i = 0; i < 8; i++) beta.l[i] = FqParams::BETA(i);
#pragma unroll 1
    for (int i = 0; i < 8; i++) {
        T[1][i] = T[0][i];
        T[1][i].x = T[1][i].x * beta;                    // phi(x, y) = (beta x, y); x = X / ZZ
    }
    write_g1(out, glv_mul(T, Fr::from_canonical(ld_vec(r1p)).inverse().to_canonical()).to_affine());
    G1XYZZ Cn = glv_mul(T, ld_vec(r2p));
    Cn.madd_cold(C);
    write_g1(out + 192, Cn.to_affine());
}

// Three passes over the rows, one thread per row each.  k_rerandomize_check decides every row (ok, and 0xFF over a row
// that fails); the two others skip failing rows and write disjoint parts of a passing one: B' (bytes 64..191) and
// A', C' (bytes 0..63, 192..255), each reading only the part it replaces, so out may be proofs.
__global__ void __launch_bounds__(kThreads) k_rerandomize_check(const uint8_t *proofs, const Fr *__restrict__ r1s,
                                                                const Fr *__restrict__ r2s, uint32_t n, uint8_t *out,
                                                                uint8_t *__restrict__ ok) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const uint8_t *pb = proofs + (size_t)i * 256;
    bool good;
    {
        const Fr r1 = ld_vec(r1s + i), r2 = ld_vec(r2s + i);
        good = fr_is_canonical(r1) && fr_is_canonical(r2) && !r1.is_zero() && !r2.is_zero();
    }
    // both flags on a y coordinate are illegal in ark-serialize (SWFlags); the shared readers take them for infinity
    good = good && (pb[63] & 0xC0) != 0xC0 && (pb[191] & 0xC0) != 0xC0 && (pb[255] & 0xC0) != 0xC0;
    {
        G1Affine P;
        good = read_g1_checked(pb, P) && good;
        good = read_g1_checked(pb + 192, P) && good;
    }
    {
        G2Affine Q;
        good = good && read_g2_checked(pb + 64, Q);
    }
    ok[i] = good ? 1 : 0;
    if (good) return;
    uint4 *o = reinterpret_cast<uint4 *>(out + (size_t)i * 256);
#pragma unroll
    for (int w = 0; w < 16; w++) o[w] = make_uint4(~0u, ~0u, ~0u, ~0u);
}
__global__ void __launch_bounds__(kThreads) k_rerandomize_g2(const G2Affine *__restrict__ delta_neg, const uint8_t *proofs,
                                                             const Fr *__restrict__ r1s, const Fr *__restrict__ r2s, uint32_t n,
                                                             uint8_t *out, const uint8_t *__restrict__ ok) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !ok[i]) return;
    G2Affine B;
    read_g2_on_curve(proofs + (size_t)i * 256 + 64, B);
    g2_rerandomize(B, delta_neg, r1s + i, r2s + i, out + (size_t)i * 256 + 64);
}
__global__ void __launch_bounds__(kThreads) k_rerandomize_g1(const uint8_t *proofs, const Fr *__restrict__ r1s,
                                                             const Fr *__restrict__ r2s, uint32_t n, uint8_t *out,
                                                             const uint8_t *__restrict__ ok) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n || !ok[i]) return;
    G1Affine A, C;
    read_g1_checked(proofs + (size_t)i * 256, A);
    read_g1_checked(proofs + (size_t)i * 256 + 192, C);
    g1_rerandomize(A, C, r1s + i, r2s + i, out + (size_t)i * 256);
}

int enqueue_rerandomize(eng::VerifyingKeyDev *V, size_t n, const uint8_t *proofs, const uint8_t *r1, const uint8_t *r2,
                        uint8_t *out, uint8_t *ok, cudaStream_t st) {
    const unsigned grid = (unsigned)((n + kThreads - 1) / kThreads);
    const Fr *f1 = reinterpret_cast<const Fr *>(r1), *f2 = reinterpret_cast<const Fr *>(r2);
    LAUNCH(k_rerandomize_check, grid, kThreads, 0, st, proofs, f1, f2, (uint32_t)n, out, ok);
    LAUNCH(k_rerandomize_g2, grid, kThreads, 0, st, eng::vk_delta_neg(V), proofs, f1, f2, (uint32_t)n, out, ok);
    LAUNCH(k_rerandomize_g1, grid, kThreads, 0, st, proofs, f1, f2, (uint32_t)n, out, ok);
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

}  // namespace

namespace eng {

int proofs_rerandomize(VerifyingKeyDev *V, size_t n, const uint8_t *proofs, const uint8_t *r1, const uint8_t *r2, uint8_t *proofs_out,
                       uint8_t *ok_out) {
    if (n == 0) return LZKP_OK;
    const size_t chunk = std::min(n, kChunk);
    DBuf d_p, d_r1, d_r2, d_ok;
    TRY(d_p.alloc(chunk * 256));
    TRY(d_r1.alloc(chunk * 32));
    TRY(d_r2.alloc(chunk * 32));
    TRY(d_ok.alloc(chunk));
    for (size_t off = 0; off < n; off += chunk) {
        const size_t m = std::min(chunk, n - off);
        CUDA_TRY(cudaMemcpy(d_p.p, proofs + off * 256, m * 256, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d_r1.p, r1 + off * 32, m * 32, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(d_r2.p, r2 + off * 32, m * 32, cudaMemcpyHostToDevice));
        TRY(enqueue_rerandomize(V, m, d_p.as<uint8_t>(), d_r1.as<uint8_t>(), d_r2.as<uint8_t>(), d_p.as<uint8_t>(), d_ok.as<uint8_t>(), 0));
        CUDA_TRY(cudaMemcpy(proofs_out + off * 256, d_p.p, m * 256, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(ok_out + off, d_ok.p, m, cudaMemcpyDeviceToHost));
    }
    return LZKP_OK;
}

int proofs_rerandomize_device(VerifyingKeyDev *V, size_t n, const uint8_t *d_proofs, const uint8_t *d_r1, const uint8_t *d_r2,
                              uint8_t *d_proofs_out, uint8_t *d_ok, cudaStream_t st) {
    if (n == 0) return LZKP_OK;
    if (n > 0xFFFFFFFFull) return fail(LZKP_E_INVALID, "lzkp_proofs_rerandomize_device: more than 2^32 - 1 proofs");
    // the kernel reads and writes proofs and factors with 128-bit accesses
    if ((reinterpret_cast<uintptr_t>(d_proofs) | reinterpret_cast<uintptr_t>(d_r1) | reinterpret_cast<uintptr_t>(d_r2) |
         reinterpret_cast<uintptr_t>(d_proofs_out)) & 15)
        return fail(LZKP_E_INVALID, "lzkp_proofs_rerandomize_device: proofs and factors must be 16-byte aligned");
    TRY(check_device_buffer(V, d_proofs, "proofs"));
    TRY(check_device_buffer(V, d_r1, "r1"));
    TRY(check_device_buffer(V, d_r2, "r2"));
    TRY(check_device_buffer(V, d_proofs_out, "rerandomized proofs"));
    TRY(check_device_buffer(V, d_ok, "ok"));
    return enqueue_rerandomize(V, n, d_proofs, d_r1, d_r2, d_proofs_out, d_ok, st);
}

}  // namespace eng
}  // namespace lzkp
