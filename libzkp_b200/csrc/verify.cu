// verify.cu — batched Groth16/BN254 verification on the device (lzkp_vk_load / lzkp_verify_batch; SURVEY.md §8f-3).
//
// Replaces, for batches, what the reference does one proof at a time on the CPU (src/backend/snark.rs:377-401 and
// :455-495): Proof::deserialize_uncompressed (validating), Groth16::process_vk — recomputed there on EVERY call,
// here once per key at lzkp_vk_load —, the public-input accumulation and verify_with_processed_vk:
//     e(A, B) * e(vk_x, -gamma) * e(C, -delta) == e(alpha, beta),   vk_x = gamma_abc[0] + sum_i x_i gamma_abc[i+1].
// Three forms, chosen by the size of the call, with the same decisions (tests/test_gpu_verify.py):
//   * up to three proofs per SM: one proof per CTA, warps and lanes share the pairing's arithmetic (k_verify_coop, coop.cuh);
//   * larger calls: random-linear-combination form - per proof ONE Miller loop e(rho A, B), the format / curve / subgroup
//     checks and rho C (k_rlc_prepare: four role warps per 32 proofs; k_rlc_prepare_seq beyond one resident wave), per group
//     of 64 one cooperative combined check (k_rlc_scalars, k_rlc_inputs2, k_rlc_tail_coop); a failing group is re-verified
//     proof by proof;
//   * one proof per lane (k_verify4): keys without the latency form's tables, no OS entropy, large failing ranges.
// Keys above kCoopScanMax public inputs take the same forms; there vk_x of each proof comes from its own kernel (k_vkx)
// and the combined form's scalar sums from k_rlc_input_sums.
// lzkp_verify_batch_device runs the same stages on the caller's stream from device buffers; its coefficients come from
// k_rlc_rho and its failing groups are listed by k_rlc_failed and re-verified by the Listed instantiations of the forms.
#include <cstddef>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "chacha20.cuh"
#include "dev_util.cuh"
#include "host_util.h"
#include "coop.cuh"
#include "pairing.cuh"
#include "proof_read.cuh"
#include "verify.h"

namespace lzkp {

namespace {

struct VkDev {
    G1Affine alpha;
    G2Affine beta, gamma_neg, delta_neg;
    Fq12 alpha_beta;                 // e(alpha, beta), filled by k_vk_prepare
};

// e(alpha, beta) once per key (what process_vk precomputes)
// What VerifyingKey::deserialize_uncompressed (Validate::Yes, snark.rs:66) checks: every point of the key is on its
// curve and, in G2, in the r-torsion.  One thread per point of the raw ark-serialize bytes.
__global__ void k_vk_validate(const uint8_t *vk_bytes, uint32_t n_abc, int *bad) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= 4 + n_abc) return;
    // the readers use 128-bit loads; offsets inside a key (456 + 64 i) are only 8-byte aligned: stage the point
    __align__(16) uint8_t buf[128];
    const uint8_t *src = i == 0 ? vk_bytes : i < 4 ? vk_bytes + 64 + 128 * (i - 1) : vk_bytes + 456 + 64 * (size_t)(i - 4);
    const uint32_t len = (i >= 1 && i < 4) ? 128 : 64;
    for (uint32_t b = 0; b < len; b++) buf[b] = src[b];
    bool ok;
    if (len == 128) { G2Affine q; ok = read_g2_checked(buf, q); }
    else { G1Affine p; ok = read_g1_checked(buf, p); }
    if (!ok) atomicAdd(bad, 1);
}

__global__ void k_vk_prepare(VkDev *vk) {
    G1Affine P[1] = {vk->alpha};
    G2Affine Q[1] = {vk->beta};
    bool skip[1] = {vk->alpha.is_inf() || vk->beta.is_inf()};
    Fq12 f, e;
    multi_miller_loop<1>(f, P, Q, skip);
    final_exponentiation(e, f);
    vk->alpha_beta = e;
}

// ok[p] = 1 iff proof p verifies against its public inputs.  The independent strands of one proof run on four
// warps of the CTA (warp-uniform roles, lane = proof): the three Miller loops and the G2 subgroup test side by
// side, then warp 0 multiplies the three Miller values, runs the final exponentiation and compares.  (Measured
// against one thread per proof: 22 vs 39 ms for a single proof, 128 k vs 98 k verifies/s at 4096.)
//   warp 0: A, B (curve checks), Miller(A, B)           warp 2: C, Miller(C, -delta)
//   warp 1: vk_x, Miller(vk_x, -gamma)                   warp 3: B in the r-torsion subgroup?
// vkx (keys above kCoopScanMax inputs that have the byte-window tables): vk_x of every proof, computed by k_vkx; warp 1
// then only checks that the inputs are canonical.
// Listed: the proofs of the list k_rlc_failed wrote (lzkp_verify_batch_device re-verifying failing groups without the
// host).  Entry i of the launch is proof list[i]; the kernel runs only while i < F = *count and lo < F <= hi, the
// range of F for which the host path would pick this form, so that one launch per form covers every F.
struct ListGate {
    const uint32_t *list, *count;
    uint32_t lo, hi;
};
template <bool Listed>
__global__ void __launch_bounds__(128) k_verify4(const VkDev *__restrict__ vk, const G1Affine *__restrict__ gamma_abc,
                                                 uint32_t n_pub, const uint8_t *__restrict__ proofs,
                                                 const Fr *__restrict__ inputs, const G1Affine *__restrict__ vkx, uint32_t n,
                                                 uint8_t *__restrict__ ok, ListGate lg) {
    extern __shared__ uint4 smem_raw[];
    Fq12 *sf = reinterpret_cast<Fq12 *>(smem_raw);                       // [2][32] Miller values of warps 1, 2
    __shared__ uint8_t sgood[4][32];
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t p = blockIdx.x * 32 + lane;
    if (Listed) {
        n = *lg.count;
        if (n <= lg.lo || n > lg.hi) return;
    }
    const bool live = p < n;
    if (Listed && live) p = lg.list[p];
    const uint8_t *pb = proofs + (size_t)p * 256;
    Fq12 f;
    bool good = true;
    if (live) {
        G1Affine P[1];
        G2Affine Q[1];
        bool skip[1];
        if (role == 0) {
            good = read_g1_checked(pb, P[0]);
            good = read_g2_on_curve(pb + 64, Q[0]) && good;
            skip[0] = !good || P[0].is_inf() || Q[0].is_inf();
            multi_miller_loop<1>(f, P, Q, skip);
        } else if (role == 1) {
            const Fr *x = inputs + (size_t)p * n_pub;
            if (vkx) {
#pragma unroll 1
                for (uint32_t i = 0; i < n_pub; i++) good = fr_is_canonical(ld_vec(x + i)) && good;
                P[0] = ld_vec(vkx + p);
            } else {
                G1XYZZ acc = G1XYZZ::from_affine(ldg_vec(gamma_abc));
#pragma unroll 1
                for (uint32_t i = 0; i < n_pub; i++) {
                    Fr xi = ld_vec(x + i);
                    if (!fr_is_canonical(xi)) { good = false; continue; }
                    if (xi.is_zero()) continue;
                    acc.add_cold(scalar_mul(G1XYZZ::from_affine(ldg_vec(gamma_abc + 1 + i)), xi));
                }
                P[0] = acc.to_affine();
            }
            Q[0] = vk->gamma_neg;
            skip[0] = !good || P[0].is_inf() || Q[0].is_inf();
            multi_miller_loop<1>(f, P, Q, skip);
            sf[lane] = f;
        } else if (role == 2) {
            good = read_g1_checked(pb + 192, P[0]);
            Q[0] = vk->delta_neg;
            skip[0] = !good || P[0].is_inf() || Q[0].is_inf();
            multi_miller_loop<1>(f, P, Q, skip);
            sf[32 + lane] = f;
        } else {
            G2Affine B;
            good = read_g2_checked(pb + 64, B);
        }
    }
    sgood[role][lane] = good ? 1 : 0;
    __syncthreads();
    if (role == 0 && live) {
        good = sgood[0][lane] && sgood[1][lane] && sgood[2][lane] && sgood[3][lane];
        if (!good) { ok[p] = 0; return; }
        Fq12 t, e;
        f12_mul(t, f, sf[lane]);
        f12_mul(f, t, sf[32 + lane]);
        final_exponentiation(e, f);
        ok[p] = f12_eq(e, vk->alpha_beta) ? 1 : 0;
    }
}

// ---------------------------------------------------------------- random-linear-combination batching (large batches)
// With independent random rho_p (128 random bits each, used as rho = k1 + lambda k2 with 64-bit halves: ec.cuh
// scalar_mul_glv64 / glv64_coefficient - still 2^128 distinct values), all proofs of a GROUP of kRlcGroup hold iff (up to 2^-128)
//     prod_p e(rho_p A_p, B_p) * e(sum_p rho_p vk_x_p, -gamma) * e(sum_p rho_p C_p, -delta) * e(-(sum_p rho_p) alpha, beta) == 1:
// one Miller loop per proof instead of three and ONE final exponentiation per group instead of per proof.  Four kernels:
//   k_rlc_prepare  lane = proof: format / curve / subgroup checks (exactly k_verify4's), f_p = Miller(rho_p A_p, B_p),
//                  rho_p C_p, and per CTA of 32 proofs the sums  sum_p rho_p x_pj  (the vk_x combination happens ONCE per
//                  group and input: sum_p rho_p vk_x_p = sum_j (sum_p rho_p x_pj) gamma_abc_j with x_p0 = 1)
//   k_rlc_reduce   thread = group: product of its f_p, sum of its rho_p C_p, sum of its CTAs' scalar sums
//   k_rlc_inputs   thread = (group, input j): (sum_p rho_p x_pj) * gamma_abc_j
//   k_rlc_tail     lane = group, four warps: the three remaining Miller loops side by side, final exponentiation
// Malformed proofs are excluded (f = 1, zero contributions) and reported individually; a group whose combined check
// fails is re-verified proof by proof with k_verify4, so the decisions are those of independent verification.
constexpr uint32_t kRlcGroup = 64;      // proofs per combined check (two CTAs of k_rlc_prepare)

__device__ __forceinline__ Fr warp_sum_fr(Fr v) {
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        Fr o;
#pragma unroll
        for (int i = 0; i < 8; i++) o.l[i] = __shfl_down_sync(0xffffffffu, v.l[i], off);
        v = v + o;
    }
    return v;
}

// sx_out == nullptr (keys above kCoopScanMax inputs): no scalar sums here, k_rlc_input_sums forms them per (group, input).
// Four role warps per 32 proofs, lane = proof, balanced so that the longest strand is ~2200 Fq2 products (a single warp
// running rho * A and the whole Miller loop was ~3400):
//   warp 0: A, rho * A -> shared; upper share of Miller(rho A, B), then its 41 squarings; at the end upper * lower
//   warp 1: B on the twist; walks the twist point through the upper iterations, then the lower share of the loop
//   warp 2: C, rho * C; the public-input scan and the scalar sums           warp 3: B in the r-torsion subgroup
constexpr int kLaneSplit = 38;       // iterations kAteTop .. kLaneSplit on warp 0, kLaneSplit-1 .. 0 and the final lines on warp 1
__global__ void __launch_bounds__(128) k_rlc_prepare(const VkDev *__restrict__ vk, uint32_t n_pub, const uint8_t *__restrict__ proofs,
                                                     const Fr *__restrict__ inputs, const uint32_t *__restrict__ rho, uint32_t n,
                                                     Fq12 *__restrict__ f_out, G1XYZZ *__restrict__ rc_out, Fr *__restrict__ sx_out,
                                                     uint8_t *__restrict__ ok) {
    extern __shared__ uint4 smem_raw[];
    Fq12 *s_lower = reinterpret_cast<Fq12 *>(smem_raw);                          // [32] lower shares
    G1Affine *s_P = reinterpret_cast<G1Affine *>(s_lower + 32);                  // [32] rho * A
    __shared__ uint8_t sgood[4][32], s_goodA[32];
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31, p = blockIdx.x * 32 + lane;
    const bool live = p < n;
    const uint8_t *pb = proofs + (size_t)p * 256;
    uint32_t k[4] = {0, 0, 0, 0};
    if (live) {
        const uint4 r4 = reinterpret_cast<const uint4 *>(rho)[p];
        k[0] = r4.x; k[1] = r4.y; k[2] = r4.z; k[3] = r4.w;
    }
    bool good = true;
    Fq12 f;
    G1XYZZ rc = G1XYZZ::inf();
    if (role == 0) {
        G1Affine P = G1Affine::inf();
        G2Affine Q = G2Affine::inf();
        if (live) {
            good = read_g1_checked(pb, P);
            if (good && !P.is_inf()) P = scalar_mul_glv64(G1XYZZ::from_affine(P), k).to_affine();
            st_vec(s_P + lane, P);
            s_goodA[lane] = good ? 1 : 0;
        }
        asm volatile("bar.sync 1, 64;" ::: "memory");                           // rho * A is there (warps 0 and 1)
        if (live) {
            good = read_g2_on_curve(pb + 64, Q) && good;
            if (!good || P.is_inf() || Q.is_inf()) f12_one(f);
            else {
                G2Proj R{Q.x, Q.y, Fq2::one()};
                miller_share(f, P, Q, R, kAteTop, kLaneSplit, kLaneSplit, false);
            }
        }
    } else if (role == 1) {
        G2Affine Q = G2Affine::inf();
        G2Proj R{Fq2::one(), Fq2::one(), Fq2::one()};
        if (live) {
            good = read_g2_on_curve(pb + 64, Q);
            if (good && !Q.is_inf()) {
                R = G2Proj{Q.x, Q.y, Fq2::one()};
                miller_advance(R, Q, kAteTop, kLaneSplit);
            }
        }
        asm volatile("bar.sync 1, 64;" ::: "memory");
        if (live) {
            const G1Affine P = ld_vec(s_P + lane);
            if (!good || !s_goodA[lane] || P.is_inf() || Q.is_inf()) f12_one(f);
            else miller_share(f, P, Q, R, kLaneSplit - 1, 0, 0, true);
            s_lower[lane] = f;
        }
    } else if (role == 2) {
        if (live) {
            G1Affine C;
            good = read_g1_checked(pb + 192, C);
            if (good && !C.is_inf()) rc = scalar_mul_glv64(G1XYZZ::from_affine(C), k);
            const Fr *x = inputs + (size_t)p * n_pub;
#pragma unroll 1
            for (uint32_t i = 0; i < n_pub; i++) good = fr_is_canonical(ld_vec(x + i)) && good;
        }
    } else if (live) {
        G2Affine B;
        good = read_g2_checked(pb + 64, B);
    }
    sgood[role][lane] = good ? 1 : 0;
    __syncthreads();
    good = live && sgood[0][lane] && sgood[1][lane] && sgood[2][lane] && sgood[3][lane];
    if (role == 0 && live) {
        if (!good) f12_one(f);
        else { Fq12 t; f12_mul(t, f, s_lower[lane]); f = t; }
        f_out[p] = f;
        ok[p] = good ? 1 : 0;
    } else if (role == 2) {
        if (live) st_vec(rc_out + p, good ? rc : G1XYZZ::inf());
        if (!sx_out) return;                                                     // k_rlc_input_sums forms the sums
        // sums over this CTA's 32 proofs of rho_p * x_pj, j = 0 .. n_pub (x_p0 = 1), as plain (canonical) residues mod r
        Fr rho_c = Fr::zero(), rho_m = Fr::zero();
        if (good) {
            rho_c = glv64_coefficient(k);
            rho_m = Fr::from_canonical(rho_c);
        }
        Fr *dst = sx_out + (size_t)blockIdx.x * (n_pub + 1);
        Fr s0 = warp_sum_fr(rho_c);
        if (lane == 0) st_vec(dst, s0);
        const Fr *x = inputs + (size_t)(live ? p : 0) * n_pub;
#pragma unroll 1
        for (uint32_t j = 0; j < n_pub; j++) {
            Fr t = good ? rho_m * ld_vec(x + j) : Fr::zero();      // (rho R)(x) R^-1 = rho x, canonical x: plain value of the product
            t = warp_sum_fr(t);
            if (lane == 0) st_vec(dst + 1 + j, t);
        }
    }
}

// The same per-proof work with ONE warp per 32 proofs running the four strands one after the other.  k_rlc_prepare's
// four role warps finish at very different times (Miller loop ~2800 Fq2 products, subgroup ladder ~1500, rho * C ~500,
// the input scan ~0) and at 255 registers only two such CTAs fit an SM: on average 3.4 of the 8 resident warps work.
// Here every resident warp works all the time; CTAs of two warps = one group of 64 proofs.
__global__ void __launch_bounds__(64) k_rlc_prepare_seq(const VkDev *__restrict__ vk, uint32_t n_pub, const uint8_t *__restrict__ proofs,
                                                        const Fr *__restrict__ inputs, const uint32_t *__restrict__ rho, uint32_t n,
                                                        Fq12 *__restrict__ f_out, G1XYZZ *__restrict__ rc_out, Fr *__restrict__ sx_out,
                                                        uint8_t *__restrict__ ok) {
    const uint32_t gw = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, p = gw * 32 + lane;
    if (gw * 32 >= n) return;
    const bool live = p < n;
    const uint8_t *pb = proofs + (size_t)p * 256;
    uint32_t k[4] = {0, 0, 0, 0};
    if (live) {
        const uint4 r4 = reinterpret_cast<const uint4 *>(rho)[p];
        k[0] = r4.x; k[1] = r4.y; k[2] = r4.z; k[3] = r4.w;
    }
    bool good = live;
    G1Affine A = G1Affine::inf();
    G2Affine B = G2Affine::inf();
    if (live) {
        good = read_g1_checked(pb, A);
        good = read_g2_checked(pb + 64, B) && good;                       // curve and subgroup
        const Fr *x = inputs + (size_t)p * n_pub;
#pragma unroll 1
        for (uint32_t i = 0; i < n_pub; i++) good = fr_is_canonical(ld_vec(x + i)) && good;
    }
    {   // rho * C
        G1XYZZ rc = G1XYZZ::inf();
        if (live) {
            G1Affine C;
            good = read_g1_checked(pb + 192, C) && good;
            if (good && !C.is_inf()) rc = scalar_mul_glv64(G1XYZZ::from_affine(C), k);
            st_vec(rc_out + p, good ? rc : G1XYZZ::inf());
        }
    }
    if (sx_out) {   // sums over these 32 proofs of rho_p * x_pj, j = 0 .. n_pub (x_p0 = 1), as plain (canonical) residues mod r
        Fr rho_c = Fr::zero(), rho_m = Fr::zero();
        if (good) {
            rho_c = glv64_coefficient(k);
            rho_m = Fr::from_canonical(rho_c);
        }
        Fr *dst = sx_out + (size_t)gw * (n_pub + 1);
        const Fr s0 = warp_sum_fr(rho_c);
        if (lane == 0) st_vec(dst, s0);
        const Fr *x = inputs + (size_t)(live ? p : 0) * n_pub;
#pragma unroll 1
        for (uint32_t j = 0; j < n_pub; j++) {
            Fr t = good ? rho_m * ld_vec(x + j) : Fr::zero();
            t = warp_sum_fr(t);
            if (lane == 0) st_vec(dst + 1 + j, t);
        }
    }
    if (live) {
        Fq12 f;
        G1Affine P[1] = {A};
        G2Affine Q[1] = {B};
        bool skip[1];
        if (good && !A.is_inf()) P[0] = scalar_mul_glv64(G1XYZZ::from_affine(A), k).to_affine();
        skip[0] = !good || P[0].is_inf() || Q[0].is_inf();
        multi_miller_loop<1>(f, P, Q, skip);
        if (!good) f12_one(f);
        f_out[p] = f;
        ok[p] = good ? 1 : 0;
    }
}

__global__ void __launch_bounds__(64) k_rlc_reduce(const Fq12 *__restrict__ f_in, const G1XYZZ *__restrict__ rc_in,
                                                   const Fr *__restrict__ sx_in, uint32_t n, uint32_t n_pub, uint32_t groups,
                                                   Fq12 *__restrict__ gF, G1XYZZ *__restrict__ gC, Fr *__restrict__ gS) {
    const uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= groups) return;
    const uint32_t lo = g * kRlcGroup, hi = min(n, lo + kRlcGroup);
    Fq12 acc = f_in[lo], t;
    G1XYZZ c = ld_vec(rc_in + lo);
    for (uint32_t p = lo + 1; p < hi; p++) {
        f12_mul(t, acc, f_in[p]);
        acc = t;
        c.add_cold(ld_vec(rc_in + p));
    }
    gF[g] = acc;
    st_vec(gC + g, c);
    const uint32_t cta_lo = lo / 32, cta_hi = (hi + 31) / 32;
    for (uint32_t j = 0; j <= n_pub; j++) {
        Fr sum = Fr::zero();
        for (uint32_t b = cta_lo; b < cta_hi; b++) sum = sum + ld_vec(sx_in + (size_t)b * (n_pub + 1) + j);
        st_vec(gS + (size_t)g * (n_pub + 1) + j, sum);
    }
}

// X[g][j] = S[g][j] * gamma_abc[j]   (S: canonical residues)
__global__ void __launch_bounds__(64) k_rlc_inputs(const Fr *__restrict__ gS, const G1Affine *__restrict__ gamma_abc, uint32_t n_pub,
                                                   uint32_t groups, G1XYZZ *__restrict__ gX) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= groups * (n_pub + 1)) return;
    const uint32_t j = t % (n_pub + 1);
    const Fr s = ld_vec(gS + t);
    G1XYZZ r = G1XYZZ::inf();
    const G1Affine base = ldg_vec(gamma_abc + j);
    if (!s.is_zero() && !base.is_inf()) r = scalar_mul(G1XYZZ::from_affine(base), s);
    st_vec(gX + t, r);
}

__global__ void __launch_bounds__(128) k_rlc_tail(const VkDev *__restrict__ vk, const Fq12 *__restrict__ gF, const G1XYZZ *__restrict__ gC,
                                                  const Fr *__restrict__ gS, const G1XYZZ *__restrict__ gX, uint32_t n_pub,
                                                  uint32_t groups, uint8_t *__restrict__ group_ok) {
    extern __shared__ uint4 smem_raw[];
    Fq12 *sf = reinterpret_cast<Fq12 *>(smem_raw);                       // [3][32] Miller values of warps 1, 2, 3
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31, g = blockIdx.x * 32 + lane;
    const bool live = g < groups;
    if (live && role > 0) {
        G1Affine P[1];
        G2Affine Q[1];
        bool skip[1];
        Fq12 f;
        if (role == 1) {
            G1XYZZ acc = G1XYZZ::inf();
            for (uint32_t j = 0; j <= n_pub; j++) acc.add_cold(ld_vec(gX + (size_t)g * (n_pub + 1) + j));
            P[0] = acc.to_affine();
            Q[0] = vk->gamma_neg;
        } else if (role == 2) {
            P[0] = ld_vec(gC + g).to_affine();
            Q[0] = vk->delta_neg;
        } else {
            const Fr srho = ld_vec(gS + (size_t)g * (n_pub + 1));
            G1XYZZ t = G1XYZZ::inf();
            if (!srho.is_zero() && !vk->alpha.is_inf()) t = scalar_mul(G1XYZZ::from_affine(vk->alpha), srho);
            P[0] = t.to_affine().neg();
            Q[0] = vk->beta;
        }
        skip[0] = P[0].is_inf() || Q[0].is_inf();
        multi_miller_loop<1>(f, P, Q, skip);
        sf[(role - 1) * 32 + lane] = f;
    }
    __syncthreads();
    if (live && role == 0) {
        Fq12 f = gF[g], t, e, one;
        f12_mul(t, f, sf[lane]);
        f12_mul(f, t, sf[32 + lane]);
        f12_mul(t, f, sf[64 + lane]);
        final_exponentiation(e, t);
        f12_one(one);
        group_ok[g] = f12_eq(e, one) ? 1 : 0;
    }
}

// ---------------------------------------------------------------- latency form: one proof per CTA (coop.cuh)
// Line coefficients of the Miller loops against the key's fixed G2 points -gamma and -delta, in the order
// multi_miller_loop consumes them (what ark-groth16's PreparedVerifyingKey stores).  Thread 0: -gamma, thread 1: -delta,
// thread 2: beta (the combined check of the random-linear-combination path pairs -(sum rho) alpha with it).
__global__ void k_prepare_lines(const VkDev *vk, Fq2 *lines_gamma, Fq2 *lines_delta, Fq2 *lines_beta) {
    if (threadIdx.x > 2) return;
    const G2Affine Q = threadIdx.x == 0 ? vk->gamma_neg : threadIdx.x == 1 ? vk->delta_neg : vk->beta;
    Fq2 *out = threadIdx.x == 0 ? lines_gamma : threadIdx.x == 1 ? lines_delta : lines_beta;
    if (Q.is_inf()) return;
    G2Proj R{Q.x, Q.y, Fq2::one()};
    LineCoeffs L;
    int n = 0;
    auto put = [&]() { out[3 * n] = L.c0; out[3 * n + 1] = L.c1; out[3 * n + 2] = L.c2; n++; };
#pragma unroll 1
    for (int i = kAteTop; i >= 0; i--) {
        pairing_dbl_step(R, L); put();
        const int d = ate_digit(i);
        if (d) { pairing_add_step(R, d > 0 ? Q : Q.neg(), L); put(); }
    }
    Fq2 twx{PairingConsts::TW_X_C0(), PairingConsts::TW_X_C1()}, twy{PairingConsts::TW_Y_C0(), PairingConsts::TW_Y_C1()};
    G2Affine q1{fq2_conj(Q.x) * twx, fq2_conj(Q.y) * twy};
    G2Affine q2{fq2_conj(q1.x) * twx, (fq2_conj(q1.y) * twy).neg()};
    pairing_add_step(R, q1, L); put();
    pairing_add_step(R, q2, L); put();
}
// tab[((i * 32 + w) * 255 + d - 1)] = d * 256^w * base_i: fixed-base byte windows.  Rows i < n_pub: gamma_abc[i + 1] (vk_x of
// the latency form); row n_pub: gamma_abc[0], row n_pub + 1: alpha (the combined check's public-input shares).  Thread = (i, w).
__global__ void __launch_bounds__(64) k_vk_tables(const VkDev *__restrict__ vk, const G1Affine *__restrict__ gamma_abc, uint32_t n_pub,
                                                  G1Affine *__restrict__ tab) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= (n_pub + 2) * coop::kTabWindows) return;
    const uint32_t i = t / coop::kTabWindows, w = t % coop::kTabWindows;
    G1XYZZ b = G1XYZZ::from_affine(i < n_pub ? ldg_vec(gamma_abc + 1 + i) : i == n_pub ? ldg_vec(gamma_abc) : vk->alpha);
#pragma unroll 1
    for (uint32_t k = 0; k < 8 * w; k++) b.dbl_cold();
    G1XYZZ acc = G1XYZZ::inf();
    G1Affine *dst = tab + (size_t)t * coop::kTabDigits;
#pragma unroll 1
    for (uint32_t d = 0; d < coop::kTabDigits; d++) {
        acc.add_cold(b);
        st_vec(dst + d, acc.to_affine());
    }
}

struct FChain {
    Fq2 f[6], ln[12], emb[3];      // ln: two dense line operands, slots 1, 2, 5 stay zero
    coop::Scratch s;
};
struct CoopSmem {
    Fq2 lines[coop::kLines * 3];      // scaled lines of (A, B); afterwards the final exponentiation's ten Fq12 slots
    FChain fc[4];                     // (A, B) upper share / -gamma / -delta / (A, B) lower share, then the exponentiation helper
    coop::LineState ls;
    coop::LadderState lad;
    Fq2 ref[6];                       // self-test only
    G1Affine A, C;
    G2Affine B;
    int ready, done[4], good[4], sub_ok, xcount, xdone;
};
static_assert(coop::kLines * 3 >= 60 + 6 * coop::kXBits, "final_exp slots and the exponentiation's shared powers");
constexpr uint32_t kCoopThreads = 224;   // seven warps, one of them idle (CoopRole)

__device__ __forceinline__ void coop_prologue(CoopSmem &sm) {
    if (threadIdx.x == 0) { sm.ready = 0; sm.done[0] = sm.done[1] = sm.done[2] = sm.done[3] = 0; sm.sub_ok = 0; sm.xcount = 0; sm.xdone = 0; }
    if (threadIdx.x < 4) st_vec(&sm.fc[threadIdx.x].s.P[18], Fq2::zero());
    if (threadIdx.x < 48) st_vec(&sm.fc[threadIdx.x / 12].ln[threadIdx.x % 12], Fq2::zero());
}
__device__ __forceinline__ coop::ExpShare exp_share(CoopSmem &sm) {
    return coop::ExpShare{sm.lines + 60, sm.fc[3].f, &sm.xcount, &sm.xdone};
}
__device__ __forceinline__ void set_emb(FChain &c, const G1Affine &P) {
    if (coop::lane_id() == 0) {
        st_vec(&c.emb[0], coop::fq2_embed(P.y));
        st_vec(&c.emb[1], coop::fq2_embed(P.x));
        st_vec(&c.emb[2], Fq2::one());
    }
    __syncwarp();
}

// ok[p] as k_verify4 decides it; one CTA per proof.  Roles by warp (warp w runs on SM partition w % 4; the two warps
// that end the proof - role 0 and the exponentiation helper - have their partition to themselves by then):
//   warp 0  AB_UPPER: upper share of the (A, B) f chain, product of the Miller values, final exponentiation (squaring side)
//   warp 4  GAMMA:    vk_x from the tables, Miller(vk_x, -gamma) on prepared lines                   (beside warp 0)
//   warp 1  LINES:    twist-point chain of (A, B) -> scaled lines in shared memory
//   warp 2  AB_LOWER: lower share of the (A, B) f chain, then the multiplying side of the three exponentiations by x
//   warp 6  DELTA:    Miller(C, -delta) on prepared lines                                            (beside warp 2)
//   warp 3  LADDER:   B in the r-torsion subgroup?                                                    warp 5: idle
// vkx: keys above kCoopScanMax inputs, whose scan would be the longest strand; k_vkx has computed vk_x of every proof.
enum CoopRole { kAbUpper = 0, kLines = 1, kAbLower = 2, kLadder = 3, kGamma = 4, kIdle = 5, kDelta = 6 };
// MIN_CTAS = 1: all the registers the code wants (250; one CTA per SM) for calls of at most one proof per SM; MIN_CTAS = 2: 128
// registers, two proofs per SM side by side - 10 % slower each (1.99 against 1.80 ms), 1.5x the throughput from 149 proofs on.
// Listed: as for k_verify4, CTA i verifies proof list[i] while i < F and lo < F <= hi.
template <int MIN_CTAS, bool Listed>
__global__ void __launch_bounds__(kCoopThreads, MIN_CTAS) k_verify_coop(const VkDev *__restrict__ vk, const G1Affine *__restrict__ gamma_abc,
                                                              const G1Affine *__restrict__ tab, const Fq2 *__restrict__ lines_gamma,
                                                              const Fq2 *__restrict__ lines_delta, uint32_t n_pub,
                                                              const uint8_t *__restrict__ proofs, const uint8_t *__restrict__ inputs,
                                                              const G1Affine *__restrict__ vkx, uint8_t *__restrict__ ok, ListGate lg) {
    extern __shared__ uint4 smem_raw[];
    CoopSmem &sm = *reinterpret_cast<CoopSmem *>(smem_raw);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    uint32_t p = blockIdx.x;
    if (Listed) {
        const uint32_t F = *lg.count;
        if (p >= F || F <= lg.lo || F > lg.hi) return;
        p = lg.list[p];
    }
    const uint8_t *pb = proofs + (size_t)p * 256;
    const uint8_t *x = inputs + (size_t)p * n_pub * 32;
    coop_prologue(sm);
    if (warp == kAbUpper && lane == 0) { G1Affine A; sm.good[0] = read_g1_checked(pb, A) ? 1 : 0; st_vec(&sm.A, A); }
    if (warp == kLines && lane == 0) { G2Affine B; sm.good[1] = read_g2_on_curve(pb + 64, B) ? 1 : 0; st_vec(&sm.B, B); }
    if (warp == kDelta && lane == 0) { G1Affine C; sm.good[2] = read_g1_checked(pb + 192, C) ? 1 : 0; st_vec(&sm.C, C); }
    if (warp == kGamma) {
        bool g = true;
        for (uint32_t i = lane; i < n_pub; i += 32) g = fr_is_canonical(ld_vec(reinterpret_cast<const Fr *>(x) + i)) && g;
        g = __all_sync(0xffffffffu, g);
        if (lane == 0) sm.good[3] = g ? 1 : 0;
    }
    __syncthreads();
    const bool all_good = sm.good[0] && sm.good[1] && sm.good[2] && sm.good[3];
    const G1Affine A = ld_vec(&sm.A);
    const G2Affine B = ld_vec(&sm.B);
    const bool skip_ab = !(sm.good[0] && sm.good[1]) || A.is_inf() || B.is_inf();
    if (warp == kAbUpper) {
        if (!all_good) { if (lane == 0) ok[p] = 0; return; }
        FChain &c = sm.fc[0];
        if (skip_ab) coop::f12_set_one(c.f);
        else coop::miller_f<true>(c.f, sm.lines, &sm.ready, c.ln, nullptr, &c.s, kAteTop, coop::kMillerSplit, coop::kMillerSplit, false);
        coop::flag_wait(&sm.done[0], 1);
        coop::f12_mul<false>(c.f, c.f, sm.fc[1].f, &c.s);
        coop::flag_wait(&sm.done[1], 1);
        coop::f12_mul<false>(c.f, c.f, sm.fc[2].f, &c.s);
        coop::flag_wait(&sm.done[3], 1);                                  // the lower share of the (A, B) loop; its warp has left the lines
        coop::f12_mul<false>(c.f, c.f, sm.fc[3].f, &c.s);
        coop::final_exp(c.f, c.f, sm.lines, &c.s, exp_share(sm));
        const bool eq = coop::f12_equal(c.f, reinterpret_cast<const Fq2 *>(&vk->alpha_beta));
        coop::flag_wait(&sm.done[2], 1);
        if (lane == 0) ok[p] = (eq && sm.sub_ok) ? 1 : 0;
    } else if (warp == kGamma) {
        FChain &c = sm.fc[1];
        bool skip = true;
        if (all_good) {
            const G1Affine P = vkx ? ld_vec(vkx + p) : coop::vkx_from_tables(tab, gamma_abc, x, n_pub);
            skip = P.is_inf() || vk->gamma_neg.is_inf();
            if (!skip) set_emb(c, P);
        }
        if (skip) coop::f12_set_one(c.f);
        else coop::miller_f<false>(c.f, lines_gamma, nullptr, c.ln, c.emb, &c.s);
        coop::flag_publish(&sm.done[0], 1);
    } else if (warp == kDelta) {
        FChain &c = sm.fc[2];
        const G1Affine C = ld_vec(&sm.C);
        const bool skip = !all_good || C.is_inf() || vk->delta_neg.is_inf();
        if (!skip) set_emb(c, C);
        if (skip) coop::f12_set_one(c.f);
        else coop::miller_f<false>(c.f, lines_delta, nullptr, c.ln, c.emb, &c.s);
        coop::flag_publish(&sm.done[1], 1);
    } else if (warp == kLines) {
        if (all_good && !skip_ab) coop::line_chain(&sm.ls, A, B, sm.lines, &sm.ready);
    } else if (warp == kAbLower) {
        if (!all_good) return;
        FChain &c = sm.fc[3];
        if (skip_ab) coop::f12_set_one(c.f);
        else coop::miller_f<true>(c.f, sm.lines, &sm.ready, c.ln, nullptr, &c.s, coop::kMillerSplit - 1, 0, 0, true);
        coop::flag_publish(&sm.done[3], 1);
        const coop::ExpShare sh = exp_share(sm);
        for (int g = 0; g < 3; g++) coop::f12_exp_helper(&c.s, sh, g);
    } else if (warp == kLadder) {
        bool in = false;
        if (all_good) in = B.is_inf() ? true : coop::g2_in_subgroup(&sm.lad, B);
        if (lane == 0) sm.sub_ok = in ? 1 : 0;
        coop::flag_publish(&sm.done[2], 1);
    }
}

// ---- the combined check of a GROUP, cooperative form (the lane-per-group k_rlc_reduce + k_rlc_tail put a whole pairing
// and 63 Fq12 products on one thread: 14.7 of the 70 ms of kernel time at 65 536 proofs).  One CTA per group:
//   warp 0: Miller(-(sum rho) alpha, beta) on prepared lines, product of everything, final exponentiation (squaring side)
//   warp 1: sum_j X[g][j] (shuffle tree), Miller(., -gamma)      warp 2: sum_p rho_p C_p (shuffle tree), Miller(., -delta)
//   warp 3: the product of the group's 64 Miller values f_p, then the multiplying side of the exponentiations by x
// gX holds n_pub + 2 columns per group: the public-input shares and, last, (sum rho) alpha (k_rlc_inputs).
struct TailSmem {
    Fq2 slots[60 + 6 * coop::kXBits];
    FChain fc[4];
    int done[3], xcount, xdone;
};
__device__ __noinline__ G1Affine coop_sum_g1(const G1XYZZ *src, uint32_t count) {     // whole warp; result on every lane
    const int lane = coop::lane_id();
    G1XYZZ acc = G1XYZZ::inf();
#pragma unroll 1
    for (uint32_t i = lane; i < count; i += 32) acc.add_cold(ld_vec(src + i));
#pragma unroll 1
    for (int off = 16; off > 0; off >>= 1) {
        G1XYZZ o;
        uint32_t *ow = reinterpret_cast<uint32_t *>(&o);
        const uint32_t *aw = reinterpret_cast<const uint32_t *>(&acc);
#pragma unroll
        for (int k = 0; k < (int)(sizeof(G1XYZZ) / 4); k++) ow[k] = __shfl_down_sync(0xffffffffu, aw[k], off);
        acc.add_cold(o);
    }
    G1Affine r = G1Affine::inf();
    if (lane == 0) r = acc.to_affine();
    uint32_t *rw = reinterpret_cast<uint32_t *>(&r);
#pragma unroll
    for (int k = 0; k < (int)(sizeof(G1Affine) / 4); k++) rw[k] = __shfl_sync(0xffffffffu, rw[k], 0);
    return r;
}
template <int MIN_CTAS>       // 2: the registers the code wants; 4: capped at 128 for twice the resident groups (large batches)
__global__ void __launch_bounds__(128, MIN_CTAS) k_rlc_tail_coop(const VkDev *__restrict__ vk, const Fq2 *__restrict__ lines_gamma,
                                                       const Fq2 *__restrict__ lines_delta, const Fq2 *__restrict__ lines_beta,
                                                       const Fq12 *__restrict__ f_in, const G1XYZZ *__restrict__ rc_in,
                                                       const G1XYZZ *__restrict__ gX, uint32_t n, uint32_t n_pub,
                                                       uint8_t *__restrict__ group_ok) {
    extern __shared__ uint4 smem_raw[];
    TailSmem &sm = *reinterpret_cast<TailSmem *>(smem_raw);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = blockIdx.x;
    const uint32_t lo = g * kRlcGroup, hi = min(n, lo + kRlcGroup), cols = n_pub + 2;
    if (threadIdx.x == 0) { sm.done[0] = sm.done[1] = sm.done[2] = 0; sm.xcount = 0; sm.xdone = 0; }
    if (threadIdx.x < 4) st_vec(&sm.fc[threadIdx.x].s.P[18], Fq2::zero());
    if (threadIdx.x < 48) st_vec(&sm.fc[threadIdx.x / 12].ln[threadIdx.x % 12], Fq2::zero());
    __syncthreads();
    const coop::ExpShare sh{sm.slots + 60, sm.fc[3].f, &sm.xcount, &sm.xdone};
    FChain &c = sm.fc[warp];
    if (warp == 3) {
        // the group's Miller values: f[0] * f[1] * ... (a malformed proof contributed 1)
        for (uint32_t k = lane; k < 6; k += 32) st_vec(&c.f[k], ld_vec(reinterpret_cast<const Fq2 *>(f_in + lo) + k));
        __syncwarp();
#pragma unroll 1
        for (uint32_t p = lo + 1; p < hi; p++) {
            for (uint32_t k = lane; k < 6; k += 32) st_vec(&c.ln[k], ld_vec(reinterpret_cast<const Fq2 *>(f_in + p) + k));
            __syncwarp();
            coop::f12_mul<false>(c.f, c.f, c.ln, &c.s);
        }
        // hand the product to warp 0 in fc[3].ln (fc[3].f becomes the exponentiation helper's running product)
        coop::f12_copy(c.ln + 6, c.f);
        coop::flag_publish(&sm.done[2], 1);
        for (int e = 0; e < 3; e++) coop::f12_exp_helper(&c.s, sh, e);
        return;
    }
    G1Affine P;
    const Fq2 *lines;
    bool skip;
    if (warp == 0) {
        P = ld_vec(gX + (size_t)g * cols + n_pub + 1).to_affine().neg();
        lines = lines_beta;
        skip = P.is_inf() || vk->beta.is_inf();
    } else if (warp == 1) {
        P = coop_sum_g1(gX + (size_t)g * cols, n_pub + 1);
        lines = lines_gamma;
        skip = P.is_inf() || vk->gamma_neg.is_inf();
    } else {
        P = coop_sum_g1(rc_in + lo, hi - lo);
        lines = lines_delta;
        skip = P.is_inf() || vk->delta_neg.is_inf();
    }
    if (skip) coop::f12_set_one(c.f);
    else { set_emb(c, P); coop::miller_f<false>(c.f, lines, nullptr, c.ln, c.emb, &c.s); }
    if (warp) { coop::flag_publish(&sm.done[warp - 1], 1); return; }
    coop::flag_wait(&sm.done[0], 1);
    coop::f12_mul<false>(c.f, c.f, sm.fc[1].f, &c.s);
    coop::flag_wait(&sm.done[1], 1);
    coop::f12_mul<false>(c.f, c.f, sm.fc[2].f, &c.s);
    coop::flag_wait(&sm.done[2], 1);
    coop::f12_mul<false>(c.f, c.f, sm.fc[3].ln + 6, &c.s);
    coop::final_exp(c.f, c.f, sm.slots, &c.s, sh);
    coop::f12_set_one(c.ln);                    // c.ln is free again (the loop's dense line operand)
    const bool eq = coop::f12_equal(c.f, c.ln);
    if (lane == 0) group_ok[g] = eq ? 1 : 0;
}
// gS[g][j] = sum over the group's CTAs of the scalar sums of k_rlc_prepare (what k_rlc_reduce does beside its products)
__global__ void __launch_bounds__(128) k_rlc_scalars(const Fr *__restrict__ sx_in, uint32_t n, uint32_t n_pub, uint32_t groups,
                                                     Fr *__restrict__ gS) {
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= groups * (n_pub + 1)) return;
    const uint32_t g = t / (n_pub + 1), j = t % (n_pub + 1);
    const uint32_t lo = g * kRlcGroup, hi = min(n, lo + kRlcGroup), cta_lo = lo / 32, cta_hi = (hi + 31) / 32;
    Fr sum = Fr::zero();
    for (uint32_t b = cta_lo; b < cta_hi; b++) sum = sum + ld_vec(sx_in + (size_t)b * (n_pub + 1) + j);
    st_vec(gS + t, sum);
}
// gS[g][j] straight from the inputs, thread = (group g, column j): keys above kCoopScanMax inputs.  There the scalar sums of
// k_rlc_prepare are one warp walking all n_pub columns per 32 proofs (a shuffle tree per column) beside the Miller loop;
// here the group's 64 coefficients are formed once in shared memory and every thread sums 64 products of one column.
// ok[p] (k_rlc_prepare's verdict on the proof's form) decides whether rho_p takes part, as `good` does there.
__global__ void __launch_bounds__(128) k_rlc_input_sums(const Fr *__restrict__ inputs, const uint32_t *__restrict__ rho,
                                                        const uint8_t *__restrict__ ok, uint32_t n, uint32_t n_pub,
                                                        Fr *__restrict__ gS) {
    __shared__ Fr s_c[kRlcGroup], s_m[kRlcGroup];          // rho_p canonical / as a Montgomery residue; zero if malformed
    const uint32_t g = blockIdx.x, j = blockIdx.y * blockDim.x + threadIdx.x, lo = g * kRlcGroup, cnt = min(n - lo, kRlcGroup);
    if (threadIdx.x < cnt) {
        const uint32_t p = lo + threadIdx.x;
        Fr c = Fr::zero();
        if (ok[p]) {
            const uint4 r4 = reinterpret_cast<const uint4 *>(rho)[p];
            uint32_t k[4] = {r4.x, r4.y, r4.z, r4.w};
            c = glv64_coefficient(k);
        }
        st_vec(s_c + threadIdx.x, c);
        st_vec(s_m + threadIdx.x, Fr::from_canonical(c));
    }
    __syncthreads();
    if (j > n_pub) return;
    Fr sum = Fr::zero();
    if (j == 0) {
        for (uint32_t q = 0; q < cnt; q++) sum = sum + ld_vec(s_c + q);
    } else {
        const Fr *x = inputs + (size_t)lo * n_pub + (j - 1);
#pragma unroll 4
        for (uint32_t q = 0; q < cnt; q++) sum = sum + ld_vec(s_m + q) * ld_vec(x + (size_t)q * n_pub);
    }
    st_vec(gS + (size_t)g * (n_pub + 1) + j, sum);
}
// X[g][j] = S[g][j] * gamma_abc[j] for j <= n_pub, and the extra column X[g][n_pub + 1] = S[g][0] * alpha, from the byte-window
// tables: one warp per (g, j), lane = byte of the scalar, then a shuffle tree.  (As a 254-bit scalar multiplication on one
// thread per (g, j) this stage was a 1.4 ms chain in EVERY combined-form call, whatever its size.)
__global__ void __launch_bounds__(128) k_rlc_inputs2(const Fr *__restrict__ gS, const G1Affine *__restrict__ tab, uint32_t n_pub,
                                                     uint32_t groups, G1XYZZ *__restrict__ gX) {
    const uint32_t t = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31, cols = n_pub + 2;
    if (t >= groups * cols) return;
    const uint32_t g = t / cols, j = t % cols;
    const uint8_t *sbytes = reinterpret_cast<const uint8_t *>(gS + (size_t)g * (n_pub + 1) + (j <= n_pub ? j : 0));
    const uint32_t row = j == 0 ? n_pub : j <= n_pub ? j - 1 : n_pub + 1, d = sbytes[lane];
    G1XYZZ acc = G1XYZZ::inf();
    if (d) acc = G1XYZZ::from_affine(ldg_vec(tab + ((size_t)row * coop::kTabWindows + lane) * coop::kTabDigits + (d - 1)));
#pragma unroll 1
    for (int off = 16; off > 0; off >>= 1) {
        G1XYZZ o;
        uint32_t *ow = reinterpret_cast<uint32_t *>(&o);
        const uint32_t *aw = reinterpret_cast<const uint32_t *>(&acc);
#pragma unroll
        for (int k = 0; k < (int)(sizeof(G1XYZZ) / 4); k++) ow[k] = __shfl_down_sync(0xffffffffu, aw[k], off);
        acc.add_cold(o);
    }
    if (lane == 0) st_vec(gX + t, acc);
}

// ---- the combined form without the host (lzkp_verify_batch_device)
// rho of every proof from a 256-bit seed, thread = ChaCha20 block of four proofs (chacha20.cuh): the call passes the seed
// as a kernel argument, so nothing is staged in host memory that a later call could overwrite before the copy ran.
struct RhoSeed { uint32_t w[8]; };
__global__ void __launch_bounds__(128) k_rlc_rho(RhoSeed seed, uint32_t n, uint32_t *__restrict__ rho) {
    const uint32_t blk = blockIdx.x * blockDim.x + threadIdx.x;
    if (blk >= (n + 3) / 4) return;
    rlc_rho_block(seed.w, blk, n, rho);
}
// list[0 .. F) = the proofs of every group whose combined check failed, ascending, and count[0] = F.  One CTA: a scan of
// the group flags in chunks of one flag per thread (1024 groups at 65 536 proofs).
constexpr uint32_t kFailedThreads = 1024;
__global__ void __launch_bounds__(kFailedThreads) k_rlc_failed(const uint8_t *__restrict__ group_ok, uint32_t n, uint32_t groups,
                                                               uint32_t *__restrict__ list, uint32_t *__restrict__ count) {
    __shared__ uint32_t s_warp[kFailedThreads / 32], s_base;
    const uint32_t t = threadIdx.x, lane = t & 31, warp = t >> 5;
    if (t == 0) s_base = 0;
#pragma unroll 1
    for (uint32_t g0 = 0; g0 < groups; g0 += kFailedThreads) {
        const uint32_t g = g0 + t, lo = g * kRlcGroup;
        const uint32_t cnt = g < groups && !group_ok[g] ? min(n - lo, kRlcGroup) : 0;
        uint32_t incl = cnt;                                              // inclusive scan: warp, then across warps
#pragma unroll
        for (int off = 1; off < 32; off <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, incl, off);
            if (lane >= (uint32_t)off) incl += v;
        }
        if (lane == 31) s_warp[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            uint32_t w = s_warp[lane];
#pragma unroll
            for (int off = 1; off < 32; off <<= 1) {
                const uint32_t v = __shfl_up_sync(0xffffffffu, w, off);
                if (lane >= (uint32_t)off) w += v;
            }
            s_warp[lane] = w;
        }
        __syncthreads();
        const uint32_t base = s_base + (warp ? s_warp[warp - 1] : 0) + incl - cnt;
        for (uint32_t k = 0; k < cnt; k++) list[base + k] = lo + k;
        __syncthreads();
        if (t == 0) s_base += s_warp[kFailedThreads / 32 - 1];
        __syncthreads();
    }
    if (t == 0) *count = s_base;
}

// ---- vk_x of every proof of a call, keys above kCoopScanMax public inputs.  The latency form's GAMMA warp scans all
// n_pub x 32 (input, byte) pairs itself (coop::vkx_from_tables), and the Miller loop against -gamma waits for it: at 2049
// inputs that is ~2000 steps on the critical path.  Here one CTA per proof: warp w takes the slices w, w + warps, ... of
// `slice` inputs; a lane holds one input (32 bytes in registers) and walks its bytes upwards, with a ballot skipping the
// windows where no lane of the warp has a nonzero byte and ending the chunk once no lane has one left (64-bit values: 8
// windows, bits: 1).  Partial XYZZ sums, gamma_abc[0] on warp 0, one shuffle-tree reduction, affine result in vkx[p].
constexpr uint32_t kCoopScanMax = 256;       // keys of up to this many inputs keep the in-kernel scan
constexpr uint32_t kVkxWarps = 8;
// Inputs per slice.  At 2049 inputs (B200, 1000 W) k_vkx takes 0.22 / 0.49 / 1.07 ms for 1 / 64 / 444 proofs with slices of 64;
// 32 and 128 tie at 1 and 64 proofs and lose at 444 (1.16, 1.18 ms), 256 and 512 lose at 64 proofs (0.57, 0.83 ms).
constexpr uint32_t kVkxSlice = 64;
// Listed: CTA i computes vk_x of proof list[i] while i < F (every F: all re-verifying forms read it).
template <bool Listed>
__global__ void __launch_bounds__(kVkxWarps * 32) k_vkx(const G1Affine *__restrict__ tab, const G1Affine *__restrict__ gamma_abc,
                                                        uint32_t n_pub, uint32_t slice, const uint8_t *__restrict__ inputs,
                                                        G1Affine *__restrict__ vkx, ListGate lg) {
    __shared__ G1XYZZ part[kVkxWarps * 32];
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31, warps = blockDim.x >> 5;
    uint32_t p = blockIdx.x;
    if (Listed) {
        if (p >= *lg.count) return;
        p = lg.list[p];
    }
    const uint4 *x = reinterpret_cast<const uint4 *>(inputs + (size_t)p * n_pub * 32);
    G1XYZZ acc = G1XYZZ::inf();
    if (threadIdx.x == 0) acc = G1XYZZ::from_affine(ldg_vec(gamma_abc));
#pragma unroll 1
    for (uint32_t s0 = warp * slice; s0 < n_pub; s0 += warps * slice) {
        const uint32_t end = min(n_pub, s0 + slice);
#pragma unroll 1
        for (uint32_t c = s0; c < end; c += 32) {
            const uint32_t i = c + lane;
            uint32_t v[8] = {0, 0, 0, 0, 0, 0, 0, 0};
            if (i < end) {
                const uint4 lo = __ldg(x + 2 * (size_t)i), hi = __ldg(x + 2 * (size_t)i + 1);
                v[0] = lo.x; v[1] = lo.y; v[2] = lo.z; v[3] = lo.w; v[4] = hi.x; v[5] = hi.y; v[6] = hi.z; v[7] = hi.w;
            }
            const G1Affine *row = tab + (size_t)i * coop::kTabWindows * coop::kTabDigits;
#pragma unroll 1
            for (uint32_t w = 0; w < coop::kTabWindows; w++) {
                const uint32_t rest = v[0] | v[1] | v[2] | v[3] | v[4] | v[5] | v[6] | v[7];
                if (__ballot_sync(0xffffffffu, rest != 0) == 0) break;
                const uint32_t d = v[0] & 0xFFu;
                if (d) acc.madd(ldg_vec(row + w * coop::kTabDigits + (d - 1)));
#pragma unroll
                for (int k = 0; k < 7; k++) v[k] = __funnelshift_r(v[k], v[k + 1], 8);
                v[7] >>= 8;
            }
        }
    }
    st_vec(part + threadIdx.x, acc);
    __syncthreads();
    if (warp == 0) {
        const G1Affine r = coop_sum_g1(part, blockDim.x);
        if (lane == 0) st_vec(vkx + p, r);
    }
}

// LZKP_COOP_SELFTEST=1 at key load: the cooperative Miller loop (both line sources), final exponentiation and subgroup
// test against the serial code of pairing.cuh on the key's own points.  result: bit per failing stage.
__global__ void __launch_bounds__(kCoopThreads) k_coop_selftest(const VkDev *__restrict__ vk, const Fq2 *__restrict__ lines_gamma, int *result, long long *stamps, int solo) {
    extern __shared__ uint4 smem_raw[];
    CoopSmem &sm = *reinterpret_cast<CoopSmem *>(smem_raw);
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    coop_prologue(sm);
    __syncthreads();
    const G1Affine A = vk->alpha;
    const G2Affine B = vk->beta;
    const long long t_start = clock64();
    auto stamp = [&](int k) { if (lane == 0) stamps[k] = clock64() - t_start; };
    if (solo) {              // timing only: the (A, B) Miller loop's two warps with nothing beside them (solo = 2: line chain alone first)
        if (warp == kLines) { coop::line_chain(&sm.ls, A, B, sm.lines, &sm.ready); stamp(11); }
        if (warp == kAbUpper) {
            if (solo == 2) coop::flag_wait(&sm.ready, coop::kLines);
            const long long t0 = clock64();
            coop::miller_f<true>(sm.fc[0].f, sm.lines, &sm.ready, sm.fc[0].ln, nullptr, &sm.fc[0].s);
            if (lane == 0) { stamps[10] = clock64() - t_start; stamps[9] = clock64() - t0; }
        }
        return;
    }
    if (warp == kAbUpper) {
        FChain &c = sm.fc[0];
        coop::miller_f<true>(c.f, sm.lines, &sm.ready, c.ln, nullptr, &c.s, kAteTop, coop::kMillerSplit, coop::kMillerSplit, false);
        coop::flag_wait(&sm.done[3], 1);
        coop::f12_mul<false>(c.f, c.f, sm.fc[3].f, &c.s);
        stamp(0);
        {   // timing only: the whole f chain on one warp with every line already there, and 64 plain products
            const long long t0 = clock64();
            coop::miller_f<true>(c.ln, sm.lines, &sm.ready, c.ln + 6, nullptr, &c.s);
            if (lane == 0) stamps[5] = clock64() - t0;
            const long long t1 = clock64();
            for (int i = 0; i < 64; i++) coop::f12_mul<false>(c.ln, c.ln, c.f, &c.s);
            if (lane == 0) stamps[6] = clock64() - t1;
            const long long t3 = clock64();
            if (lane == 0) { Fq6 *n6 = reinterpret_cast<Fq6 *>(c.ln); f6_inv(*n6, *n6); }
            __syncwarp();
            if (lane == 0) stamps[7] = clock64() - t3;
            const long long t5 = clock64();
            if (lane == 0) { Fq v = ld_vec(&c.ln[0].c0); v = v.inverse(); st_vec(&c.ln[0].c0, v); }
            __syncwarp();
            if (lane == 0) stamps[8] = clock64() - t5;
            const long long t6 = clock64();
            if (lane == 0) { Fq2 v = ld_vec(&c.ln[0]); for (int i = 0; i < 16; i++) v = v * v; st_vec(&c.ln[0], v); }
            __syncwarp();
            if (lane == 0) stamps[9] = clock64() - t6;
        }
        coop::flag_wait(&sm.done[0], 1);
        if (!coop::f12_equal(c.f, sm.fc[1].f) && lane == 0) atomicOr(result, 1);
        coop::flag_publish(&sm.done[2], 1);                              // the lines may now be overwritten: warp 4 turns helper
        const long long t2 = clock64();
        coop::final_exp(c.f, c.f, sm.lines, &c.s, exp_share(sm));
        if (lane == 0) stamps[1] = clock64() - t2;
        if (!coop::f12_equal(c.f, reinterpret_cast<const Fq2 *>(&vk->alpha_beta)) && lane == 0) atomicOr(result, 2);
    } else if (warp == kAbLower) {
        FChain &c = sm.fc[3];
        coop::miller_f<true>(c.f, sm.lines, &sm.ready, c.ln, nullptr, &c.s, coop::kMillerSplit - 1, 0, 0, true);
        coop::flag_publish(&sm.done[3], 1);
        coop::flag_wait(&sm.done[2], 1);
        const coop::ExpShare sh = exp_share(sm);
        for (int g = 0; g < 3; g++) coop::f12_exp_helper(&c.s, sh, g);
    } else if (warp == kGamma) {
        if (lane == 0) {
            G1Affine P[1] = {A};
            G2Affine Q[1] = {B};
            bool skip[1] = {false};
            Fq12 f;
            multi_miller_loop<1>(f, P, Q, skip);
            *reinterpret_cast<Fq12 *>(sm.fc[1].f) = f;
        }
        coop::flag_publish(&sm.done[0], 1);
    } else if (warp == kDelta) {
        FChain &c = sm.fc[2];
        set_emb(c, A);
        coop::miller_f<false>(c.f, lines_gamma, nullptr, c.ln, c.emb, &c.s);
        stamp(2);
        coop::flag_wait(&sm.done[1], 1);
        if (!coop::f12_equal(c.f, sm.ref) && lane == 0) atomicOr(result, 4);
    } else if (warp == kLines) {
        coop::line_chain(&sm.ls, A, B, sm.lines, &sm.ready);
        stamp(3);
    } else if (warp == kLadder) {
        if (lane == 0) {
            G1Affine P[1] = {A};
            G2Affine Q[1] = {vk->gamma_neg};
            bool skip[1] = {false};
            Fq12 f;
            multi_miller_loop<1>(f, P, Q, skip);
            *reinterpret_cast<Fq12 *>(sm.ref) = f;
        }
        coop::flag_publish(&sm.done[1], 1);
        const long long t4 = clock64();
        if (!coop::g2_in_subgroup(&sm.lad, B) && lane == 0) atomicOr(result, 8);
        if (lane == 0) stamps[4] = clock64() - t4;
    }
}

__global__ void k_fq_mont(Fq *v, size_t count) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    st_vec(v + k, Fq::from_canonical(ld_vec(v + k)));
}

}  // namespace

namespace eng {

struct VerifyingKeyDev {
    DBuf vk, gamma_abc;
    DBuf d_p, d_x, d_ok;          // grow-only staging of lzkp_verify_batch's host buffers
    DBuf d_rho, d_f, d_rc, d_sx, d_gF, d_gC, d_gS, d_gX, d_gok;     // random-linear-combination path (large batches)
    DBuf d_list;                                                                 // failing groups' proofs and their count (k_rlc_failed)
    DBuf lines_gamma, lines_delta, lines_beta, tab;                             // latency form (coop.cuh): prepared lines, vk_x byte-window tables
    DBuf d_vkx;                                                                  // vk_x per proof (k_vkx; keys above kCoopScanMax inputs)
    bool coop_ok = false;
    uint32_t n_pub = 0;
    int device = 0;                                                              // the device the key was loaded on
    // Last use of the per-call buffers above, on whatever stream it was enqueued (lzkp_verify_batch_device returns before
    // its work has run).  Every call waits on it in its stream before touching them and records it after its last
    // enqueue: event_acquire / event_release.  mu only orders the ENQUEUES.
    cudaEvent_t last_use = nullptr;
    std::mutex mu;
    ~VerifyingKeyDev() {
        if (last_use) { cudaEventSynchronize(last_use); cudaEventDestroy(last_use); }
    }
};
// A call that needs a larger buffer than the key holds first waits on the host for the calls still using the old one.
static int grow(VerifyingKeyDev *V, DBuf &b, size_t bytes) {
    if (bytes <= b.bytes) return LZKP_OK;
    if (V->last_use) CUDA_TRY(cudaEventSynchronize(V->last_use));
    return b.alloc(bytes);
}
// size x count bytes from the OS CSPRNG (the soundness of the combined check rests on their unpredictability)
static bool os_entropy(void *dst, size_t size, size_t count) {
    FILE *ur = fopen("/dev/urandom", "rb");
    const bool got = ur && fread(dst, size, count, ur) == count;
    if (ur) fclose(ur);
    return got;
}

// The latency and combined forms' per-key data: prepared lines of -gamma / -delta / beta and the byte-window tables of
// gamma_abc and alpha, (n_pub + 2) x 32 x 255 affine points = 0.52 MB per public input (68.4 MB for the 129 inputs of the
// membership key, 1.07 GB for the 2049 of membership with 1024 slots).  When they cannot be allocated the key still loads
// and verifies one proof per lane (k_verify4).
static size_t coop_table_bytes(uint32_t n_pub) {
    return (size_t)(n_pub + 2) * coop::kTabWindows * coop::kTabDigits * sizeof(G1Affine);
}
static int coop_prepare(VerifyingKeyDev *V) {
    const size_t line_bytes = (size_t)coop::kLines * 3 * sizeof(Fq2);
    if (V->lines_gamma.alloc(line_bytes) != LZKP_OK || V->lines_delta.alloc(line_bytes) != LZKP_OK ||
        V->lines_beta.alloc(line_bytes) != LZKP_OK || V->tab.alloc(coop_table_bytes(V->n_pub)) != LZKP_OK) {
        V->lines_gamma.release(); V->lines_delta.release(); V->lines_beta.release(); V->tab.release();
        cudaGetLastError();
        return LZKP_OK;                                                          // coop_ok stays false
    }
    CUDA_TRY(cudaMemset(V->lines_gamma.p, 0, line_bytes)); CUDA_TRY(cudaMemset(V->lines_delta.p, 0, line_bytes));
    CUDA_TRY(cudaMemset(V->lines_beta.p, 0, line_bytes));
    LAUNCH(k_prepare_lines, 1, 32, 0, 0, V->vk.as<VkDev>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(), V->lines_beta.as<Fq2>());
    {
        const uint32_t threads = (V->n_pub + 2) * coop::kTabWindows;
        LAUNCH(k_vk_tables, (threads + 63) / 64, 64, 0, 0, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(), V->n_pub, V->tab.as<G1Affine>());
    }
    CUDA_TRY(cudaDeviceSynchronize());
    if (getenv("LZKP_COOP_SELFTEST")) {
        DBuf d_res;
        TRY(d_res.alloc(sizeof(int) + 16 * sizeof(long long)));
        CUDA_TRY(cudaMemset(d_res.p, 0, d_res.bytes));
        long long *d_st = reinterpret_cast<long long *>(d_res.as<char>() + 8);
        LAUNCH(k_coop_selftest, 1, kCoopThreads, sizeof(CoopSmem), 0, V->vk.as<VkDev>(), V->lines_gamma.as<Fq2>(), d_res.as<int>(), d_st, 0);
        int res = -1;
        long long st[10];
        CUDA_TRY(cudaMemcpy(&res, d_res.p, sizeof(int), cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemcpy(st, d_st, sizeof(st), cudaMemcpyDeviceToHost));
        fprintf(stderr, "lzkp coop selftest cycles: Miller(A,B) f chain done %lld, line chain done %lld, f chain alone %lld, prepared-line Miller %lld, "
                        "64 products %lld, final exponentiation %lld, subgroup test %lld, serial f6_inv %lld, Fq inverse %lld, 16 serial Fq2 products %lld\n",
                st[0], st[3], st[5], st[2], st[6], st[1], st[4], st[7], st[8], st[9]);
        for (int solo = 1; solo <= 2; solo++) {
            long long s2[12];
            LAUNCH(k_coop_selftest, 1, kCoopThreads, sizeof(CoopSmem), 0, V->vk.as<VkDev>(), V->lines_gamma.as<Fq2>(), d_res.as<int>(), d_st, solo);
            CUDA_TRY(cudaMemcpy(s2, d_st, sizeof(s2), cudaMemcpyDeviceToHost));
            fprintf(stderr, "lzkp coop selftest cycles, two warps only (%s): line chain done %lld, f chain done %lld (its own span %lld)\n",
                    solo == 1 ? "side by side" : "line chain first", s2[11], s2[10], s2[9]);
        }
#ifdef LZKP_COOP_PROF
        {
            long long pr[8];
            CUDA_TRY(cudaMemcpyFromSymbol(pr, coop::g_coop_prof, sizeof(pr)));
            fprintf(stderr, "lzkp coop f12_mul phases over %lld products of warp 0 (cycles each): operands %lld, Fq2 product %lld, Fq6 level %lld, Fq12 level %lld\n",
                    pr[4], pr[0] / pr[4], pr[1] / pr[4], pr[2] / pr[4], pr[3] / pr[4]);
        }
#endif
        fprintf(stderr, "lzkp coop selftest: %s (mask %d: 1 Miller(A,B), 2 final exponentiation, 4 Miller on prepared lines, 8 subgroup)\n",
                res == 0 ? "ok" : "MISMATCH", res);
        if (res != 0) return fail(LZKP_E_CUDA, "cooperative verifier self-test failed");
    }
    V->coop_ok = true;
    return LZKP_OK;
}

int vk_load(const uint8_t *bytes, size_t len, VerifyingKeyDev **out) {
    // ark-serialize VerifyingKey<Bn254>: alpha_g1, beta_g2, gamma_g2, delta_g2, Vec<gamma_abc_g1>
    if (len < 64 + 3 * 128 + 8) return fail(LZKP_E_INVALID, "verifying key: truncated");
    host::G1Canon alpha;
    host::G2Canon beta, gamma, delta;
    const uint8_t *p = bytes;
    bool ok = host::read_g1(p, alpha) && host::read_g2(p + 64, beta) && host::read_g2(p + 192, gamma) && host::read_g2(p + 320, delta);
    uint64_t cnt;
    memcpy(&cnt, p + 448, 8);
    if (!ok || cnt < 1 || cnt > (len - 456) / 64 || 456 + cnt * 64 != len) return fail(LZKP_E_INVALID, "verifying key: malformed bytes");
    std::vector<host::G1Canon> abc(cnt);
    for (uint64_t i = 0; i < cnt; i++)
        if (!host::read_g1(p + 456 + 64 * i, abc[i])) return fail(LZKP_E_INVALID, "verifying key: non-canonical coordinate");
    auto neg2 = [](host::G2Canon q) {
        if (host::is_inf(q)) return q;
        Fq m = Fq::modulus();
        host::G2Canon r = q;
        if (!q.y0.is_zero()) sub8(r.y0.l, m.l, q.y0.l);
        if (!q.y1.is_zero()) sub8(r.y1.l, m.l, q.y1.l);
        return r;
    };
    {
        DBuf d_raw, d_bad;
        TRY(d_raw.alloc(len)); TRY(d_bad.alloc(sizeof(int)));
        CUDA_TRY(cudaMemcpy(d_raw.p, bytes, len, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemset(d_bad.p, 0, sizeof(int)));
        LAUNCH(k_vk_validate, (unsigned)((cnt + 4 + 63) / 64), 64, 0, 0, d_raw.as<uint8_t>(), (uint32_t)cnt, d_bad.as<int>());
        int bad = 0;
        CUDA_TRY(cudaMemcpy(&bad, d_bad.p, sizeof(int), cudaMemcpyDeviceToHost));
        if (bad) return fail(LZKP_E_INVALID, "verifying key: " + std::to_string(bad) + " point(s) off-curve or outside the subgroup");
    }
    VerifyingKeyDev *V = new (std::nothrow) VerifyingKeyDev();
    if (!V) return fail(LZKP_E_NOMEM, "host allocation failed");
    V->n_pub = (uint32_t)cnt - 1;
    V->device = current_device();
    struct Packed { host::G1Canon alpha; host::G2Canon beta, gneg, dneg; } pk{alpha, beta, neg2(gamma), neg2(delta)};
    static_assert(sizeof(Packed) == sizeof(G1Affine) + 3 * sizeof(G2Affine), "layout");
    int rc = V->vk.alloc(sizeof(VkDev));
    if (rc == LZKP_OK) rc = upload(V->gamma_abc, abc);
    if (rc != LZKP_OK) { delete V; return rc; }
    cudaMemset(V->vk.p, 0, sizeof(VkDev));
    cudaMemcpy(V->vk.p, &pk, sizeof(pk), cudaMemcpyHostToDevice);
    k_fq_mont<<<1, 64>>>(V->vk.as<Fq>(), sizeof(pk) / 32);
    k_fq_mont<<<(unsigned)((cnt * 2 + 127) / 128), 128>>>(V->gamma_abc.as<Fq>(), cnt * 2);
    k_vk_prepare<<<1, 1>>>(V->vk.as<VkDev>());
    g_launches.fetch_add(3, std::memory_order_relaxed);
    cudaError_t e = cudaDeviceSynchronize();
    if (e != cudaSuccess) { delete V; return fail(LZKP_E_CUDA, std::string("vk_load: ") + cudaGetErrorString(e)); }
    rc = coop_prepare(V);
    if (rc != LZKP_OK) { delete V; return rc; }
    *out = V;
    return LZKP_OK;
}
void vk_free(VerifyingKeyDev *V) { delete V; }
const G2Affine *vk_delta_neg(const VerifyingKeyDev *V) {
    return reinterpret_cast<const G2Affine *>(V->vk.as<char>() + offsetof(VkDev, delta_neg));
}
uint32_t vk_num_inputs(const VerifyingKeyDev *V) { return V->n_pub; }
void vk_info(const VerifyingKeyDev *V, uint64_t info[4]) {
    info[0] = V->n_pub;
    info[1] = V->coop_ok ? V->tab.bytes : 0;     // (n_pub + 2) x 32 x 255 x 64 B; the prepared lines add 3 x 17 KB
    info[2] = V->coop_ok ? 1 : 0;          // the latency form (one proof per CTA)
    info[3] = V->coop_ok ? 1 : 0;          // the combined form with the cooperative check from 3 x SMs + 1 proofs
}

// Picks the form for n proofs and enqueues its stages on `st`, from proofs / inputs / ok in device memory.  The one
// stage sequence of both entry points; on_device selects the two places where they differ:
//   * the combined form's coefficients: 16 B per proof read from the OS and uploaded (lzkp_verify_batch), or a 256-bit
//     seed read from the OS and expanded on the device by k_rlc_rho (lzkp_verify_batch_device);
//   * groups whose combined check failed: their flags read back and their ranges re-verified from the host, or listed
//     by k_rlc_failed and re-verified by one gated launch per form (no host round trip).
// The caller holds V->mu and has made `st` wait on V->last_use.
static int enqueue_verify(VerifyingKeyDev *V, size_t n, const uint8_t *proofs, const uint8_t *inputs, size_t n_pub, uint8_t *ok,
                          cudaStream_t st, bool on_device) {
    // Calls of up to coop_max proofs are bound by ONE proof's dependent chain: there a proof gets a whole CTA whose warps
    // and lanes share the pairing's arithmetic (coop.cuh): 1 / 64 / 148 proofs in 1.8 / 1.9 / 2.2 ms with one CTA per SM,
    // 296 / 444 proofs in 2.7 / 5.2 ms with two per SM, against 5.9 ms for the random-linear-combination form at any
    // count up to ~4000 and 13.4 ms for one proof per lane: three proofs per SM is where the combined form takes over.
    int sm_count = 148;
    cudaDeviceGetAttribute(&sm_count, cudaDevAttrMultiProcessorCount, current_device() < 0 ? 0 : current_device());
    const size_t coop_max = getenv("LZKP_VERIFY_COOP_MAX") ? (size_t)atoll(getenv("LZKP_VERIFY_COOP_MAX")) : (size_t)3 * sm_count;
    // Keys above kCoopScanMax inputs: vk_x of the proofs of a range comes from k_vkx, for the latency form and k_verify4 alike.
    const bool vkx_kernel = V->coop_ok && n_pub > kCoopScanMax;
    if (vkx_kernel) TRY(grow(V, V->d_vkx, n * sizeof(G1Affine)));
    const uint32_t vkx_warps = std::min<uint32_t>(kVkxWarps, ((uint32_t)n_pub + kVkxSlice - 1) / kVkxSlice);
    const ListGate unlisted{nullptr, nullptr, 0, 0};
    auto verify_range = [&](size_t off, size_t cnt) {             // independent verification of proofs [off, off + cnt)
        const G1Affine *vkx = nullptr;
        if (vkx_kernel) {
            LAUNCH(k_vkx<false>, (unsigned)cnt, vkx_warps * 32, 0, st, V->tab.as<G1Affine>(), V->gamma_abc.as<G1Affine>(), (uint32_t)n_pub,
                   kVkxSlice, inputs + off * n_pub * 32, V->d_vkx.as<G1Affine>() + off, unlisted);
            vkx = V->d_vkx.as<G1Affine>() + off;
        }
        if (V->coop_ok && cnt <= coop_max) {
            if (cnt <= (size_t)sm_count)
                LAUNCH((k_verify_coop<1, false>), (unsigned)cnt, kCoopThreads, sizeof(CoopSmem), st, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(),
                       V->tab.as<G1Affine>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(), (uint32_t)n_pub,
                       proofs + off * 256, inputs + off * n_pub * 32, vkx, ok + off, unlisted);
            else
                LAUNCH((k_verify_coop<2, false>), (unsigned)cnt, kCoopThreads, sizeof(CoopSmem), st, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(),
                       V->tab.as<G1Affine>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(), (uint32_t)n_pub,
                       proofs + off * 256, inputs + off * n_pub * 32, vkx, ok + off, unlisted);
            return;
        }
        LAUNCH(k_verify4<false>, (unsigned)((cnt + 31) / 32), 128, 64 * sizeof(Fq12), st, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(),
               (uint32_t)n_pub, proofs + off * 256, reinterpret_cast<const Fr *>(inputs) + off * n_pub, vkx, (uint32_t)cnt, ok + off,
               unlisted);
    };
    // Above the latency form's range the random-linear-combination form takes over: 2.4x less work per proof (one Miller
    // loop instead of three, one final exponentiation per 64 proofs) and, with the cooperative combined check, a short
    // tail - 1024 / 4096 proofs in 5.9 / 6.3 ms against 13.4 / 14.0 ms for one proof per lane (k_verify4, which remains
    // the path for keys without the latency form's tables, for re-verifying large failing ranges and when the OS has no
    // entropy).
    const size_t rlc_min = getenv("LZKP_VERIFY_RLC_MIN") ? (size_t)atoll(getenv("LZKP_VERIFY_RLC_MIN")) : (V->coop_ok ? (size_t)3 * sm_count + 1 : 16384);
    if (n < rlc_min || n > 0xFFFFFFFFull) {
        static const bool timing = getenv("LZKP_VERIFY_TIMING") != nullptr;
        cudaEvent_t e0 = nullptr, e1 = nullptr;
        const bool timed = timing && !on_device;
        if (timed) { cudaEventCreate(&e0); cudaEventCreate(&e1); cudaEventRecord(e0, st); }
        verify_range(0, n);
        if (timed) {
            cudaEventRecord(e1, st); cudaEventSynchronize(e1);
            float ms = 0; cudaEventElapsedTime(&ms, e0, e1);
            fprintf(stderr, "lzkp verify_batch: %zu proofs, kernel %.3f ms (events)\n", n, ms);
            cudaEventDestroy(e0); cudaEventDestroy(e1);
        }
        return LZKP_OK;
    }
    const uint32_t ctas = (uint32_t)((n + 31) / 32), groups = (uint32_t)((n + kRlcGroup - 1) / kRlcGroup), np1 = (uint32_t)n_pub + 1;
    std::vector<uint32_t> rho(on_device ? 0 : n * 4);
    RhoSeed seed;
    if (!(on_device ? os_entropy(seed.w, sizeof(seed.w), 1) : os_entropy(rho.data(), 16, n))) {
        verify_range(0, n);                                       // no entropy source: verify independently instead
        return LZKP_OK;
    }
    TRY(grow(V, V->d_rho, n * 16)); TRY(grow(V, V->d_f, n * sizeof(Fq12))); TRY(grow(V, V->d_rc, n * sizeof(G1XYZZ)));
    static const bool tail_lanes = getenv("LZKP_RLC_TAIL_LANES") != nullptr;      // A/B switch: the lane-per-group tail
    // Keys above kCoopScanMax inputs: the scalar sums per (group, input) in k_rlc_input_sums, not in the per-proof kernel.  At
    // 2049 inputs (B200, 1000 W) the per-proof kernel's sums strand outlasts its Miller loop: k_rlc_prepare 5.83 against
    // 3.97 ms at 445 proofs, 6.89 against 4.12 at 4096; k_rlc_input_sums itself takes 0.04 / 0.18 ms.
    const bool input_sums = V->coop_ok && !tail_lanes && n_pub > kCoopScanMax;
    if (!input_sums) TRY(grow(V, V->d_sx, (size_t)ctas * np1 * sizeof(Fr)));
    TRY(grow(V, V->d_gF, (size_t)groups * sizeof(Fq12))); TRY(grow(V, V->d_gC, (size_t)groups * sizeof(G1XYZZ)));
    TRY(grow(V, V->d_gS, (size_t)groups * np1 * sizeof(Fr))); TRY(grow(V, V->d_gX, (size_t)groups * (np1 + 1) * sizeof(G1XYZZ)));
    TRY(grow(V, V->d_gok, groups));
    if (on_device) {
        TRY(grow(V, V->d_list, (n + 1) * sizeof(uint32_t)));
        LAUNCH(k_rlc_rho, (unsigned)(((n + 3) / 4 + 127) / 128), 128, 0, st, seed, (uint32_t)n, V->d_rho.as<uint32_t>());
    } else {
        CUDA_TRY(cudaMemcpy(V->d_rho.p, rho.data(), n * 16, cudaMemcpyHostToDevice));
    }
    // One launch per stage for the whole batch.  (Measured: cutting the batch into 16 384-proof chunks so that a chunk's
    // tail runs under the next chunk's k_rlc_prepare on a second stream is SLOWER - 98 to 108 ms against 81 ms at 65 536
    // proofs: the per-proof kernel is a latency-bound chain per CTA, and four 512-CTA launches fill whole waves worse
    // than one 2048-CTA launch.)
    // Up to one resident wave of the four-role kernel (2 CTAs of 32 proofs per SM at 255 registers: 9472 proofs on 148 SMs)
    // a call is bound by ONE CTA's chain and the role warps shorten it (8192 proofs: 11.2 against 12.7 ms); beyond, work per
    // resident warp decides (16 384: 18.7 against 13.6 ms, 65 536: 67.3 against 46.4 ms).  LZKP_RLC_PREPARE_ROLES=1/0 forces one.
    const char *force = getenv("LZKP_RLC_PREPARE_ROLES");
    // (a 128-register build of the role kernel, four CTAs per SM, for calls of up to two of these waves: 15.0 - 19.0 ms against
    // 13.3 - 13.7 ms for the sequential kernel at 12 288 - 18 944 proofs - rejected)
    const bool prep_roles = force ? atoi(force) != 0 : n <= (size_t)sm_count * 2 * 32;
    Fr *sx = input_sums ? nullptr : V->d_sx.as<Fr>();
    const Fr *x = reinterpret_cast<const Fr *>(inputs);
    if (prep_roles)
        LAUNCH(k_rlc_prepare, ctas, 128, 32 * (sizeof(Fq12) + sizeof(G1Affine)), st, V->vk.as<VkDev>(), (uint32_t)n_pub, proofs, x, V->d_rho.as<uint32_t>(),
               (uint32_t)n, V->d_f.as<Fq12>(), V->d_rc.as<G1XYZZ>(), sx, ok);
    else
        LAUNCH(k_rlc_prepare_seq, (ctas + 1) / 2, 64, 0, st, V->vk.as<VkDev>(), (uint32_t)n_pub, proofs, x,
               V->d_rho.as<uint32_t>(), (uint32_t)n, V->d_f.as<Fq12>(), V->d_rc.as<G1XYZZ>(), sx, ok);
    if (V->coop_ok && !tail_lanes) {
        if (input_sums)
            LAUNCH(k_rlc_input_sums, dim3(groups, (np1 + 127) / 128), 128, 0, st, x, V->d_rho.as<uint32_t>(), ok,
                   (uint32_t)n, (uint32_t)n_pub, V->d_gS.as<Fr>());
        else
            LAUNCH(k_rlc_scalars, (groups * np1 + 127) / 128, 128, 0, st, V->d_sx.as<Fr>(), (uint32_t)n, (uint32_t)n_pub, groups, V->d_gS.as<Fr>());
        LAUNCH(k_rlc_inputs2, (groups * (np1 + 1) + 3) / 4, 128, 0, st, V->d_gS.as<Fr>(), V->tab.as<G1Affine>(), (uint32_t)n_pub, groups,
               V->d_gX.as<G1XYZZ>());
        if (groups <= 2u * (uint32_t)sm_count)
            LAUNCH(k_rlc_tail_coop<2>, groups, 128, sizeof(TailSmem), st, V->vk.as<VkDev>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(),
                   V->lines_beta.as<Fq2>(), V->d_f.as<Fq12>(), V->d_rc.as<G1XYZZ>(), V->d_gX.as<G1XYZZ>(), (uint32_t)n, (uint32_t)n_pub,
                   V->d_gok.as<uint8_t>());
        else
            LAUNCH(k_rlc_tail_coop<4>, groups, 128, sizeof(TailSmem), st, V->vk.as<VkDev>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(),
                   V->lines_beta.as<Fq2>(), V->d_f.as<Fq12>(), V->d_rc.as<G1XYZZ>(), V->d_gX.as<G1XYZZ>(), (uint32_t)n, (uint32_t)n_pub,
                   V->d_gok.as<uint8_t>());
    } else {
    LAUNCH(k_rlc_reduce, (groups + 63) / 64, 64, 0, st, V->d_f.as<Fq12>(), V->d_rc.as<G1XYZZ>(), V->d_sx.as<Fr>(), (uint32_t)n,
           (uint32_t)n_pub, groups, V->d_gF.as<Fq12>(), V->d_gC.as<G1XYZZ>(), V->d_gS.as<Fr>());
    LAUNCH(k_rlc_inputs, (groups * np1 + 63) / 64, 64, 0, st, V->d_gS.as<Fr>(), V->gamma_abc.as<G1Affine>(), (uint32_t)n_pub, groups,
           V->d_gX.as<G1XYZZ>());
    LAUNCH(k_rlc_tail, (groups + 31) / 32, 128, 96 * sizeof(Fq12), st, V->vk.as<VkDev>(), V->d_gF.as<Fq12>(), V->d_gC.as<G1XYZZ>(),
           V->d_gS.as<Fr>(), V->d_gX.as<G1XYZZ>(), (uint32_t)n_pub, groups, V->d_gok.as<uint8_t>());
    }
    if (on_device) {
        // The failing groups' proofs, listed on the device, are re-verified by the form the host path would pick for
        // their count F: one launch per form sized for its largest F, whose CTAs leave unless F is in that form's range.
        uint32_t *list = V->d_list.as<uint32_t>(), *count = list + n;
        LAUNCH(k_rlc_failed, 1, kFailedThreads, 0, st, V->d_gok.as<uint8_t>(), (uint32_t)n, groups, list, count);
        const G1Affine *vkx = nullptr;
        if (vkx_kernel) {
            LAUNCH(k_vkx<true>, (unsigned)n, vkx_warps * 32, 0, st, V->tab.as<G1Affine>(), V->gamma_abc.as<G1Affine>(), (uint32_t)n_pub,
                   kVkxSlice, inputs, V->d_vkx.as<G1Affine>(), ListGate{list, count, 0, 0xFFFFFFFFu});
            vkx = V->d_vkx.as<G1Affine>();
        }
        const uint32_t cmax = V->coop_ok ? (uint32_t)std::min<size_t>(coop_max, n) : 0, one = std::min<uint32_t>(cmax, sm_count);
        if (one)
            LAUNCH((k_verify_coop<1, true>), one, kCoopThreads, sizeof(CoopSmem), st, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(),
                   V->tab.as<G1Affine>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(), (uint32_t)n_pub, proofs, inputs, vkx, ok,
                   ListGate{list, count, 0, one});
        if (cmax > (uint32_t)sm_count)
            LAUNCH((k_verify_coop<2, true>), cmax, kCoopThreads, sizeof(CoopSmem), st, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(),
                   V->tab.as<G1Affine>(), V->lines_gamma.as<Fq2>(), V->lines_delta.as<Fq2>(), (uint32_t)n_pub, proofs, inputs, vkx, ok,
                   ListGate{list, count, (uint32_t)sm_count, cmax});
        if (n > cmax)
            LAUNCH(k_verify4<true>, (unsigned)((n + 31) / 32), 128, 64 * sizeof(Fq12), st, V->vk.as<VkDev>(), V->gamma_abc.as<G1Affine>(),
                   (uint32_t)n_pub, proofs, x, vkx, (uint32_t)n, ok, ListGate{list, count, cmax, 0xFFFFFFFFu});
        return LZKP_OK;
    }
    std::vector<uint8_t> gok(groups);
    CUDA_TRY(cudaMemcpy(gok.data(), V->d_gok.p, groups, cudaMemcpyDeviceToHost));
    // groups whose combined check failed hold at least one false proof: decide those proofs one by one
    // (adjacent failing groups are merged into one launch; the well-formedness flags of k_rlc_prepare stand for the rest)
    for (uint32_t g = 0; g < groups;) {
        if (gok[g]) { g++; continue; }
        uint32_t h = g;
        while (h < groups && !gok[h]) h++;
        const size_t off = (size_t)g * kRlcGroup, end = std::min<size_t>(n, (size_t)h * kRlcGroup);
        verify_range(off, end - off);
        g = h;
    }
    return LZKP_OK;
}

// Waits on the key's last use in `st`, enqueues the call and records the last use, even when the enqueue failed halfway.
static int enqueue_ordered(VerifyingKeyDev *V, size_t n, const uint8_t *proofs, const uint8_t *inputs, size_t n_pub, uint8_t *ok,
                           cudaStream_t st, bool on_device) {
    TRY(event_acquire(V->last_use, st));
    const int rc = enqueue_verify(V, n, proofs, inputs, n_pub, ok, st, on_device);
    TRY(event_release(V->last_use, st));
    return rc;
}

int verify_batch(VerifyingKeyDev *V, size_t n, const uint8_t *proofs, const uint8_t *inputs, size_t n_pub, uint8_t *ok_out) {
    std::lock_guard<std::mutex> lk(V->mu);
    if (n_pub != V->n_pub) {                   // wrong number of public inputs: nothing verifies (reference: Err -> false)
        memset(ok_out, 0, n);
        return LZKP_OK;
    }
    if (n == 0) return LZKP_OK;
    DBuf &d_p = V->d_p, &d_x = V->d_x, &d_ok = V->d_ok;
    TRY(grow(V, d_p, n * 256)); TRY(grow(V, d_x, n * std::max<size_t>(n_pub, 1) * 32)); TRY(grow(V, d_ok, n));
    CUDA_TRY(cudaMemcpy(d_p.p, proofs, n * 256, cudaMemcpyHostToDevice));
    if (n_pub) CUDA_TRY(cudaMemcpy(d_x.p, inputs, n * n_pub * 32, cudaMemcpyHostToDevice));
    TRY(enqueue_ordered(V, n, d_p.as<uint8_t>(), d_x.as<uint8_t>(), n_pub, d_ok.as<uint8_t>(), 0, false));
    CUDA_TRY(cudaMemcpy(ok_out, d_ok.p, n, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

// Device memory of the key's device, not host memory (cudaPointerGetAttributes: unregistered or pinned host memory).
int check_device_buffer(const VerifyingKeyDev *V, const void *p, const char *what) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return fail(LZKP_E_INVALID, std::string(what) + ": not a CUDA pointer");
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != V->device)
        return fail(LZKP_E_INVALID, std::string(what) + ": not device memory of the key's device");
    return LZKP_OK;
}

int verify_batch_device(VerifyingKeyDev *V, size_t n, const uint8_t *d_proofs, const uint8_t *d_inputs, size_t n_pub, uint8_t *d_ok,
                        cudaStream_t st) {
    // A graph replay would reuse the coefficients drawn at capture: refuse capture rather than weaken the combined check.
    cudaStreamCaptureStatus capturing = cudaStreamCaptureStatusNone;
    CUDA_TRY(cudaStreamIsCapturing(st, &capturing));
    if (capturing != cudaStreamCaptureStatusNone)
        return fail(LZKP_E_UNSUPPORTED, "lzkp_verify_batch_device: stream capture is not supported (coefficients are drawn per call)");
    if (n == 0) return LZKP_OK;
    // the kernels read proofs and inputs with 128-bit loads
    if ((reinterpret_cast<uintptr_t>(d_proofs) | reinterpret_cast<uintptr_t>(d_inputs)) & 15)
        return fail(LZKP_E_INVALID, "lzkp_verify_batch_device: proofs and public inputs must be 16-byte aligned");
    TRY(check_device_buffer(V, d_proofs, "proofs"));
    if (n_pub) TRY(check_device_buffer(V, d_inputs, "public inputs"));
    TRY(check_device_buffer(V, d_ok, "ok"));
    if (n_pub != V->n_pub) {                   // wrong number of public inputs: nothing verifies
        CUDA_TRY(cudaMemsetAsync(d_ok, 0, n, st));
        return LZKP_OK;
    }
    std::lock_guard<std::mutex> lk(V->mu);
    TRY(enqueue_ordered(V, n, d_proofs, d_inputs, n_pub, d_ok, st, true));
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

}  // namespace eng
}  // namespace lzkp
