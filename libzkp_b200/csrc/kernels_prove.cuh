// kernels.cuh — device kernels of the batched Groth16/BN254 prover (sm_100a).
//
// What each kernel replaces in the reference's prover (all [UPSTREAM] ark-groth16 /
// ark-poly / ark-ec code reached from src/backend/snark.rs:364 and :442; SURVEY §8a):
//   k_witgen_equality / k_witgen_membership  a2  generate_constraints' assignment (snark.rs:263-290, 515-584)
//   k_spmv_abc                               a3  witness_map_from_matrices: A.z, B.z, C.z rows
//   k_ntt_icoset                             a4+a5  ifft_in_place, then coset fft_in_place
//   k_ntt_final                              a6+a7  (ab - c) / Z(g), coset ifft_in_place -> h
//   k_digits                                 into_bigint + signed window recoding of MSM scalars
//   k_tb_*                                   (pk load) fixed-base window tables, the resident form of a16
//   k_msm_batch / k_msm_reduce               a8-a12 the five MSMs, as table gathers + XYZZ mixed adds
//   k_assemble                               a13-a15 proof assembly, into_affine, serialize_uncompressed
#pragma once
#include "dev_util.cuh"

namespace lzkp {

// ---------------------------------------------------------------- constant tables
// out[k] = scale * base^e(k), e(k) = bitrev(k) if log_rev else k.  All Montgomery unless
// `scale` itself is given in canonical form (then the products come out canonical-scaled).
__global__ void k_pow_table(Fr *out, Fr base, Fr scale, uint32_t count, uint32_t log_rev) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    uint32_t e = log_rev ? bitrev(k, log_rev) : k;
    Fr acc = Fr::one(), b = base;
    while (e) {
        if (e & 1u) acc = acc * b;
        b = b.sqr();
        e >>= 1;
    }
    st_vec(out + k, acc * scale);
}
// in-place canonical -> val * R^2 (so that val (*) canonical_z is the Montgomery form of coeff*z)
__global__ void k_to_r2_form(Fr *v, uint32_t count) {
    uint32_t k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    Fr r3;
#pragma unroll
    for (int i = 0; i < 8; i++) r3.l[i] = FrParams::R3(i);
    st_vec(v + k, ld_vec(v + k) * r3);
}
// canonical <-> Montgomery for arrays of base-field elements (points are 2 or 4 Fq each)
__global__ void k_fq_to_mont(Fq *v, size_t count) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    st_vec(v + k, Fq::from_canonical(ld_vec(v + k)));
}

// ---------------------------------------------------------------- witness generation
// MiMC-5 round constants (Montgomery), filled by the host from SHA-256 (snark.rs:186-198).
__constant__ Fr c_mimc[110];

// z = [1, commitment, a, b, (t^2, t^4, t^5) x rounds], canonical (snark.rs:263-290).
// If commit_in is null the commitment is MiMC5(a) computed here (commit_value_snark).
// status[p] = 1 when a != b (prove_equality_zk returns an empty Vec, snark.rs:344).
__global__ void k_witgen_equality(const uint64_t *a, const uint64_t *b, const Fr *commit_in, Fr *z, Fr *commit_out,
                                  int32_t *status, uint32_t P, uint32_t rounds, uint32_t nv) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    if (a[p] != b[p]) status[p] = 1;
    Fr *zp = z + (size_t)p * nv;
    Fr one = Fr::zero();
    one.l[0] = 1;
    st_vec(zp + 0, one);
    st_vec(zp + 2, fr_from_u64(a[p]));
    st_vec(zp + 3, fr_from_u64(b[p]));
    Fr x = Fr::from_canonical(fr_from_u64(a[p]));
    for (uint32_t i = 0; i < rounds; i++) {
        Fr t = x + c_mimc[i % 110];
        Fr t2 = t.sqr(), t4 = t2.sqr();
        x = t4 * t;
        st_vec(zp + 4 + 3 * i, t2);           // Montgomery form: k_wires_to_canonical converts the wires in parallel,
        st_vec(zp + 5 + 3 * i, t4);           // off this thread's serial chain of 3 products per round
        st_vec(zp + 6 + 3 * i, x);
    }
    Fr cm = commit_in ? ld_vec(commit_in + p) : x.to_canonical();
    st_vec(zp + 1, cm);
    if (commit_out) st_vec(commit_out + p, cm);
}

// z[p][first .. first + count) : Montgomery -> canonical (the MiMC wires the witness kernels leave in Montgomery form)
__global__ void __launch_bounds__(128) k_wires_to_canonical(Fr *z, uint32_t P, uint32_t nv, uint32_t first, uint32_t count) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (size_t)P * count) return;
    Fr *e = z + (i / count) * nv + first + (uint32_t)(i % count);
    st_vec(e, ld_vec(e).to_canonical());
}

// z = [1, commitment, set[S], is_real[S], value, 330 MiMC wires, sel[S], sel*(1-is_real)[S],
//      sel*(value-set)[S]] (snark.rs:515-584; padding and selector as snark.rs:420-427).
// status[p] = 2 when the set is empty / too long / does not contain value (snark.rs:406,415-418).
__global__ void k_witgen_membership(const uint64_t *value, const uint64_t *sets, const uint32_t *set_len,
                                    uint32_t set_stride, const Fr *commit_in, Fr *z, Fr *commit_out, int32_t *status,
                                    uint32_t P, uint32_t S, uint32_t nv) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    Fr *zp = z + (size_t)p * nv;
    const uint64_t *set = sets + (size_t)p * set_stride;
    uint32_t len = set_len[p];
    uint64_t v = value[p];
    uint32_t pos = 0xffffffffu;
    if (len >= 1 && len <= S && len <= set_stride)      // a row is set_stride wide: a longer claimed length is rejected, never read
        for (uint32_t i = 0; i < len; i++)
            if (set[i] == v) { pos = i; break; }
    if (pos == 0xffffffffu) { status[p] = 2; len = 0; }
    Fr one = Fr::zero(), zero = Fr::zero();
    one.l[0] = 1;
    st_vec(zp + 0, one);
    for (uint32_t i = 0; i < S; i++) {
        st_vec(zp + 2 + i, i < len ? fr_from_u64(set[i]) : zero);
        st_vec(zp + 2 + S + i, i < len ? one : zero);
    }
    const uint32_t w0 = 2 + 2 * S;          // first witness column
    st_vec(zp + w0, fr_from_u64(v));
    Fr x = Fr::from_canonical(fr_from_u64(v));
    for (uint32_t i = 0; i < 110; i++) {
        Fr t = x + c_mimc[i];
        Fr t2 = t.sqr(), t4 = t2.sqr();
        x = t4 * t;
        st_vec(zp + w0 + 1 + 3 * i, t2);      // Montgomery form, see k_wires_to_canonical
        st_vec(zp + w0 + 2 + 3 * i, t4);
        st_vec(zp + w0 + 3 + 3 * i, x);
    }
    Fr cm = commit_in ? ld_vec(commit_in + p) : x.to_canonical();
    st_vec(zp + 1, cm);
    if (commit_out) st_vec(commit_out + p, cm);
    const uint32_t s0 = w0 + 331;
    Fr r = Fr::modulus();
    for (uint32_t i = 0; i < S; i++) {
        bool sel = (i == pos);
        st_vec(zp + s0 + i, sel ? one : zero);
        // sel * (1 - is_real): selected slots are always real
        st_vec(zp + s0 + S + i, zero);
        // sel * (value - set[i]) mod r (zero for the honest selector; kept general)
        Fr d = zero;
        if (sel) {
            Fr sv = fr_from_u64(i < len ? set[i] : 0), vv = fr_from_u64(v), t;
            uint32_t bw = sub8(t.l, vv.l, sv.l);
            if (bw) add8(d.l, t.l, r.l); else d = t;
        }
        st_vec(zp + s0 + 2 * S + i, d);
    }
}

// ---------------------------------------------------------------- witness map
struct CsrDev {
    const uint32_t *rowptr;
    const uint32_t *col;
    const Fr *val;              // coefficient * R^2 mod r
};

__device__ __forceinline__ Fr spmv_row(const CsrDev &M, uint32_t row, const Fr *z) {
    Fr acc = Fr::zero();
    uint32_t lo = __ldg(M.rowptr + row), hi = __ldg(M.rowptr + row + 1);
    for (uint32_t t = lo; t < hi; t++) acc = acc + ldg_vec(M.val + t) * ld_vec(z + __ldg(M.col + t));
    return acc;
}
// abc[k][p][i], k = 0 (a), 1 (b), 2 (c); rows m..m+n_inst of a carry the instance (input consistency).
__global__ void __launch_bounds__(128) k_spmv_abc(CsrDev A, CsrDev B, CsrDev C, const Fr *z, Fr *abc, uint32_t P,
                                                  uint32_t nv, uint32_t m, uint32_t n_inst, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x, p = blockIdx.y;
    if (i >= n) return;
    const Fr *zp = z + (size_t)p * nv;
    Fr a = Fr::zero(), b = Fr::zero(), c = Fr::zero();
    if (i < m) {
        a = spmv_row(A, i, zp);
        b = spmv_row(B, i, zp);
        c = spmv_row(C, i, zp);
    } else if (i < m + n_inst) {
        a = Fr::from_canonical(ld_vec(zp + (i - m)));
    }
    size_t plane = (size_t)P * n, off = (size_t)p * n + i;
    st_vec(abc + off, a);
    st_vec(abc + plane + off, b);
    st_vec(abc + 2 * plane + off, c);
}

// Shared-memory radix-2 NTT on two 128-bit planes (conflict-free LDS.128 / STS.128).
struct SmemPoly {
    uint4 *lo, *hi;
    __device__ __forceinline__ Fr get(uint32_t i) const {
        Fr r;
        uint4 a = lo[i], b = hi[i];
        r.l[0] = a.x; r.l[1] = a.y; r.l[2] = a.z; r.l[3] = a.w;
        r.l[4] = b.x; r.l[5] = b.y; r.l[6] = b.z; r.l[7] = b.w;
        return r;
    }
    __device__ __forceinline__ void put(uint32_t i, const Fr &v) const {
        lo[i] = make_uint4(v.l[0], v.l[1], v.l[2], v.l[3]);
        hi[i] = make_uint4(v.l[4], v.l[5], v.l[6], v.l[7]);
    }
};
// natural order in -> bit-reversed out (Gentleman-Sande); tw[k] = w^k, k < n/2
__device__ __forceinline__ void ntt_dif(const SmemPoly &s, uint32_t log_n, const Fr *tw) {
    const uint32_t n = 1u << log_n;
    for (uint32_t lh = log_n; lh-- > 0;) {
        const uint32_t h = 1u << lh;
        for (uint32_t bf = threadIdx.x; bf < n / 2; bf += blockDim.x) {
            uint32_t k = bf & (h - 1), i = ((bf >> lh) << (lh + 1)) | k;
            Fr x = s.get(i), y = s.get(i + h);
            s.put(i, x + y);
            Fr d = x - y;
            s.put(i + h, lh == 0 ? d : d * ldg_vec(tw + (k << (log_n - 1 - lh))));
        }
        __syncthreads();
    }
}
// bit-reversed in -> natural order out (Cooley-Tukey)
__device__ __forceinline__ void ntt_dit(const SmemPoly &s, uint32_t log_n, const Fr *tw) {
    const uint32_t n = 1u << log_n;
    for (uint32_t lh = 0; lh < log_n; lh++) {
        const uint32_t h = 1u << lh;
        for (uint32_t bf = threadIdx.x; bf < n / 2; bf += blockDim.x) {
            uint32_t k = bf & (h - 1), i = ((bf >> lh) << (lh + 1)) | k;
            Fr x = s.get(i), y = s.get(i + h);
            if (lh != 0) y = y * ldg_vec(tw + (k << (log_n - 1 - lh)));
            s.put(i, x + y);
            s.put(i + h, x - y);
        }
        __syncthreads();
    }
}
struct NttTables {
    const Fr *tw_fwd;      // w^k,  k < n/2 (Montgomery)
    const Fr *tw_inv;      // w^-k
    const Fr *coset_br;    // n^-1 * g^bitrev(k)        (Montgomery)
    const Fr *uncoset_br;  // n^-1 * g^-bitrev(k), stored in CANONICAL form so products leave the Montgomery domain
    const Fr *ninv_br;     // n^-1 replicated is not needed; plain inverse uses ninv below
    Fr ninv;               // n^-1 (Montgomery)
    Fr zinv;               // (g^n - 1)^-1 (Montgomery)
};
// poly (evaluations on the domain) -> evaluations on the coset g*H:  iNTT, *g^i/n, NTT.  grid (P, 3)
__global__ void k_ntt_icoset(Fr *abc, NttTables T, uint32_t P, uint32_t log_n) {
    extern __shared__ uint4 smem[];
    const uint32_t n = 1u << log_n;
    SmemPoly s{smem, smem + n};
    Fr *poly = abc + ((size_t)blockIdx.y * P + blockIdx.x) * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s.put(i, ld_vec(poly + i));
    __syncthreads();
    ntt_dif(s, log_n, T.tw_inv);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s.put(i, s.get(i) * ldg_vec(T.coset_br + i));
    __syncthreads();
    ntt_dit(s, log_n, T.tw_fwd);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) st_vec(poly + i, s.get(i));
}
// h = coset_iNTT((a*b - c) * zinv), canonical output.  grid (P)
__global__ void k_ntt_final(const Fr *abc, Fr *h, NttTables T, uint32_t P, uint32_t log_n) {
    extern __shared__ uint4 smem[];
    const uint32_t n = 1u << log_n;
    SmemPoly s{smem, smem + n};
    const size_t plane = (size_t)P * n, off = (size_t)blockIdx.x * n;
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
        Fr a = ld_vec(abc + off + i), b = ld_vec(abc + plane + off + i), c = ld_vec(abc + 2 * plane + off + i);
        s.put(i, (a * b - c) * T.zinv);
    }
    __syncthreads();
    ntt_dif(s, log_n, T.tw_inv);
    for (uint32_t i = threadIdx.x; i < n; i += blockDim.x)
        st_vec(h + off + bitrev(i, log_n), s.get(i) * ldg_vec(T.uncoset_br + i));
}
// Stand-alone transform for lzkp_ntt on n <= 4096: canonical in/out, any of the 4 variants.  grid (count)
__global__ void k_ntt_small(Fr *data, NttTables T, uint32_t log_n, int inverse, int coset) {
    extern __shared__ uint4 smem[];
    const uint32_t n = 1u << log_n;
    SmemPoly s{smem, smem + n};
    Fr *poly = data + (size_t)blockIdx.x * n;
    Fr one_c = Fr::zero();
    one_c.l[0] = 1;
    if (!inverse) {
        // natural load; coset pre-scale g^i = n * coset_br[bitrev(i)]; DIF -> bit-reversed, store un-reversed
        Fr nn = T.ninv.inverse();
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            Fr v = Fr::from_canonical(ld_vec(poly + i));
            if (coset) v = v * ldg_vec(T.coset_br + bitrev(i, log_n)) * nn;
            s.put(i, v);
        }
        __syncthreads();
        ntt_dif(s, log_n, T.tw_fwd);
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) st_vec(poly + bitrev(i, log_n), s.get(i).to_canonical());
    } else {
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) s.put(i, Fr::from_canonical(ld_vec(poly + i)));
        __syncthreads();
        ntt_dif(s, log_n, T.tw_inv);
        for (uint32_t i = threadIdx.x; i < n; i += blockDim.x) {
            Fr v = s.get(i);
            v = coset ? v * ldg_vec(T.uncoset_br + i) : (v * T.ninv).to_canonical();
            st_vec(poly + bitrev(i, log_n), v);
        }
    }
}

// Large-domain witness map helpers (the transforms themselves are ntt_large.cu's tiled passes).
// hq[i] = (a[i] * b[i] - c[i]) * zinv on the coset (Montgomery in / out)
__global__ void k_pointwise_h(const Fr *a, const Fr *b, const Fr *c, Fr *hq, Fr zinv, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st_vec(hq + i, (ld_vec(a + i) * ld_vec(b + i) - ld_vec(c + i)) * zinv);
}
__global__ void k_fr_to_canonical(Fr *v, size_t n) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    st_vec(v + i, ld_vec(v + i).to_canonical());
}
// status[0] = 1 when any of the count scalars is not canonical (>= r)
__global__ void k_check_canonical(const Fr *v, uint32_t count, int32_t *status) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    if (!fr_is_canonical(ld_vec(v + i))) status[0] = 1;
}

// ---------------------------------------------------------------- scalar recoding
// Signed c-bit digits via the offset trick: s' = s + K, K = sum_w 2^(c*w + c-1); the unsigned
// windows u_w of s' give d_w = u_w - 2^(c-1) in [-2^(c-1), 2^(c-1)), independently per window.
// dig[(row * W + w) * P + p].  grid (ceil(P/128), count), row = row0 + blockIdx.y.
// DigT: int16_t for c <= 16 (half the digit traffic: the digit matrix of a 4096-proof batch then stays in L2), int32_t for c = 17.
template <class DigT>
__global__ void __launch_bounds__(128) k_digits(const Fr *scalars, uint32_t stride, uint32_t first, DigT *dig,
                                                uint32_t row0, uint32_t P, uint32_t c, uint32_t W, int32_t *status,
                                                uint32_t count) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    for (uint32_t j = blockIdx.y; j < count; j += gridDim.y) {       // rows beyond the grid's y limit: stride loop
        Fr s = ld_vec(scalars + (size_t)p * stride + first + j);
        if (!fr_is_canonical(s)) {
            status[p] = 1;                  // non-canonical input: the reference's deserializer rejects it
            s = Fr::zero();
        }
        uint32_t v[10];
        recode_offset(s, c, W, v);
        const size_t base = ((size_t)(row0 + j) * W) * P + p;
        for (uint32_t w = 0; w < W; w++) dig[base + (size_t)w * P] = (DigT)recoded_digit(v, c, w);
    }
}
// Digits of scalars[p][first + j] * mult[p] mod r (canonical in): the rows s * z_i and r * z_i of the latency form.
template <class DigT>
__global__ void __launch_bounds__(128) k_digits_scaled(const Fr *scalars, uint32_t stride, uint32_t first, const Fr *mult,
                                                       DigT *dig, uint32_t row0, uint32_t P, uint32_t c, uint32_t W,
                                                       uint32_t count) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    Fr m = ld_vec(mult + p);
    if (!fr_is_canonical(m)) m = Fr::zero();               // (k_digits flags the proof; here only keep the arithmetic defined)
    const Fr mr2 = m * Fr::r2();                            // Montgomery form of mult: (z * mR) R^-1 = z * mult, canonical
    for (uint32_t j = blockIdx.y; j < count; j += gridDim.y) {
        Fr z = ld_vec(scalars + (size_t)p * stride + first + j);
        if (!fr_is_canonical(z)) z = Fr::zero();
        const Fr s = z * mr2;
        uint32_t v[10];
        recode_offset(s, c, W, v);
        const size_t base = ((size_t)(row0 + j) * W) * P + p;
        for (uint32_t w = 0; w < W; w++) dig[base + (size_t)w * P] = (DigT)recoded_digit(v, c, w);
    }
}
// rs[p] = r[p] * s[p] mod r, canonical in / out
__global__ void k_fr_mul_canonical(const Fr *r, const Fr *s, Fr *rs, uint32_t P) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= P) return;
    st_vec(rs + p, (ld_vec(r + p) * ld_vec(s + p)) * Fr::r2());
}

// ---------------------------------------------------------------- assembly + serialization
struct ProofConsts {
    G1Affine a0;        // alpha_g1 + a_query[0]
    G1Affine b0;        // beta_g1 + b_g1_query[0]
    G2Affine b2;        // beta_g2 + b_g2_query[0]
};
// g1[q * P + p]: q = 0 A-sum (incl. r*delta), 1 B1-sum (incl. s*delta), 2 L-sum (incl. -rs*delta), 3 H-sum,
// 4 the terms the A and B1 sums share (variables whose A and B1 query points are the same point): A = q0 + q4, B1 = q1 + q4.
// The stage is a chain of dependent field products per proof (two variable-base scalar multiplications,
// three inversions), so it is latency-bound.  Its independent strands run on six warps of the CTA
// (warp-uniform roles, lane = proof) and meet once in shared memory; each scalar multiplication is split by
// the GLV endomorphism into two 128-bit ladders (k = +-k1 +- k2 lambda, phi(P) = (beta x, y)):
//   warp 0: k1(s) * A, then C = s*A + r*B1 + L + H -> affine -> bytes      warp 4: A -> affine -> bytes
//   warp 1: k2(s) * phi(A)     warp 2: k1(r) * B1     warp 3: k2(r) * phi(B1)     warp 5: B (G2) -> affine -> bytes
__device__ __forceinline__ G1XYZZ glv_half(const G1XYZZ &P, const Fr &k, int half) {
    GlvSplit sp = glv_split(k);
    if (!sp.ok) return half == 0 ? scalar_mul(P, k) : G1XYZZ::inf();
    G1XYZZ Q = P;
    if (half == 1) {
        Fq beta;
#pragma unroll
        for (int i = 0; i < 8; i++) beta.l[i] = FqParams::BETA(i);
        Q.x = Q.x * beta;
    }
    if (half == 0 ? sp.neg1 : sp.neg2) Q.y = Q.y.neg();
    return half == 0 ? scalar_mul_u128(Q, sp.k1) : scalar_mul_u128(Q, sp.k2);
}
// Four warps per 32 proofs, one per SM partition: warp w runs GLV strand w of C = s*A + r*B1 + ... (the long serial
// chain), then warp 0 sums the strands and converts C, while warps 1 and 2 convert A and B (short) beside it.
__global__ void __launch_bounds__(128) k_assemble(const G1XYZZ *g1, const G2XYZZ *g2, ProofConsts K, const Fr *r,
                                                  const Fr *s, uint32_t P, uint8_t *proofs) {
    __shared__ uint4 sm_raw[3 * 32 * sizeof(G1XYZZ) / 16];
    G1XYZZ *sm = reinterpret_cast<G1XYZZ *>(sm_raw);
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31, p = blockIdx.x * 32 + lane;
    const bool live = p < P;
    uint8_t *out = proofs + (size_t)p * 256;
    G1XYZZ acc = G1XYZZ::inf(), A = G1XYZZ::inf();
    if (live) {
        if (role <= 1) {
            A = ld_vec(g1 + p);
            A.add_cold(ld_vec(g1 + 4 * (size_t)P + p));
            A.madd_cold(K.a0);
            if (role == 0) acc = glv_half(A, ld_vec(s + p), 0);
            else st_vec(sm + lane, glv_half(A, ld_vec(s + p), 1));
        } else {
            G1XYZZ B1 = ld_vec(g1 + (size_t)P + p);
            B1.add_cold(ld_vec(g1 + 4 * (size_t)P + p));
            B1.madd_cold(K.b0);
            st_vec(sm + (role - 1) * 32 + lane, glv_half(B1, ld_vec(r + p), role - 2));
        }
    }
    __syncthreads();
    if (!live) return;
    if (role == 0) {
        acc.add_cold(ld_vec(sm + lane));
        acc.add_cold(ld_vec(sm + 32 + lane));
        acc.add_cold(ld_vec(sm + 64 + lane));
        acc.add_cold(ld_vec(g1 + 2 * (size_t)P + p));
        acc.add_cold(ld_vec(g1 + 3 * (size_t)P + p));
        write_g1(out + 192, acc.to_affine());
    } else if (role == 1) {
        write_g1(out, A.to_affine());
    } else if (role == 2) {
        G2XYZZ B2 = ld_vec(g2 + p);
        B2.madd_cold(K.b2);
        write_g2(out + 64, B2.to_affine());
    }
}

// One large proof (P = 1).  C = s*A + r*B1 + L + H needs neither B1 itself nor a variable-base multiplication after the
// MSMs: the B1 MSM runs on the scalars r * z_i (k_scalars_times), so slot 1 IS r * (B1-sum), and
//     slot 4 <- s * (slot 0 [+ alpha + a_0]) [+ r * (beta + b_0)]
// runs here as soon as the A-sum exists, beside the remaining MSMs: the GLV strands of s * A on warps 0 and 1, those
// of the constant term on warps 2 and 3 (with_consts: the shard whose sums carry the key's constant terms).  The
// first version ran s*A + r*B1 after everything else: 0.83 ms of serial chain at the end of every proof.
__global__ void __launch_bounds__(128) k_scale_a(G1XYZZ *g1, ProofConsts K, const Fr *r, const Fr *s, int with_consts) {
    __shared__ uint4 sm_raw[3 * sizeof(G1XYZZ) / 16];
    G1XYZZ *sm = reinterpret_cast<G1XYZZ *>(sm_raw);
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31;
    G1XYZZ acc = G1XYZZ::inf();
    if (lane == 0 && (role <= 1 || with_consts)) {
        G1XYZZ X = role <= 1 ? ld_vec(g1) : G1XYZZ::from_affine(K.b0);
        if (role <= 1 && with_consts) X.madd_cold(K.a0);
        acc = glv_half(X, ld_vec(role <= 1 ? s : r), role & 1);
    }
    if (lane == 0 && role) st_vec(sm + (role - 1), acc);
    __syncthreads();
    if (threadIdx.x == 0) {
        acc.add_cold(ld_vec(sm));
        acc.add_cold(ld_vec(sm + 1));
        acc.add_cold(ld_vec(sm + 2));
        st_vec(g1 + 4, acc);
    }
}
// out[i] = k * z[i] (canonical in and out)
__global__ void k_scalars_times(const Fr *z, const Fr *k, Fr *out, uint32_t count) {
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= count) return;
    st_vec(out + i, (ld_vec(z + i) * ld_vec(k)) * Fr::r2());
}
// g1[dst] += g1[src] (one thread)
__global__ void k_add_slot(G1XYZZ *g1, int dst, int src) {
    G1XYZZ a = ld_vec(g1 + dst);
    a.add_cold(ld_vec(g1 + src));
    st_vec(g1 + dst, a);
}

// Latency form (small calls): g1[q * P + p] additionally holds q = 4: s*(alpha + a0) + sum (s z_i) a_i and
// q = 5: r*(beta + b0) + sum (r z_i) b_i + 2 rs delta, so C is a sum of four MSM results and the tail of a proof is
// three conversions to affine on three warps (no scalar multiplication).
// (q0, q1) name the slots that hold the s*A and r*B1 shares: (4, 5) in the latency form; (1, -1) for one large proof,
// where slot 1 holds r * B1 plus the share k_scale_a computed (s * A and the constant terms).
__global__ void __launch_bounds__(96) k_assemble_sums(const G1XYZZ *g1, const G2XYZZ *g2, ProofConsts K, uint32_t P,
                                                      uint8_t *proofs, int q0, int q1) {
    const uint32_t role = threadIdx.x >> 5, lane = threadIdx.x & 31, p = blockIdx.x * 32 + lane;
    if (p >= P) return;
    uint8_t *out = proofs + (size_t)p * 256;
    if (role == 0) {
        G1XYZZ acc = ld_vec(g1 + (size_t)q0 * P + p);
        if (q1 >= 0) acc.add_cold(ld_vec(g1 + (size_t)q1 * P + p));
        acc.add_cold(ld_vec(g1 + 2 * (size_t)P + p));
        acc.add_cold(ld_vec(g1 + 3 * (size_t)P + p));
        write_g1(out + 192, acc.to_affine());
    } else if (role == 1) {
        G1XYZZ A = ld_vec(g1 + p);
        A.madd_cold(K.a0);
        write_g1(out, A.to_affine());
    } else {
        G2XYZZ B2 = ld_vec(g2 + p);
        B2.madd_cold(K.b2);
        write_g2(out + 64, B2.to_affine());
    }
}

// ---------------------------------------------------------------- libzkp envelopes (SURVEY.md §8f-4)
// Proof::to_bytes (src/proof/mod.rs:23-36): [version = 2][scheme][proof_len u32 LE][comm_len u32 LE][proof][commitment].
// Equality (scheme 2, equality_proof.rs:30-31): proof = the 256 Groth16 bytes -> 298 B per proof.
// Membership (scheme 4, set_membership.rs:29-37): proof = u32 len || u64[len] set || 256 Groth16 bytes.
// One warp per proof copies the pieces; failed proofs (status != 0) get out_len = 0.
__global__ void __launch_bounds__(128) k_envelope(const uint8_t *proofs, const uint8_t *commit, const int32_t *status,
                                                  const uint64_t *sets, const uint32_t *set_len, uint32_t set_stride,
                                                  uint32_t scheme, uint32_t P, uint8_t *out, uint32_t out_stride,
                                                  uint32_t *out_len) {
    const uint32_t p = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
    if (p >= P) return;
    uint8_t *o = out + (size_t)p * out_stride;
    if (status[p] != 0) {
        if (lane == 0) out_len[p] = 0;
        return;
    }
    const uint32_t len = sets ? set_len[p] : 0, prefix = sets ? 4 + 8 * len : 0, payload = prefix + 256;
    if (lane == 0) {
        o[0] = 2; o[1] = (uint8_t)scheme;
        for (int i = 0; i < 4; i++) { o[2 + i] = (uint8_t)(payload >> (8 * i)); o[6 + i] = (uint8_t)(32u >> (8 * i)); }
        if (sets) for (int i = 0; i < 4; i++) o[10 + i] = (uint8_t)(len >> (8 * i));
        out_len[p] = 10 + payload + 32;
    }
    if (sets) {
        const uint8_t *sv = reinterpret_cast<const uint8_t *>(sets + (size_t)p * set_stride);
        for (uint32_t i = lane; i < 8 * len; i += 32) o[14 + i] = sv[i];
    }
    for (uint32_t i = lane; i < 256; i += 32) o[10 + prefix + i] = proofs[(size_t)p * 256 + i];
    o[10 + payload + lane] = commit[(size_t)p * 32 + lane];
}

// Sharded single proof: partial[i] = 4 G1 XYZZ sums (a, b1, l, h) then 1 G2 XYZZ sum (b2) of rank i's point ranges.
// Warp q < 4 adds up G1 slot q over the ranks, warp 4 the G2 slot (one lane each: five independent chains side by side).
constexpr uint32_t kPartialBytes = 4 * sizeof(G1XYZZ) + sizeof(G2XYZZ);
__global__ void k_sum_partials(const uint8_t *partials, uint32_t n, G1XYZZ *g1, G2XYZZ *g2) {
    const uint32_t q = threadIdx.x >> 5;
    if (threadIdx.x & 31) return;
    if (q < 4) {
        G1XYZZ acc = G1XYZZ::inf();
        for (uint32_t i = 0; i < n; i++)
            acc.add_cold(ld_vec(reinterpret_cast<const G1XYZZ *>(partials + (size_t)i * kPartialBytes) + q));
        st_vec(g1 + q, acc);
    } else if (q == 4) {
        G2XYZZ acc = G2XYZZ::inf();
        for (uint32_t i = 0; i < n; i++)
            acc.add_cold(ld_vec(reinterpret_cast<const G2XYZZ *>(partials + (size_t)i * kPartialBytes + 4 * sizeof(G1XYZZ))));
        st_vec(g2, acc);
    }
}

// ---------------------------------------------------------------- pk-load helpers
// out = a + b (affine), one thread
template <class F>
__global__ void k_affine_add(const Affine<F> *a, const Affine<F> *b, Affine<F> *out, int negate_b) {
    XYZZ<F> s = XYZZ<F>::from_affine(ld_vec(a));
    Affine<F> q = ld_vec(b);
    if (negate_b) q = q.neg();
    s.madd_cold(q);
    st_vec(out, s.to_affine());
}
// bad[0] += points off the curve; for G2 also points outside the r-torsion (r*P != inf)
__global__ void k_check_g1(const G1Affine *pts, uint32_t n, int *bad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    if (!g1_on_curve(ld_vec(pts + i))) atomicAdd(bad, 1);
}
__global__ void k_check_g2(const G2Affine *pts, uint32_t n, int *bad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    G2Affine p = ld_vec(pts + i);
    if (!g2_on_curve(p)) { atomicAdd(bad, 1); return; }
    if (p.is_inf()) return;
    // r * P == inf  <=>  (r-1) * P == -P ; scalar_mul takes a 254-bit canonical scalar < r
    Fr rm1 = Fr::modulus();
    rm1.l[0] -= 1;
    G2XYZZ t = scalar_mul(G2XYZZ::from_affine(p), rm1);
    t.madd_cold(p);
    if (!t.is_inf()) atomicAdd(bad, 1);
}

}  // namespace lzkp
