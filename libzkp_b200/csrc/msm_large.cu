// msm_large.cu — variable-base MSM over BN254 G1 / G2 for large sizes (Pippenger bucket method).
//
// Replaces ark-ec's VariableBaseMSM::msm_bigint, which ark-groth16's prover calls five times per
// proof (a_query, b_g1_query, b_g2_query, l_query, h_query; reached from src/backend/snark.rs:364
// and :442; SURVEY.md §8a rows a8-a12).  The result is the unique group element, so its affine
// serialization is bit-identical to arkworks' whatever the window size or summation order.
//
// Pipeline (no host synchronisation between stages):
//   1. k_msm_digits      signed c-bit window recoding of every scalar -> (bucket key, point ref | sign)
//   2. cub::DeviceRadixSort::SortPairs on the keys (zero digits carry a sentinel key and sort last)
//   3. k_bucket_accum    perfectly balanced segmented accumulation: every thread owns L consecutive
//                        sorted pairs whatever the bucket sizes; runs strictly inside a chunk go
//                        straight to their bucket, the first/last run of a chunk become partial sums
//   4. k_partial_merge   partial sums of one bucket are adjacent: the head of each run adds them up
//                        (runs longer than a cap go to k_long_run: one CTA per run, tree reduction)
//   5. k_red_*           sum_b (b+1) * B[b]: per-thread running sums over groups of 16 buckets, then
//                        bit-plane tree sums over the group index (log depth, no long serial chain)
//   6. k_horner_* / k_finish combine windows (generic mode only), to affine, ark-serialize bytes
//
// Two modes.  "Resident" bases (the proving key's queries: loaded once, kept in HBM) also hold
// 2^(c*w) * P for every window w, so all windows share ONE bucket set, there is no Horner tail, and
// the reduction handles 2^(c-1) buckets instead of W * 2^(c-1): HBM capacity traded for work.
// "Generic" bases (lzkp_msm_g1/_g2 one-shot calls) use one bucket set per window.
#include <cub/cub.cuh>

#include "dev_util.cuh"
#include "host_util.h"
#include "large.h"

#ifndef LZKP_G2_MINB
#define LZKP_G2_MINB 6
#endif
// minimum resident CTAs per SM: G1 kernels leave it to ptxas, G2 kernels (64-thread CTAs) trade registers for warps
#ifndef LZKP_G1_MINB
#define LZKP_G1_MINB 1
#endif
#define LZKP_G2_MINB_SEL(F) (sizeof(F) == sizeof(::lzkp::Fq) ? LZKP_G1_MINB : LZKP_G2_MINB)
namespace lzkp {

namespace {

constexpr uint32_t SENT = 0xFFFFFFFFu;
#ifndef LZKP_G2_CHUNK
#define LZKP_G2_CHUNK 32
#endif
// sorted pairs per thread in k_bucket_accum
template <class F> constexpr int chunk_of() { return sizeof(F) == sizeof(Fq) ? 32 : LZKP_G2_CHUNK; }
constexpr int kSeg = 8;             // partial slots per thread in k_seg_reduce
constexpr int kSegLevels = 2;       // balanced partial-reduction passes before the final merge
constexpr int kMergeCap = 48;       // partials merged serially before a run counts as "long"
constexpr int kGroup = 16;          // buckets per running-sum group
constexpr int kGroupLog = 4;

// ---------------------------------------------------------------- 1. digits
// keys/vals[w * n + i].  Resident mode: key = |d| - 1, point ref = w * n + i.  Generic: key = w * NB + |d| - 1, ref = i.
__global__ void __launch_bounds__(256) k_msm_digits(const Fr *__restrict__ scalars, uint32_t n_used, uint32_t n,
                                                    uint32_t c, uint32_t W, uint32_t NB, int resident,
                                                    uint32_t *__restrict__ keys, uint32_t *__restrict__ vals,
                                                    int *__restrict__ bad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_used) return;
    Fr s = ld_vec(scalars + i);
    if (!fr_is_canonical(s)) {
        atomicAdd(bad, 1);
        s = Fr::zero();
    }
    uint32_t v[10];
    recode_offset(s, c, W, v);
    for (uint32_t w = 0; w < W; w++) {
        int d = recoded_digit(v, c, w);
        uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
        uint32_t key = SENT, val = 0;
        if (d) {
            key = (resident ? 0u : w * NB) + mag - 1u;
            val = (resident ? w * n + i : i) | (d < 0 ? 0x80000000u : 0u);
        }
        keys[(size_t)w * n + i] = key;
        vals[(size_t)w * n + i] = val;
    }
}

// GLV form of the generic (one bucket set per window) G1 MSM: k P = (+-k1) P + (+-k2) phi(P) with phi(x, y) = (beta x, y)
// and |k1|, |k2| < 2^128, so the 2n "virtual" points (P_i at i, phi(P_i) at n + i) carry 128-bit scalars: half as many
// windows - the window combination's chain of dependent doublings drops from c (W - 1) = 240 to 128 and the number of
// bucket sets to reduce from 16 to 9 - for the same number of (point, window) pairs.
// Magnitudes of the lattice split stay below ~2^128 (ec.cuh glv_split: never above 2^127 over 2 * 10^5 scalars);
// the W = ceil(130 / c) windows used here hold anything below 2^(c W - 2) (s + K < 2^(c W) with the recoding offset
// K < 2^(c W - 1) (1 + 2^(1-c)); c W >= 130, so every 128-bit magnitude fits), and a split beyond that is counted in
// `bad` like a non-canonical scalar rather than silently mis-added.
__device__ __forceinline__ void glv_split_wide(const Fr &k, Fr &m1, bool &neg1, Fr &m2, bool &neg2) {
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
    uint32_t p1[8], p2[8], p3[8], p4[8], t[8];
    mul_limbs<8, 5, 4>(p1, c1, A1);
    mul_limbs<8, 3, 2>(p2, c2, A2);
    mul_limbs<8, 5, 2>(p3, c1, A2);
    mul_limbs<8, 3, 4>(p4, c2, B2);
    sub8(t, k.l, p1);
    sub8(m1.l, t, p2);
    sub8(m2.l, p3, p4);
    neg1 = (m1.l[7] >> 31) != 0;
    neg2 = (m2.l[7] >> 31) != 0;
    const uint32_t zero[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    if (neg1) { sub8(t, zero, m1.l);
#pragma unroll
        for (int i = 0; i < 8; i++) m1.l[i] = t[i]; }
    if (neg2) { sub8(t, zero, m2.l);
#pragma unroll
        for (int i = 0; i < 8; i++) m2.l[i] = t[i]; }
}
__global__ void __launch_bounds__(256) k_msm_digits_glv(const Fr *__restrict__ scalars, uint32_t n_used, uint32_t n,
                                                        uint32_t c, uint32_t W, uint32_t NB, uint32_t *__restrict__ keys,
                                                        uint32_t *__restrict__ vals, int *__restrict__ bad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_used) return;
    Fr s = ld_vec(scalars + i);
    if (!fr_is_canonical(s)) {
        atomicAdd(bad, 1);
        s = Fr::zero();
    }
    Fr m[2];
    bool neg[2];
    glv_split_wide(s, m[0], neg[0], m[1], neg[1]);
    const uint32_t top = c * W - 2;                       // magnitudes must stay below 2^top for the offset recoding
    for (int h = 0; h < 2; h++) {
        uint32_t over = 0;
        for (uint32_t b = top >> 5; b < 8; b++) over |= b == (top >> 5) ? (m[h].l[b] >> (top & 31)) : m[h].l[b];
        if (over) {
            atomicAdd(bad, 1);
            m[h] = Fr::zero();
        }
    }
    const size_t nv = (size_t)2 * n;
    for (int h = 0; h < 2; h++) {
        uint32_t v[10];
        recode_offset(m[h], c, W, v);
        for (uint32_t w = 0; w < W; w++) {
            int d = recoded_digit(v, c, w);
            if (neg[h]) d = -d;
            uint32_t mag = d < 0 ? (uint32_t)(-d) : (uint32_t)d;
            uint32_t key = SENT, val = 0;
            if (d) {
                key = w * NB + mag - 1u;
                val = ((uint32_t)h * n + i) | (d < 0 ? 0x80000000u : 0u);
            }
            keys[(size_t)w * nv + (size_t)h * n + i] = key;
            vals[(size_t)w * nv + (size_t)h * n + i] = val;
        }
    }
}
// pts[n + i] = phi(pts[i]) = (beta * x, y); infinity (0, 0) stays infinity
__global__ void k_phi_points(G1Affine *pts, uint32_t n) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    G1Affine p = ld_vec(pts + i);
    Fq beta;
#pragma unroll
    for (int j = 0; j < 8; j++) beta.l[j] = FqParams::BETA(j);
    p.x = p.x * beta;
    st_vec(pts + n + i, p);
}

// count[0] = number of sorted pairs with a real key (sentinels sort last)
__global__ void k_find_count(const uint32_t *keys, uint32_t total, uint32_t *count) {
    uint32_t lo = 0, hi = total;
    while (lo < hi) {
        uint32_t mid = lo + (hi - lo) / 2;
        if (keys[mid] == SENT) hi = mid; else lo = mid + 1;
    }
    count[0] = lo;
    count[1] = 0;      // long-run counter
}

// ---------------------------------------------------------------- 3. balanced segmented accumulation
template <class F>
__device__ __forceinline__ Affine<F> fetch_point(const Affine<F> *__restrict__ points, uint32_t v) {
    Affine<F> p = ldg_vec(points + (v & 0x7FFFFFFFu));
    if (v >> 31) p.y = p.y.neg();
    return p;
}

template <class F, int L, int BLOCK>
__global__ void __launch_bounds__(BLOCK, LZKP_G2_MINB_SEL(F)) k_bucket_accum(const uint32_t *__restrict__ keys, const uint32_t *__restrict__ vals,
                                                        const uint32_t *__restrict__ count,
                                                        const Affine<F> *__restrict__ points, XYZZ<F> *__restrict__ buckets,
                                                        uint32_t *__restrict__ pkey, XYZZ<F> *__restrict__ ppt) {
    const size_t t = (size_t)blockIdx.x * BLOCK + threadIdx.x;
    const size_t M = count[0], start = t * L;
    if (start >= M) return;
    const uint32_t len = (uint32_t)min((size_t)L, M - start);
    const uint32_t *kp = keys + start, *vp = vals + start;
    uint32_t cur = kp[0];
    int run = 0;
    XYZZ<F> acc = XYZZ<F>::inf();
    // G1: the next point is loaded into registers under the current add.  G2 is register-starved (a 256-byte
    // accumulator, 128-byte points, 255 registers): it only issues an L2 prefetch for the next point instead.
    constexpr bool kRegPrefetch = sizeof(F) == sizeof(Fq);
    Affine<F> pt = Affine<F>::inf();
    if constexpr (kRegPrefetch) pt = fetch_point(points, vp[0]);
    uint32_t vn = len > 1 ? vp[1] : 0u;                                  // point ref of pair j + 1, one step ahead of its use
    for (uint32_t j = 0; j < len; j++) {
        uint32_t k = kp[j];
        Affine<F> nxt = Affine<F>::inf();
        if constexpr (kRegPrefetch) {
            const uint32_t vnn = j + 2 < len ? vp[j + 2] : 0u;
            if (j + 1 < len) nxt = fetch_point(points, vn);              // prefetch under the current add
            vn = vnn;
        } else {
            if (j + 1 < len) {
                const char *np_ = reinterpret_cast<const char *>(points + (vp[j + 1] & 0x7FFFFFFFu));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(np_));
                asm volatile("prefetch.global.L2 [%0];" ::"l"(np_ + 64));
            }
            pt = fetch_point(points, vp[j]);
        }
        if (k != cur) {
            if (run == 0) { pkey[2 * t] = cur; st_vec(ppt + 2 * t, acc); }
            else st_vec(buckets + cur, acc);                          // a run strictly inside the chunk: complete
            run++;
            acc = XYZZ<F>::inf();
            cur = k;
        }
        acc.madd(pt);
        if constexpr (kRegPrefetch) pt = nxt;
    }
    if (run == 0) {
        pkey[2 * t] = cur; st_vec(ppt + 2 * t, acc);
        pkey[2 * t + 1] = SENT;
    } else {
        pkey[2 * t + 1] = cur; st_vec(ppt + 2 * t + 1, acc);
    }
}

// ---------------------------------------------------------------- 3b. balanced reduction of the partial sums
// Same chunking one level up: every thread owns L consecutive partial slots (all lanes busy whatever the
// run lengths), adds up equal keys, sends runs strictly inside its chunk to their bucket and re-emits its
// first / last run as partials of the next level.  Each level shrinks the sequence by L / 2.
__device__ __forceinline__ uint32_t level_slots(uint32_t M, uint32_t L1, uint32_t L2, uint32_t level) {
    uint32_t n = 2u * ((M + L1 - 1) / L1);                 // level 1 output
    for (uint32_t l = 1; l < level; l++) n = 2u * ((n + L2 - 1) / L2);
    return n;
}
template <class F, int L>
__global__ void __launch_bounds__(128) k_seg_reduce(const uint32_t *__restrict__ in_key, const XYZZ<F> *__restrict__ in_pt,
                                                    const uint32_t *__restrict__ count, uint32_t L1, uint32_t level,
                                                    XYZZ<F> *__restrict__ buckets, uint32_t *__restrict__ out_key,
                                                    XYZZ<F> *__restrict__ out_pt) {
    const uint32_t n_in = level_slots(count[0], L1, L, level);
    const uint32_t t = blockIdx.x * blockDim.x + threadIdx.x, start = t * L;
    if (start >= n_in) return;
    const uint32_t end = min(start + (uint32_t)L, n_in);
    uint32_t cur = SENT;
    int run = 0;
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t j = start; j < end; j++) {
        uint32_t k = in_key[j];
        if (k == SENT) continue;
        if (cur == SENT) {
            cur = k;
            acc = ld_vec(in_pt + j);
            continue;
        }
        if (k != cur) {
            if (run == 0) { out_key[2 * t] = cur; st_vec(out_pt + 2 * t, acc); }
            else st_vec(buckets + cur, acc);
            run++;
            cur = k;
            acc = ld_vec(in_pt + j);
        } else {
            acc.add(ld_vec(in_pt + j));
        }
    }
    if (run == 0) {
        out_key[2 * t] = cur;                                 // SENT if the chunk was empty
        if (cur != SENT) st_vec(out_pt + 2 * t, acc);
        out_key[2 * t + 1] = SENT;
    } else {
        out_key[2 * t + 1] = cur; st_vec(out_pt + 2 * t + 1, acc);
    }
}

// ---------------------------------------------------------------- 4. partial merge
template <class F>
__global__ void __launch_bounds__(128) k_partial_merge(const uint32_t *__restrict__ pkey, const XYZZ<F> *__restrict__ ppt,
                                                       uint32_t *__restrict__ count, uint32_t L1, uint32_t L2,
                                                       uint32_t level, XYZZ<F> *__restrict__ buckets,
                                                       uint32_t *__restrict__ long_list) {
    const uint32_t n2 = level_slots(count[0], L1, L2, level);
    const uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n2) return;
    const uint32_t key = pkey[i];
    if (key == SENT) return;
    if (i > 0) {                        // head of its run?  (of two consecutive slots at least one is real)
        uint32_t p = pkey[i - 1];
        if (p == SENT && i > 1) p = pkey[i - 2];
        if (p == key) return;
    }
    XYZZ<F> acc = ld_vec(ppt + i);
    int merged = 0;
    for (uint32_t j = i + 1; j < n2; j++) {
        uint32_t kj = pkey[j];
        if (kj == SENT) continue;
        if (kj != key) break;
        if (++merged > kMergeCap) {
            long_list[atomicAdd(count + 1, 1u)] = i;
            return;
        }
        acc.add(ld_vec(ppt + j));
    }
    st_vec(buckets + key, acc);
}

template <class F, int THREADS>
__device__ __forceinline__ void block_tree_sum(XYZZ<F> &v, XYZZ<F> *sm) {      // result in thread 0's v
    st_vec(sm + threadIdx.x, v);
    __syncthreads();
#pragma unroll 1
    for (int s = THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) {
            v.add_cold(ld_vec(sm + threadIdx.x + s));
            st_vec(sm + threadIdx.x, v);
        }
        __syncthreads();
    }
}

template <class F>
__global__ void __launch_bounds__(128) k_long_run(const uint32_t *__restrict__ pkey, const XYZZ<F> *__restrict__ ppt,
                                                  const uint32_t *__restrict__ count, uint32_t L1, uint32_t L2,
                                                  uint32_t level, XYZZ<F> *__restrict__ buckets,
                                                  const uint32_t *__restrict__ long_list) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(smem_raw);
    if (blockIdx.x >= count[1]) return;
    const uint32_t n2 = level_slots(count[0], L1, L2, level);
    const uint32_t i0 = long_list[blockIdx.x], key = pkey[i0];
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t j = i0 + threadIdx.x; j < n2; j += 128) {
        uint32_t kj = pkey[j];
        if (kj == SENT) continue;
        if (kj != key) break;
        acc.add_cold(ld_vec(ppt + j));
    }
    block_tree_sum<F, 128>(acc, sm);
    if (threadIdx.x == 0) st_vec(buckets + key, acc);
}

// ---------------------------------------------------------------- 5. bucket reduction  sum_b (b+1) B[b]
// group g of a set covers buckets g*16 .. g*16+15:  Sg = sum_j (j+1) B[16g+j],  Ag = sum_j B[16g+j]
template <class F>
__global__ void __launch_bounds__(128) k_red_groups(const XYZZ<F> *__restrict__ buckets, uint32_t n_groups_total,
                                                    XYZZ<F> *__restrict__ Sg, XYZZ<F> *__restrict__ Ag) {
    uint32_t g = blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_groups_total) return;
    const XYZZ<F> *b = buckets + (size_t)g * kGroup;
    XYZZ<F> run = XYZZ<F>::inf(), sum = XYZZ<F>::inf();
#pragma unroll 1
    for (int j = kGroup - 1; j >= 0; j--) {
        run.add_cold(ld_vec(b + j));
        sum.add_cold(run);
    }
    st_vec(Sg + g, sum);
    st_vec(Ag + g, run);
}
// plane p < LP: sum of Ag[g] over groups with bit p of g set; plane LP: sum of Sg.  grid (nblk, LP + 1, sets)
template <class F>
__global__ void __launch_bounds__(128) k_red_planes(const XYZZ<F> *__restrict__ Sg, const XYZZ<F> *__restrict__ Ag,
                                                    uint32_t NG, uint32_t LP, XYZZ<F> *__restrict__ out1) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(smem_raw);
    const uint32_t g = blockIdx.x * 128 + threadIdx.x, p = blockIdx.y, set = blockIdx.z;
    XYZZ<F> v = XYZZ<F>::inf();
    if (g < NG) {
        if (p == LP) v = ld_vec(Sg + (size_t)set * NG + g);
        else if ((g >> p) & 1u) v = ld_vec(Ag + (size_t)set * NG + g);
    }
    block_tree_sum<F, 128>(v, sm);
    if (threadIdx.x == 0) st_vec(out1 + ((size_t)set * (LP + 1) + p) * gridDim.x + blockIdx.x, v);
}
// R[set] = sum Sg + 16 * sum_p 2^p plane_p.  grid (sets), 32 threads
template <class F>
__global__ void __launch_bounds__(32) k_red_finish(const XYZZ<F> *__restrict__ out1, uint32_t nblk, uint32_t LP,
                                                   XYZZ<F> *__restrict__ R) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(smem_raw);
    const uint32_t p = threadIdx.x, set = blockIdx.x;
    XYZZ<F> v = XYZZ<F>::inf();
    if (p <= LP) {
        const XYZZ<F> *src = out1 + ((size_t)set * (LP + 1) + p) * nblk;
#pragma unroll 1
        for (uint32_t b = 0; b < nblk; b++) v.add_cold(ld_vec(src + b));
        if (p < LP)
#pragma unroll 1
            for (uint32_t d = 0; d < p + kGroupLog; d++) v.dbl_cold();
    }
    block_tree_sum<F, 32>(v, sm);
    if (threadIdx.x == 0) st_vec(R + set, v);
}

// Resident mode (one bucket set): sum_b (b+1) B[b] straight from bit planes of (b+1).
// plane p: sum of B[b] over buckets with bit p of (b+1) set.  Every thread first adds up kRedSer masked
// buckets serially (all lanes busy), only then does the CTA run a tree.  grid (NB / (128 * kRedSer), c)
constexpr uint32_t kRedSer = 16;
template <class F>
__global__ void __launch_bounds__(128) k_red_direct1(const XYZZ<F> *__restrict__ buckets, uint32_t NB,
                                                     XYZZ<F> *__restrict__ out1) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(smem_raw);
    const uint32_t p = blockIdx.y, b0 = blockIdx.x * (128 * kRedSer) + threadIdx.x;
    XYZZ<F> v = XYZZ<F>::inf();
#pragma unroll 1
    for (uint32_t j = 0; j < kRedSer; j++) {
        const uint32_t b = b0 + j * 128;
        if (b < NB && (((b + 1) >> p) & 1u)) v.add_cold(ld_vec(buckets + b));
    }
    block_tree_sum<F, 128>(v, sm);
    if (threadIdx.x == 0) st_vec(out1 + (size_t)p * gridDim.x + blockIdx.x, v);
}
// per plane: tree over the nblk partial sums, then p doublings.  grid (c), 128 threads
template <class F>
__global__ void __launch_bounds__(128) k_red_direct2(const XYZZ<F> *__restrict__ out1, uint32_t nblk,
                                                     XYZZ<F> *__restrict__ out2) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(smem_raw);
    const uint32_t p = blockIdx.x;
    XYZZ<F> v = XYZZ<F>::inf();
    for (uint32_t i = threadIdx.x; i < nblk; i += 128) v.add_cold(ld_vec(out1 + (size_t)p * nblk + i));
    block_tree_sum<F, 128>(v, sm);
    if (threadIdx.x == 0) {
#pragma unroll 1
        for (uint32_t d = 0; d < p; d++) v.dbl_cold();
        st_vec(out2 + p, v);
    }
}
// R[0] = sum over the planes.  32 threads
template <class F>
__global__ void __launch_bounds__(32) k_red_direct3(const XYZZ<F> *__restrict__ out2, uint32_t planes, XYZZ<F> *__restrict__ R) {
    extern __shared__ uint4 smem_raw[];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(smem_raw);
    XYZZ<F> v = XYZZ<F>::inf();
    if (threadIdx.x < planes) v = ld_vec(out2 + threadIdx.x);
    block_tree_sum<F, 32>(v, sm);
    if (threadIdx.x == 0) st_vec(R, v);
}

// ---------------------------------------------------------------- 6. window combination, output
// generic mode: result = sum_w 2^(c*w) R[w]
// Window w is shifted by its own CTA (one thread: c*w doublings of R[w], in place), all windows side by side on
// different SMs; k_horner_sum then adds the W shifted sums in log depth.  The serial chain is the top window's
// c*(W-1) doublings - nothing else: the Horner form (c doublings and one addition, W - 1 times on ONE thread)
// took 1.12 ms at c = 16, W = 16.
template <class F>
__global__ void k_horner_shift(XYZZ<F> *R, uint32_t c) {
    if (threadIdx.x) return;
    const uint32_t w = blockIdx.x;
    if (w == 0) return;
    XYZZ<F> acc = ld_vec(R + w);
#pragma unroll 1
    for (uint32_t d = 0; d < c * w; d++) acc.dbl_cold();
    st_vec(R + w, acc);
}
template <class F>
__global__ void __launch_bounds__(32) k_horner_sum(XYZZ<F> *R, uint32_t W) {      // W <= 32: lane w owns window w
    __shared__ uint4 raw[32 * sizeof(XYZZ<F>) / 16];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(raw);
    const uint32_t w = threadIdx.x;
    if (w < W) st_vec(sm + w, ld_vec(R + w));
    __syncwarp();
    for (uint32_t s = 1; s < W; s <<= 1) {
        if (w < W && (w & (2 * s - 1)) == 0 && w + s < W) {
            XYZZ<F> a = ld_vec(sm + w);
            a.add_cold(ld_vec(sm + w + s));
            st_vec(sm + w, a);
        }
        __syncwarp();
    }
    if (w == 0) st_vec(R, ld_vec(sm));
}
template <class F, int BYTES>
__global__ void k_finish(const XYZZ<F> *R, uint8_t *out) {
    Affine<F> a = ld_vec(R).to_affine();
    if constexpr (BYTES == 64) write_g1(out, a);
    else write_g2(out, a);
}

// ---------------------------------------------------------------- base upload / window precomputation
// pre[w * n + i] = 2^(c*w) * base[i] (affine).  One thread per base walks the windows.
template <class F>
__global__ void __launch_bounds__(128) k_precompute_windows(Affine<F> *pre, uint32_t n, uint32_t c, uint32_t W) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    XYZZ<F> acc = XYZZ<F>::from_affine(ld_vec(pre + i));
    for (uint32_t w = 1; w < W; w++) {
#pragma unroll 1
        for (uint32_t d = 0; d < c; d++) acc.dbl_cold();
        Affine<F> a = acc.to_affine();
        st_vec(pre + (size_t)w * n + i, a);
        acc = XYZZ<F>::from_affine(a);
    }
}
__global__ void k_fq_array_to_mont(Fq *v, size_t count) {
    size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= count) return;
    st_vec(v + k, Fq::from_canonical(ld_vec(v + k)));
}
// bad[0] += points that are not on the curve (infinity = (0,0) is accepted)
template <class F>
__global__ void k_check_on_curve(const Affine<F> *pts, uint32_t n, int *bad) {
    uint32_t i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    Affine<F> p = ld_vec(pts + i);
    bool ok;
    if constexpr (sizeof(F) == sizeof(Fq)) ok = g1_on_curve(p);       // G1 has cofactor 1: on the curve = in the group
    else {
        ok = g2_on_curve(p);
        if (ok && !p.is_inf()) {       // r-torsion test, as deserialize_uncompressed does: (r - 1) P == -P
            Fr rm1 = Fr::modulus();
            rm1.l[0] -= 1;
            XYZZ<F> t = scalar_mul(XYZZ<F>::from_affine(p), rm1);
            t.madd_cold(p);
            ok = t.is_inf();
        }
    }
    if (!ok) atomicAdd(bad, 1);
}

template <class F> struct PointIO;
template <> struct PointIO<Fq> { static constexpr int BYTES = 64; };
template <> struct PointIO<Fq2> { static constexpr int BYTES = 128; };

}  // namespace

namespace eng {

struct MsmBases {
    int group = 1;                 // 1 = G1, 2 = G2
    uint32_t n = 0, c = 16, W = 16, NB = 32768;
    bool resident = false;
    bool glv = false;              // generic G1 mode: 2n virtual points (P, phi(P)) with 128-bit scalars
    uint32_t nv = 0;               // points the pipeline walks per window: n, or 2n with glv
    uint32_t sets = 16;            // bucket sets: 1 (resident) or W (generic)
    DBuf points;                   // Affine<F>[n] or [W * n]
    // workspace
    DBuf keys_a, keys_b, vals_a, vals_b, cub_tmp, count, buckets, pkey, ppt, long_list, Sg, Ag, out1, R, d_scalars,
        d_out, bad;
    size_t cub_bytes = 0;
    uint32_t key_bits = 0, T = 0, NG = 0, LP = 0, nblk = 0;
    size_t lvl_off[4] = {0, 0, 0, 0}, lvl_slots[4] = {0, 0, 0, 0};
    std::mutex mu;
};

template <class F>
static int bases_prepare(MsmBases *B, const uint8_t *bases_bytes, size_t n, int window_bits, int resident, int validate,
                         int canon_input) {
    constexpr int BYTES = PointIO<F>::BYTES;
    if (n >= (1u << 27)) return fail(LZKP_E_UNSUPPORTED, "MSM size above 2^27");
    B->group = BYTES == 64 ? 1 : 2;
    B->n = (uint32_t)n;
    B->c = window_bits ? (uint32_t)window_bits : 16u;
    if (B->c < 8 || B->c > 16) return fail(LZKP_E_INVALID, "MSM window_bits must be in [8,16]");
    B->W = (255 + B->c - 1) / B->c;
    B->NB = 1u << (B->c - 1);
    B->resident = resident != 0;
    B->glv = !B->resident && BYTES == 64 && getenv("LZKP_MSM_NO_GLV") == nullptr;
    if (B->glv) B->W = (130 + B->c - 1) / B->c;          // s + K < 2^(cW) with |s| < 2^129: 9 windows at c = 16
    B->sets = B->resident ? 1u : B->W;
    B->nv = B->glv ? 2 * B->n : B->n;
    if ((uint64_t)B->nv * B->W >= (1ull << 31)) return fail(LZKP_E_UNSUPPORTED, "MSM: n * windows must stay below 2^31");
    const uint32_t n1 = std::max<uint32_t>(B->n, 1);
    // ---- parse ark-serialize points on the host (canonical limbs, flags stripped), upload, to Montgomery
    std::vector<uint8_t> canon;
    if (!canon_input) canon.assign((size_t)n1 * BYTES, 0);
    for (size_t i = 0; i < n && !canon_input; i++) {
        bool ok;
        if constexpr (BYTES == 64) ok = host::read_g1(bases_bytes + i * 64, *reinterpret_cast<host::G1Canon *>(canon.data() + i * 64));
        else ok = host::read_g2(bases_bytes + i * 128, *reinterpret_cast<host::G2Canon *>(canon.data() + i * 128));
        if (!ok) return fail(LZKP_E_INVALID, "MSM base " + std::to_string(i) + ": non-canonical coordinate");
    }
    TRY(B->points.alloc((size_t)n1 * (B->resident ? B->W : (B->glv ? 2 : 1)) * BYTES));
    if (canon_input) {      // already parsed: canonical limbs, (0,0) = infinity
        CUDA_TRY(cudaMemset(B->points.p, 0, (size_t)n1 * BYTES));
        if (n) CUDA_TRY(cudaMemcpy(B->points.p, bases_bytes, n * BYTES, cudaMemcpyHostToDevice));
    } else {
        CUDA_TRY(cudaMemcpy(B->points.p, canon.data(), canon.size(), cudaMemcpyHostToDevice));
    }
    const size_t n_fq = (size_t)n1 * BYTES / 32;
    LAUNCH(k_fq_array_to_mont, (unsigned)((n_fq + 255) / 256), 256, 0, 0, B->points.as<Fq>(), n_fq);
    TRY(B->bad.alloc(sizeof(int)));
    CUDA_TRY(cudaMemset(B->bad.p, 0, sizeof(int)));
    if (validate && n) {
        LAUNCH((k_check_on_curve<F>), (B->n + 127) / 128, 128, 0, 0, B->points.as<Affine<F>>(), B->n, B->bad.as<int>());
        int bad = 0;
        CUDA_TRY(cudaMemcpy(&bad, B->bad.p, sizeof(int), cudaMemcpyDeviceToHost));
        if (bad) return fail(LZKP_E_INVALID, "MSM bases: " + std::to_string(bad) + " point(s) off-curve or outside the subgroup");
    }
    if (B->resident && n)
        LAUNCH((k_precompute_windows<F>), (B->n + 127) / 128, 128, 0, 0, B->points.as<Affine<F>>(), B->n, B->c, B->W);
    if constexpr (BYTES == 64) {
        if (B->glv && n) LAUNCH(k_phi_points, (B->n + 127) / 128, 128, 0, 0, B->points.as<G1Affine>(), B->n);
    }
    // ---- workspace
    const size_t total = (size_t)std::max<uint32_t>(B->nv, 1) * B->W;
    B->key_bits = 1;
    while ((1ull << B->key_bits) < (uint64_t)B->sets * B->NB) B->key_bits++;
    B->T = (uint32_t)((total + chunk_of<F>() - 1) / chunk_of<F>());
    B->NG = B->NB / kGroup;
    B->LP = 0;
    while ((1u << B->LP) < B->NG) B->LP++;
    B->nblk = (B->NG + 127) / 128;
    TRY(B->keys_a.alloc(total * 4)); TRY(B->keys_b.alloc(total * 4));
    TRY(B->vals_a.alloc(total * 4)); TRY(B->vals_b.alloc(total * 4));
    cub::DoubleBuffer<uint32_t> dk(B->keys_a.as<uint32_t>(), B->keys_b.as<uint32_t>()), dv(B->vals_a.as<uint32_t>(), B->vals_b.as<uint32_t>());
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(nullptr, B->cub_bytes, dk, dv, (int)total, 0, 32));
    TRY(B->cub_tmp.alloc(B->cub_bytes));
    TRY(B->count.alloc(16));
    TRY(B->buckets.alloc((size_t)B->sets * B->NB * sizeof(XYZZ<F>)));
    // partial-sum levels: level 1 has 2T slots, every further level 2 * ceil(prev / kSeg); stored back to back
    B->lvl_off[0] = 0;
    size_t slots = (size_t)2 * B->T, tot_slots = 0;
    for (int l = 0; l <= kSegLevels; l++) {
        B->lvl_off[l] = tot_slots;
        B->lvl_slots[l] = slots;
        tot_slots += slots;
        slots = 2 * ((slots + kSeg - 1) / kSeg);
    }
    TRY(B->pkey.alloc(tot_slots * 4));
    TRY(B->ppt.alloc(tot_slots * sizeof(XYZZ<F>)));
    TRY(B->long_list.alloc(((size_t)2 * B->T / kMergeCap + 2) * 4));
    TRY(B->Sg.alloc((size_t)B->sets * B->NG * sizeof(XYZZ<F>)));
    TRY(B->Ag.alloc((size_t)B->sets * B->NG * sizeof(XYZZ<F>)));
    TRY(B->out1.alloc(std::max((size_t)B->sets * (B->LP + 1) * B->nblk, (size_t)B->c * ((B->NB + 127) / 128)) * sizeof(XYZZ<F>)));
    TRY(B->R.alloc((size_t)B->sets * sizeof(XYZZ<F>)));
    TRY(B->d_scalars.alloc((size_t)n1 * 32));
    TRY(B->d_out.alloc(BYTES));
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

// scalars: device, canonical, n_used <= B->n of them.  out: device, ark-serialize affine bytes.
template <class F>
// raw != 0: d_out receives the XYZZ sum (sizeof(XYZZ<F>) bytes) instead of ark-serialize affine bytes
static int msm_run(MsmBases *B, const Fr *d_scalars, uint32_t n_used, uint8_t *d_out, cudaStream_t st, int raw) {
    constexpr int BYTES = PointIO<F>::BYTES;
    using X = XYZZ<F>;
    const uint32_t n = B->n;
    if (n_used > n) return fail(LZKP_E_INVALID, "MSM: more scalars than resident bases");
    if (n_used == 0) {                    // empty sum: the point at infinity
        CUDA_TRY(cudaMemsetAsync(B->R.p, 0, sizeof(X), st));
        if (raw) CUDA_TRY(cudaMemcpyAsync(d_out, B->R.p, sizeof(X), cudaMemcpyDeviceToDevice, st));
        else LAUNCH((k_finish<F, BYTES>), 1, 1, 0, st, B->R.as<X>(), d_out);
        return LZKP_OK;
    }
    CUDA_TRY(cudaMemsetAsync(B->buckets.p, 0, (size_t)B->sets * B->NB * sizeof(X), st));
    const size_t total = (size_t)B->nv * B->W;
    if (n_used < n)      // unused tail of the digit arrays: sentinels
        CUDA_TRY(cudaMemsetAsync(B->keys_a.p, 0xFF, total * 4, st));
    if (n_used && B->glv) {
        LAUNCH(k_msm_digits_glv, (n_used + 255) / 256, 256, 0, st, d_scalars, n_used, n, B->c, B->W, B->NB,
               B->keys_a.as<uint32_t>(), B->vals_a.as<uint32_t>(), B->bad.as<int>());
    } else if (n_used) {
        // digits are laid out with the resident stride n so that point refs w * n + i stay valid
        LAUNCH(k_msm_digits, (n_used + 255) / 256, 256, 0, st, d_scalars, n_used, n, B->c, B->W, B->NB, (int)B->resident,
               B->keys_a.as<uint32_t>(), B->vals_a.as<uint32_t>(), B->bad.as<int>());
    }
    cub::DoubleBuffer<uint32_t> dk(B->keys_a.as<uint32_t>(), B->keys_b.as<uint32_t>()), dv(B->vals_a.as<uint32_t>(), B->vals_b.as<uint32_t>());
    size_t tmp = B->cub_bytes;
    // sentinel keys are 0xFFFFFFFF: sort on all 32 bits only if needed; real keys fit key_bits, and one extra
    // bit separates the sentinels
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(B->cub_tmp.p, tmp, dk, dv, (int)total, 0, (int)B->key_bits + 1, st));
    g_launches.fetch_add(4, std::memory_order_relaxed);
    const uint32_t *keys = dk.Current(), *vals = dv.Current();
    uint32_t *count = B->count.as<uint32_t>();
    LAUNCH(k_find_count, 1, 1, 0, st, keys, (uint32_t)total, count);
    constexpr int AB = sizeof(F) == sizeof(Fq) ? 128 : 64;     // G2 runs at 255 registers: smaller CTAs fill the SMs better
    LAUNCH((k_bucket_accum<F, chunk_of<F>(), AB>), (B->T + AB - 1) / AB, AB, 0, st, keys, vals, count, B->points.as<Affine<F>>(),
           B->buckets.as<X>(), B->pkey.as<uint32_t>(), B->ppt.as<X>());
    uint32_t *pk = B->pkey.as<uint32_t>();
    X *pp = B->ppt.as<X>();
    for (int l = 1; l <= kSegLevels; l++) {
        const size_t threads = (B->lvl_slots[l - 1] + kSeg - 1) / kSeg;
        LAUNCH((k_seg_reduce<F, kSeg>), (unsigned)((threads + 127) / 128), 128, 0, st, pk + B->lvl_off[l - 1],
               pp + B->lvl_off[l - 1], count, (uint32_t)chunk_of<F>(), (uint32_t)l, B->buckets.as<X>(), pk + B->lvl_off[l],
               pp + B->lvl_off[l]);
    }
    const size_t fin = B->lvl_slots[kSegLevels];
    LAUNCH((k_partial_merge<F>), (unsigned)((fin + 127) / 128), 128, 0, st, pk + B->lvl_off[kSegLevels],
           pp + B->lvl_off[kSegLevels], count, (uint32_t)chunk_of<F>(), (uint32_t)kSeg, (uint32_t)(kSegLevels + 1), B->buckets.as<X>(),
           B->long_list.as<uint32_t>());
    LAUNCH((k_long_run<F>), (unsigned)(fin / kMergeCap + 1), 128, 128 * sizeof(X), st, pk + B->lvl_off[kSegLevels],
           pp + B->lvl_off[kSegLevels], count, (uint32_t)chunk_of<F>(), (uint32_t)kSeg, (uint32_t)(kSegLevels + 1), B->buckets.as<X>(),
           B->long_list.as<uint32_t>());
    if (B->sets == 1) {
        const uint32_t nb1 = (B->NB + 128 * kRedSer - 1) / (128 * kRedSer);
        LAUNCH((k_red_direct1<F>), dim3(nb1, B->c), 128, 128 * sizeof(X), st, B->buckets.as<X>(), B->NB, B->out1.as<X>());
        LAUNCH((k_red_direct2<F>), B->c, 128, 128 * sizeof(X), st, B->out1.as<X>(), nb1, B->Sg.as<X>());
        LAUNCH((k_red_direct3<F>), 1, 32, 32 * sizeof(X), st, B->Sg.as<X>(), B->c, B->R.as<X>());
    } else {
    const uint32_t ng_total = B->sets * B->NG;
    LAUNCH((k_red_groups<F>), (ng_total + 127) / 128, 128, 0, st, B->buckets.as<X>(), ng_total, B->Sg.as<X>(), B->Ag.as<X>());
    LAUNCH((k_red_planes<F>), dim3(B->nblk, B->LP + 1, B->sets), 128, 128 * sizeof(X), st, B->Sg.as<X>(), B->Ag.as<X>(), B->NG,
           B->LP, B->out1.as<X>());
    LAUNCH((k_red_finish<F>), B->sets, 32, 32 * sizeof(X), st, B->out1.as<X>(), B->nblk, B->LP, B->R.as<X>());
    LAUNCH((k_horner_shift<F>), B->sets, 32, 0, st, B->R.as<X>(), B->c);
    LAUNCH((k_horner_sum<F>), 1, 32, 0, st, B->R.as<X>(), B->sets);
    }
    if (raw) CUDA_TRY(cudaMemcpyAsync(d_out, B->R.p, sizeof(X), cudaMemcpyDeviceToDevice, st));
    else LAUNCH((k_finish<F, BYTES>), 1, 1, 0, st, B->R.as<X>(), d_out);
    CUDA_TRY(cudaGetLastError());
    return LZKP_OK;
}

int msm_bases_load(int group, const uint8_t *bases, size_t n, int window_bits, int resident, int validate, MsmBases **out,
                   int canon_input) {
    MsmBases *B = new (std::nothrow) MsmBases();
    if (!B) return fail(LZKP_E_NOMEM, "host allocation failed");
    int rc = group == 1 ? bases_prepare<Fq>(B, bases, n, window_bits, resident, validate, canon_input)
                        : bases_prepare<Fq2>(B, bases, n, window_bits, resident, validate, canon_input);
    if (rc != LZKP_OK) {
        delete B;
        return rc;
    }
    *out = B;
    return LZKP_OK;
}
void msm_bases_free(MsmBases *B) { delete B; }
uint32_t msm_bases_size(const MsmBases *B) { return B->n; }
int msm_bases_group(const MsmBases *B) { return B->group; }

static int msm_device_nolock(MsmBases *B, const void *d_scalars, size_t n_used, void *d_out, cudaStream_t st, int raw = 0) {
    return B->group == 1 ? msm_run<Fq>(B, (const Fr *)d_scalars, (uint32_t)n_used, (uint8_t *)d_out, st, raw)
                         : msm_run<Fq2>(B, (const Fr *)d_scalars, (uint32_t)n_used, (uint8_t *)d_out, st, raw);
}

int msm_device(MsmBases *B, const void *d_scalars, size_t n_used, void *d_out, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(B->mu);
    return msm_device_nolock(B, d_scalars, n_used, d_out, st);
}

int msm_device_raw(MsmBases *B, const void *d_scalars, size_t n_used, void *d_out_xyzz, cudaStream_t st) {
    std::lock_guard<std::mutex> lk(B->mu);
    return msm_device_nolock(B, d_scalars, n_used, d_out_xyzz, st, 1);
}
// number of non-canonical scalars seen since the last call (device flag; synchronises the stream)
int msm_take_bad(MsmBases *B, cudaStream_t st, int *bad) {
    CUDA_TRY(cudaMemcpyAsync(bad, B->bad.p, sizeof(int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    CUDA_TRY(cudaMemsetAsync(B->bad.p, 0, sizeof(int), st));
    return LZKP_OK;
}

int msm_host(MsmBases *B, const uint8_t *scalars, size_t n_used, uint8_t *out) {
    const int bytes = B->group == 1 ? 64 : 128;
    if (n_used > B->n) return fail(LZKP_E_INVALID, "MSM: more scalars than bases");
    std::lock_guard<std::mutex> lk(B->mu);
    if (n_used) CUDA_TRY(cudaMemcpyAsync(B->d_scalars.p, scalars, n_used * 32, cudaMemcpyHostToDevice, 0));
    CUDA_TRY(cudaMemsetAsync(B->bad.p, 0, sizeof(int), 0));
    TRY(msm_device_nolock(B, B->d_scalars.p, n_used, B->d_out.p, 0));
    int bad = 0;
    CUDA_TRY(cudaMemcpy(out, B->d_out.p, bytes, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(&bad, B->bad.p, sizeof(int), cudaMemcpyDeviceToHost));
    if (bad) return fail(LZKP_E_INVALID, "MSM: " + std::to_string(bad) + " scalar(s) not canonical (>= r)");
    return LZKP_OK;
}

static int one_shot(int group, const uint8_t *bases, const uint8_t *scalars, size_t n, uint8_t *out) {
    MsmBases *B = nullptr;
    TRY(msm_bases_load(group, bases, n, 0, 0, 0, &B));
    int rc = msm_host(B, scalars, n, out);
    msm_bases_free(B);
    return rc;
}
int large_msm_g1_host(const uint8_t *bases, const uint8_t *scalars, size_t n, uint8_t *out) { return one_shot(1, bases, scalars, n, out); }
int large_msm_g2_host(const uint8_t *bases, const uint8_t *scalars, size_t n, uint8_t *out) { return one_shot(2, bases, scalars, n, out); }

}  // namespace eng
}  // namespace lzkp
