// msm_batch.cu — the five MSMs of a batch of proofs as fixed-base table gathers + XYZZ mixed adds
// (SURVEY.md §8a rows a8-a12; replaces VariableBaseMSM::msm_bigint inside ark-groth16's prover,
// reached from src/backend/snark.rs:364 and :442).
#include <algorithm>
#include <cstdlib>
#include "tables.h"
#include "dev_util.cuh"

#ifndef LZKP_G2_MINB
#define LZKP_G2_MINB 6
#endif
// minimum resident CTAs per SM: both gather kernels trade registers for warps (G2 in 64-thread CTAs)
#ifndef LZKP_G1_MINB
#define LZKP_G1_MINB 4        // 128 registers, no spills: 16 warps per SM (measured -2.5 % against 156 registers / 12 warps)
#endif
#define LZKP_G2_MINB_SEL(F) (sizeof(F) == sizeof(::lzkp::Fq) ? LZKP_G1_MINB : LZKP_G2_MINB)
namespace lzkp {

// ---------------------------------------------------------------- batched table MSM
// A "unit" is one (base, window) pair: it names a digit row and a table row.  An "item" is a
// contiguous run of units of one MSM.  Thread (p, item) gathers table[unit][|d|-1] for its proof's
// digit d of every unit in the item and accumulates in XYZZ.  Lanes of a warp are 32 different proofs
// walking the same units, so a warp-step touches one N*sizeof(point) slab (2 MiB for G1 at c=16).
template <class F, int BLOCK, class DigT>
__global__ void __launch_bounds__(BLOCK, LZKP_G2_MINB_SEL(F)) k_msm_batch(const Affine<F> *__restrict__ table, uint32_t N,
                                                     const uint32_t *__restrict__ unit_dig,
                                                     const uint32_t *__restrict__ unit_tbl,
                                                     const uint2 *__restrict__ items, const DigT *__restrict__ dig,
                                                     uint32_t P, XYZZ<F> *__restrict__ partial) {
    const uint32_t p = blockIdx.x * BLOCK + threadIdx.x, item = blockIdx.y;
    if (p >= P) return;
    const uint2 range = items[item];
    // G1 accumulates in field.cuh's redundant form (madd_lazy: no final subtraction after each product) and is made
    // canonical before it is stored.  G2 keeps the canonical madd: with the lazy one the kernel spilled 844 B instead
    // of 308 B at its 168 registers.
    constexpr bool lazy = sizeof(F) == sizeof(Fq);
    XYZZ<F> acc = XYZZ<F>::inf();
    // Software pipeline: the table point of unit u+1 is in flight under the add of unit u.  (Also keeping the digit of
    // unit u+2 in flight gained 2 % with 4-byte digits at 156 registers, but costs the fourth resident CTA: dropped.)
    int d = dig[(size_t)__ldg(unit_dig + range.x) * P + p];
    Affine<F> pt = Affine<F>::inf();
    if (d) pt = gather_point(table, N, __ldg(unit_tbl + range.x), d);
    for (uint32_t u = range.x; u < range.y; u++) {
        int dn = 0;
        Affine<F> ptn = Affine<F>::inf();
        if (u + 1 < range.y) {
            dn = dig[(size_t)__ldg(unit_dig + u + 1) * P + p];
            if (dn) ptn = gather_point(table, N, __ldg(unit_tbl + u + 1), dn);
        }
        if (d) {
            if constexpr (lazy) acc.madd_lazy(pt);
            else acc.madd(pt);
        }
        d = dn;
        pt = ptn;
    }
    if constexpr (lazy) acc = acc.canonical();
    st_vec(partial + (size_t)item * P + p, acc);
}
// Reduction of the per-item partial sums, in two launches so that the serial chain per thread stays short:
// stage 1: thread (p, q, g) folds items first+g, first+g+G, ... of MSM q into slot first+g (in place);
// stage 2: out[q * P + p] = sum of the first min(G, count) slots.
template <class F>
__global__ void __launch_bounds__(128) k_msm_reduce1(XYZZ<F> *partial, const uint2 *msm_items, uint32_t P, uint32_t G) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x, q = blockIdx.y, g = blockIdx.z;
    if (p >= P) return;
    uint2 r = msm_items[q];
    if (r.x + g >= r.y) return;
    XYZZ<F> acc = ld_vec(partial + (size_t)(r.x + g) * P + p);
    for (uint32_t it = r.x + g + G; it < r.y; it += G) acc.add_cold(ld_vec(partial + (size_t)it * P + p));
    st_vec(partial + (size_t)(r.x + g) * P + p, acc);
}
template <class F>
__global__ void __launch_bounds__(128) k_msm_reduce(const XYZZ<F> *partial, const uint2 *msm_items, uint32_t P,
                                                    uint32_t G, XYZZ<F> *out) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x, q = blockIdx.y;
    if (p >= P) return;
    uint2 r = msm_items[q];
    uint32_t end = min(r.y, r.x + G);
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t it = r.x; it < end; it++) acc.add_cold(ld_vec(partial + (size_t)it * P + p));
    st_vec(out + (size_t)q * P + p, acc);
}

// Stage 2 in log depth: one launch per level halves the live slots of every (proof, MSM) - thread (p, q, g < half)
// adds slot g + half into slot g; the last level (half == 1) writes out[q * P + p].  Replaces the serial fold of
// k_msm_reduce for large batches (G2: 16 dependent additions of ~40 products per thread were 0.29 ms of latency).
template <class F>
__global__ void __launch_bounds__(128) k_msm_fold(XYZZ<F> *partial, const uint2 *msm_items, uint32_t P, uint32_t half,
                                                  XYZZ<F> *out) {
    uint32_t p = blockIdx.x * blockDim.x + threadIdx.x, q = blockIdx.y, g = blockIdx.z;
    if (p >= P) return;
    const uint2 r = msm_items[q];
    const uint32_t live = min(r.y - r.x, 2 * half);          // slots still holding sums at this level
    if (g >= live) {
        if (half == 1 && g == 0) st_vec(out + (size_t)q * P + p, XYZZ<F>::inf());    // an MSM without items
        return;
    }
    XYZZ<F> acc = ld_vec(partial + (size_t)(r.x + g) * P + p);
    if (g + half < live) acc.add_cold(ld_vec(partial + (size_t)(r.x + g + half) * P + p));
    if (half == 1) st_vec(out + (size_t)q * P + p, acc);
    else st_vec(partial + (size_t)(r.x + g) * P + p, acc);
}

// Small batches (P <= kSmallBatch): one CTA per (proof, MSM) folds the partial sums through shared memory in
// log2(T) levels instead of two serial chains.
template <class F, int T>
__global__ void __launch_bounds__(T) k_msm_reduce_tree(const XYZZ<F> *__restrict__ partial, const uint2 *__restrict__ msm_items,
                                                       uint32_t P, XYZZ<F> *__restrict__ out) {
    __shared__ uint4 raw[T * sizeof(XYZZ<F>) / 16];
    XYZZ<F> *sm = reinterpret_cast<XYZZ<F> *>(raw);
    const uint32_t p = blockIdx.x, q = blockIdx.y, t = threadIdx.x;
    const uint2 r = msm_items[q];
    XYZZ<F> acc = XYZZ<F>::inf();
    for (uint32_t it = r.x + t; it < r.y; it += T) acc.add_cold(ld_vec(partial + (size_t)it * P + p));
    st_vec(sm + t, acc);
    __syncthreads();
    for (uint32_t s = T / 2; s > 0; s >>= 1) {
        if (t < s) {
            XYZZ<F> a = ld_vec(sm + t);
            a.add_cold(ld_vec(sm + t + s));
            st_vec(sm + t, a);
        }
        __syncthreads();
    }
    if (t == 0) st_vec(out + (size_t)q * P + p, ld_vec(sm));
}

}  // namespace lzkp

namespace lzkp {
namespace eng {
uint32_t small_batch_limit() {
    static const uint32_t v = [] {
        const char *e = getenv("LZKP_SMALL_BATCH");
        return e ? (uint32_t)atoi(e) : 512u;     // measured crossover on B200: equal at 512 proofs, 12 % slower at 1024
    }();
    return v;
}

// CTAs of the large-batch G1 gather kernel (128 threads) resident on the whole device at once
int batch_msm_g1_resident(uint32_t dig_bytes, uint32_t *out) {
    int dev = 0, sms = 0, per_sm = 0;
    CUDA_TRY(cudaGetDevice(&dev));
    CUDA_TRY(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (dig_bytes == 2) CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_msm_batch<Fq, 128, int16_t>, 128, 0));
    else CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_msm_batch<Fq, 128, int32_t>, 128, 0));
    *out = (uint32_t)std::max(1, sms * per_sm);
    return LZKP_OK;
}

// gather + accumulate the items [item0, item0 + count) (partial sums land at their global item index)
void batch_msm_g1_items(const BatchMsmArgs &a, uint32_t item0, uint32_t count, cudaStream_t st) {
    if (!count) return;
    if (a.P <= small_batch_limit()) {          // a few warps of proofs: 32-thread CTAs so that the items spread over every SM partition
        if (a.dig_bytes == 2)
            LAUNCH((k_msm_batch<Fq, 32, int16_t>), dim3((a.P + 31) / 32, count), 32, 0, st, (const G1Affine *)a.table, a.N, a.unit_dig, a.unit_tbl,
                   (const uint2 *)a.items + item0, (const int16_t *)a.dig, a.P, (G1XYZZ *)a.partial + (size_t)item0 * a.P);
        else
            LAUNCH((k_msm_batch<Fq, 32, int32_t>), dim3((a.P + 31) / 32, count), 32, 0, st, (const G1Affine *)a.table, a.N, a.unit_dig, a.unit_tbl,
                   (const uint2 *)a.items + item0, (const int32_t *)a.dig, a.P, (G1XYZZ *)a.partial + (size_t)item0 * a.P);
        return;
    }
    if (a.dig_bytes == 2)
        LAUNCH((k_msm_batch<Fq, 128, int16_t>), dim3((a.P + 127) / 128, count), 128, 0, st, (const G1Affine *)a.table, a.N, a.unit_dig,
               a.unit_tbl, (const uint2 *)a.items + item0, (const int16_t *)a.dig, a.P, (G1XYZZ *)a.partial + (size_t)item0 * a.P);
    else
        LAUNCH((k_msm_batch<Fq, 128, int32_t>), dim3((a.P + 127) / 128, count), 128, 0, st, (const G1Affine *)a.table, a.N, a.unit_dig,
               a.unit_tbl, (const uint2 *)a.items + item0, (const int32_t *)a.dig, a.P, (G1XYZZ *)a.partial + (size_t)item0 * a.P);
}
constexpr uint32_t kReduceFan = 8;
void batch_msm_g1_reduce(const BatchMsmArgs &a, cudaStream_t st) {
    if (a.P <= small_batch_limit()) {
        LAUNCH((k_msm_reduce_tree<Fq, 128>), dim3(a.P, a.n_msm), 128, 0, st, (const G1XYZZ *)a.partial, (const uint2 *)a.msm_items,
               a.P, (G1XYZZ *)a.out);
        return;
    }
    LAUNCH((k_msm_reduce1<Fq>), dim3((a.P + 127) / 128, a.n_msm, kReduceFan), 128, 0, st, (G1XYZZ *)a.partial,
           (const uint2 *)a.msm_items, a.P, kReduceFan);
    for (uint32_t half = kReduceFan / 2; half >= 1; half >>= 1)
        LAUNCH((k_msm_fold<Fq>), dim3((a.P + 127) / 128, a.n_msm, half), 128, 0, st, (G1XYZZ *)a.partial,
               (const uint2 *)a.msm_items, a.P, half, (G1XYZZ *)a.out);
}
void batch_msm_g1(const BatchMsmArgs &a, cudaStream_t st) {
    batch_msm_g1_items(a, 0, a.n_items, st);
    batch_msm_g1_reduce(a, st);
}
void batch_msm_g2(const BatchMsmArgs &a, cudaStream_t st) {
    if (a.P <= small_batch_limit()) {
        if (a.dig_bytes == 2)
            LAUNCH((k_msm_batch<Fq2, 32, int16_t>), dim3((a.P + 31) / 32, a.n_items), 32, 0, st, (const G2Affine *)a.table, a.N, a.unit_dig,
                   a.unit_tbl, (const uint2 *)a.items, (const int16_t *)a.dig, a.P, (G2XYZZ *)a.partial);
        else
            LAUNCH((k_msm_batch<Fq2, 32, int32_t>), dim3((a.P + 31) / 32, a.n_items), 32, 0, st, (const G2Affine *)a.table, a.N, a.unit_dig,
                   a.unit_tbl, (const uint2 *)a.items, (const int32_t *)a.dig, a.P, (G2XYZZ *)a.partial);
        LAUNCH((k_msm_reduce_tree<Fq2, 128>), dim3(a.P, a.n_msm), 128, 0, st, (const G2XYZZ *)a.partial, (const uint2 *)a.msm_items,
               a.P, (G2XYZZ *)a.out);
        return;
    }
    if (a.dig_bytes == 2)
        LAUNCH((k_msm_batch<Fq2, 64, int16_t>), dim3((a.P + 63) / 64, a.n_items), 64, 0, st, (const G2Affine *)a.table, a.N,
               a.unit_dig, a.unit_tbl, (const uint2 *)a.items, (const int16_t *)a.dig, a.P, (G2XYZZ *)a.partial);
    else
        LAUNCH((k_msm_batch<Fq2, 64, int32_t>), dim3((a.P + 63) / 64, a.n_items), 64, 0, st, (const G2Affine *)a.table, a.N,
               a.unit_dig, a.unit_tbl, (const uint2 *)a.items, (const int32_t *)a.dig, a.P, (G2XYZZ *)a.partial);
    LAUNCH((k_msm_reduce1<Fq2>), dim3((a.P + 127) / 128, a.n_msm, 2 * kReduceFan), 128, 0, st, (G2XYZZ *)a.partial,
           (const uint2 *)a.msm_items, a.P, 2 * kReduceFan);
    for (uint32_t half = kReduceFan; half >= 1; half >>= 1)
        LAUNCH((k_msm_fold<Fq2>), dim3((a.P + 127) / 128, a.n_msm, half), 128, 0, st, (G2XYZZ *)a.partial,
               (const uint2 *)a.msm_items, a.P, half, (G2XYZZ *)a.out);
}

}  // namespace eng
}  // namespace lzkp
