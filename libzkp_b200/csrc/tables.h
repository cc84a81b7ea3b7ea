// tables.h — entry points of tables.cu and msm_batch.cu (opaque pointers: the point types live in ec.cuh).
#pragma once
#include "common.h"

namespace lzkp {
namespace eng {

// table[(row * W + w) * N + (k-1)] = k * 2^(c*w) * base[row] (affine, Montgomery), k = 1..N = 2^(c-1)
int build_table_g1(const void *d_bases, uint32_t rows, int c, uint32_t W, uint32_t N, void *d_table, cudaStream_t st);
int build_table_g2(const void *d_bases, uint32_t rows, int c, uint32_t W, uint32_t N, void *d_table, cudaStream_t st);

// Batched table MSM (msm_batch.cu).  A "unit" is one (base, window) pair; an "item" a run of units
// of one MSM.  partial[item * P + p] receives the XYZZ sum of proof p over the item's units.
struct BatchMsmArgs {
    const void *table;            // Affine<F>[...]
    uint32_t N;
    const uint32_t *unit_dig, *unit_tbl;
    const void *items;            // uint2[n_items]
    uint32_t n_items;
    const void *msm_items;        // uint2[n_msm]
    uint32_t n_msm;
    const void *dig;             // int16_t[...] if dig_bytes == 2 (c <= 16), int32_t[...] if 4
    uint32_t dig_bytes;
    uint32_t P;
    void *partial;                // XYZZ<F>[n_items * P]
    void *out;                    // XYZZ<F>[n_msm * P]
};
void batch_msm_g1(const BatchMsmArgs &a, cudaStream_t st);
void batch_msm_g1_items(const BatchMsmArgs &a, uint32_t item0, uint32_t count, cudaStream_t st);
void batch_msm_g1_reduce(const BatchMsmArgs &a, cudaStream_t st);
void batch_msm_g2(const BatchMsmArgs &a, cudaStream_t st);
// CTAs of batch_msm_g1's large-batch gather kernel resident on the current device at once
int batch_msm_g1_resident(uint32_t dig_bytes, uint32_t *out);
// Calls of at most this many proofs take the latency-oriented shape (8-unit items, 32-thread CTAs, tree reduction);
// LZKP_SMALL_BATCH overrides the default for experiments.
uint32_t small_batch_limit();

}  // namespace eng
}  // namespace lzkp
