// chacha20.cuh — the ChaCha20 block function (RFC 8439 §2.3) for the host and the device.
//
// lzkp_verify_batch_device draws a 256-bit seed per call and expands it on the device into the combined form's 128-bit
// coefficients (k_rlc_rho in verify.cu): key = seed, nonce = 0, block counter = proof index / 4, and proof p takes the
// 16 bytes at 16 * (p % 4) of its block.  tests/host_shim/chacha_host.cpp builds this header for the host.
#pragma once
#include <stddef.h>
#include <stdint.h>

#if defined(__CUDACC__)
#define CHACHA_HD __host__ __device__ __forceinline__
#else
#define CHACHA_HD inline
#endif

namespace lzkp {

CHACHA_HD uint32_t chacha_rotl(uint32_t v, int c) { return (v << c) | (v >> (32 - c)); }

CHACHA_HD void chacha_quarter(uint32_t *x, int a, int b, int c, int d) {
    x[a] += x[b]; x[d] = chacha_rotl(x[d] ^ x[a], 16);
    x[c] += x[d]; x[b] = chacha_rotl(x[b] ^ x[c], 12);
    x[a] += x[b]; x[d] = chacha_rotl(x[d] ^ x[a], 8);
    x[c] += x[d]; x[b] = chacha_rotl(x[b] ^ x[c], 7);
}

// out[16]: the serialized block as little-endian words
CHACHA_HD void chacha20_block(const uint32_t key[8], uint32_t counter, const uint32_t nonce[3], uint32_t out[16]) {
    uint32_t s[16] = {0x61707865u, 0x3320646eu, 0x79622d32u, 0x6b206574u,
                      key[0], key[1], key[2], key[3], key[4], key[5], key[6], key[7],
                      counter, nonce[0], nonce[1], nonce[2]};
    uint32_t x[16];
#pragma unroll
    for (int i = 0; i < 16; i++) x[i] = s[i];
#pragma unroll 1
    for (int r = 0; r < 10; r++) {
        chacha_quarter(x, 0, 4, 8, 12); chacha_quarter(x, 1, 5, 9, 13);
        chacha_quarter(x, 2, 6, 10, 14); chacha_quarter(x, 3, 7, 11, 15);
        chacha_quarter(x, 0, 5, 10, 15); chacha_quarter(x, 1, 6, 11, 12);
        chacha_quarter(x, 2, 7, 8, 13); chacha_quarter(x, 3, 4, 9, 14);
    }
#pragma unroll
    for (int i = 0; i < 16; i++) out[i] = x[i] + s[i];
}

// rho[4 * q .. 4 * q + 4) for the proofs q of block `blk` (those below n): the layout k_rlc_prepare reads, 16 B per proof
// as two 64-bit halves rho_1 (words 0, 1) and rho_2 (words 2, 3)
CHACHA_HD void rlc_rho_block(const uint32_t seed[8], uint32_t blk, uint32_t n, uint32_t *rho) {
    const uint32_t nonce[3] = {0, 0, 0};
    uint32_t w[16];
    chacha20_block(seed, blk, nonce, w);
#pragma unroll
    for (uint32_t q = 0; q < 4; q++) {
        const uint32_t p = blk * 4 + q;
        if (p >= n) break;
#pragma unroll
        for (uint32_t i = 0; i < 4; i++) rho[(size_t)p * 4 + i] = w[4 * q + i];
    }
}

}  // namespace lzkp
