// Host build of chacha20.cuh, checked against RFC 8439 and the coefficient layout by tests/test_rlc_rho_host.py.
#include "../../libzkp_b200/csrc/chacha20.cuh"
using namespace lzkp;
extern "C" {
void chacha20_block_host(const uint32_t *key, uint32_t counter, const uint32_t *nonce, uint32_t *out) {
    chacha20_block(key, counter, nonce, out);
}
// what k_rlc_rho writes for n proofs: one block per thread, 16 B per proof
void rlc_rho_host(const uint32_t *seed, uint32_t n, uint32_t *rho) {
    for (uint32_t blk = 0; blk < (n + 3) / 4; blk++) rlc_rho_block(seed, blk, n, rho);
}
}
