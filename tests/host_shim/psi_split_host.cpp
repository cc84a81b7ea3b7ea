// Host build of ec.cuh psi_split, checked against big-integer division by tests/test_rerandomize_host.py.
#include "../../libzkp_b200/csrc/ec.cuh"
using namespace lzkp;
extern "C" {
// n scalars of 8 little-endian limbs -> k0, k1 of 4 limbs each
void psi_split_host(const uint32_t *k, uint32_t *k0, uint32_t *k1, int n) {
    for (int i = 0; i < n; i++) {
        uint32_t s[8], a[4], b[4];
        for (int j = 0; j < 8; j++) s[j] = k[8 * i + j];
        psi_split(s, a, b);
        for (int j = 0; j < 4; j++) { k0[4 * i + j] = a[j]; k1[4 * i + j] = b[j]; }
    }
}
}
