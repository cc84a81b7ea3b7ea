// Host build of tests/device_shim/prim_ops.h: the same operations on the portable C++ bodies of field.cuh, so the tests
// can require the device build's output to be bit-identical to this one, and can check the tower and pairing code of
// pairing.cuh against the big-integer oracle without a GPU.
#include "../device_shim/prim_ops.h"

extern "C" {
int prim_words(int family, int *in_words, int *out_words) {
    if (family < 0 || family >= prim::FAM_COUNT) return -1;
    *in_words = prim::in_words(family);
    *out_words = prim::out_words(family);
    return 0;
}
// prim_ops.h family `family`, operation `code`, on n records
void prim_run_host(int family, int code, const uint32_t *in, uint32_t *out, int n) {
    for (int i = 0; i < n; i++)
        prim::run(family, code, in + (size_t)i * prim::in_words(family), out + (size_t)i * prim::out_words(family));
}
}
