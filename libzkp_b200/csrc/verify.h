// verify.h — batched device-side Groth16 verification (verify.cu).
#pragma once
#include <mutex>
#include "common.h"

namespace lzkp {
namespace eng {
struct VerifyingKeyDev;
int vk_load(const uint8_t *bytes, size_t len, VerifyingKeyDev **out);
void vk_free(VerifyingKeyDev *v);
uint32_t vk_num_inputs(const VerifyingKeyDev *v);
void vk_info(const VerifyingKeyDev *v, uint64_t info[4]);
int verify_batch(VerifyingKeyDev *v, size_t n, const uint8_t *proofs, const uint8_t *inputs, size_t n_pub, uint8_t *ok_out);
int verify_batch_device(VerifyingKeyDev *v, size_t n, const uint8_t *d_proofs, const uint8_t *d_inputs, size_t n_pub, uint8_t *d_ok,
                        cudaStream_t stream);
}  // namespace eng
}  // namespace lzkp
