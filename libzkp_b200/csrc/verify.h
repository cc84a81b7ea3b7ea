// verify.h — batched device-side Groth16 verification (verify.cu) and proof rerandomization (rerandomize.cu).
#pragma once
#include <mutex>
#include "common.h"

namespace lzkp {
struct Fq2;
template <class F> struct Affine;
namespace eng {
struct VerifyingKeyDev;
int vk_load(const uint8_t *bytes, size_t len, VerifyingKeyDev **out);
void vk_free(VerifyingKeyDev *v);
uint32_t vk_num_inputs(const VerifyingKeyDev *v);
void vk_info(const VerifyingKeyDev *v, uint64_t info[4]);
// -delta of the key in device memory (affine, Montgomery form); immutable from vk_load to vk_free
const Affine<Fq2> *vk_delta_neg(const VerifyingKeyDev *v);
// LZKP_E_INVALID unless p is device memory of the key's device
int check_device_buffer(const VerifyingKeyDev *v, const void *p, const char *what);
int verify_batch(VerifyingKeyDev *v, size_t n, const uint8_t *proofs, const uint8_t *inputs, size_t n_pub, uint8_t *ok_out);
int verify_batch_device(VerifyingKeyDev *v, size_t n, const uint8_t *d_proofs, const uint8_t *d_inputs, size_t n_pub, uint8_t *d_ok,
                        cudaStream_t stream);
int proofs_rerandomize(VerifyingKeyDev *v, size_t n, const uint8_t *proofs, const uint8_t *r1, const uint8_t *r2, uint8_t *proofs_out,
                       uint8_t *ok_out);
int proofs_rerandomize_device(VerifyingKeyDev *v, size_t n, const uint8_t *d_proofs, const uint8_t *d_r1, const uint8_t *d_r2,
                              uint8_t *d_proofs_out, uint8_t *d_ok, cudaStream_t stream);
}  // namespace eng
}  // namespace lzkp
