/* lzkp_b200.h — C ABI of the B200-native Groth16/BN254 proving engine for libzkp.
 *
 * Drop-in boundary (SURVEY.md §8b): these entry points are what a Rust `extern "C"`
 * FFI crate inside libzkp binds in place of the calls it makes today into
 * ark-groth16 / ark-serialize:
 *
 *   lzkp_pk_load            <- ProvingKey::<Bn254>::deserialize_uncompressed, src/backend/snark.rs:64
 *                              (and the OnceLock fill at snark.rs:295-339: upload once, keep resident)
 *   lzkp_setup /            <- Groth16::<Bn254>::circuit_specific_setup(dummy_circuit, OsRng), snark.rs:318,337
 *   lzkp_setup_builtin         (key generation when no key files exist, snark.rs:122-139); toxic waste is an input
 *   lzkp_circuit_load /     <- ConstraintSynthesizer::generate_constraints + cs.to_matrices(), done once per
 *   lzkp_circuit_builtin       circuit instead of on every prove (snark.rs:263-290, 515-584)
 *   lzkp_prove_batch        <- Groth16::<Bn254>::prove(&pk, circuit, rng) + proof.serialize_uncompressed,
 *                              snark.rs:364,369-373 and :442,447-451; n_proofs = 1 is the single-proof drop-in
 *   lzkp_prove_equality_batch / lzkp_prove_membership_batch
 *                           <- the par_iter().map(process_batch_operation) of src/advanced/batch.rs:123-131,
 *                              grouped per circuit, with the witness generated on the device
 *   lzkp_witness_map        <- LibsnarkReduction::witness_map (inside prove)        [ark-groth16, un-vendored]
 *   lzkp_msm_g1 / _g2       <- VariableBaseMSM::msm_bigint                         [ark-ec, un-vendored]
 *   lzkp_ntt                <- Radix2EvaluationDomain::{fft,ifft}_in_place, coset  [ark-poly, un-vendored]
 *   lzkp_commit_value_snark <- commit_value_snark, src/utils/commitment.rs:14-16
 *
 * Conventions
 *   - Return 0 on success, a negative LZKP_E_* code on failure.  Nothing throws or aborts across
 *     the ABI; lzkp_last_error() gives a thread-local message.  The Rust shim maps non-zero (or a
 *     non-zero per-proof status) to `vec![]`, the reference's failure convention (snark.rs:345-371).
 *   - All byte formats are ark-serialize's (SURVEY §8b): field elements 32 B canonical little-endian;
 *     G1 affine uncompressed 64 B, G2 128 B, flags in the top two bits of the last byte;
 *     Proof<Bn254> = A(G1) || B(G2) || C(G1) = 256 B; Vec<T> = u64 LE length || items.
 *   - The prover randomness r, s is an INPUT (the reference draws it from OsRng, snark.rs:363,441);
 *     the caller supplies canonical scalars.
 *   - The caller owns every buffer; the engine never frees caller memory.  Calls block until done.
 *   - There is no CPU fallback: every entry point that computes fails with LZKP_E_NO_DEVICE when
 *     no CUDA device is usable.
 */
#ifndef LZKP_B200_H
#define LZKP_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LZKP_OK 0
#define LZKP_E_INVALID (-1)    /* bad argument / malformed bytes */
#define LZKP_E_NO_DEVICE (-2)  /* CUDA device missing or unusable */
#define LZKP_E_CUDA (-3)       /* CUDA runtime error (see lzkp_last_error) */
#define LZKP_E_STATE (-4)      /* call order (e.g. prove before circuit_load) */
#define LZKP_E_NOMEM (-5)      /* device memory budget exceeded */
#define LZKP_E_UNSUPPORTED (-6)

#define LZKP_CIRCUIT_EQUALITY 0   /* param = MiMC rounds (110 = the reference's EqualityCircuit) */
#define LZKP_CIRCUIT_MEMBERSHIP 1 /* param = set slots (64 = the reference's MAX_SET_SIZE)     */

typedef struct lzkp_pk lzkp_pk;

typedef struct lzkp_pk_options {
    int window_bits;          /* fixed-base table window c in [8,17]; 0 = choose from the memory budget (<= 16) */
    uint64_t table_budget_bytes; /* cap for the resident window tables; 0 = 60% of free device memory */
    uint32_t max_chunk;       /* proofs per device pass; 0 = default (8192) */
    /* Single-proof sharding over several GPUs (large domains only): this process keeps only shard
     * `shard_index` of `shard_count` cost-weighted point ranges of the five queries.  0 / 1 = unsharded. */
    uint32_t shard_index, shard_count;
} lzkp_pk_options;
#define LZKP_PARTIAL_BYTES 768   /* 4 G1 XYZZ sums (a, b1, l, h) + 1 G2 XYZZ sum (b2), opaque device format */

/* Select the CUDA device(s) this process drives.  Idempotent; devices == NULL keeps / picks the default
 * (LOCAL_RANK, else device 0).
 *   n_devices == 1: one process per GPU (torchrun).
 *   n_devices  > 1: ONE process drives several GPUs, the shape of the reference's batch path
 *     (src/advanced/batch.rs:110-140 maps one batch over the workers of one process).  devices[0] is the primary.
 *     Every proving key loaded afterwards (resident-table mode, unsharded) is replicated on each listed device -
 *     tables, matrices, workspaces, two streams and pinned staging per device - and ONE host-buffer batch call
 *     (lzkp_prove_batch, lzkp_prove_equality_batch / _enveloped, lzkp_prove_membership_batch / _enveloped) of at
 *     least 512 proofs is cut into one contiguous block per device, each run by its own host thread, results
 *     written to disjoint slices of the caller's buffers (order preserved, no gather step).  Smaller calls, the
 *     *_device entry points, lzkp_msm*, lzkp_ntt*, lzkp_setup* and verification run on the primary device. */
int lzkp_init(const int *devices, int n_devices);
/* Devices of the list above (1 when lzkp_init was given none). */
int lzkp_device_count(void);
int lzkp_shutdown(void);
const char *lzkp_last_error(void);
/* Number of engine kernels launched by this process so far (bench.py's gpu_launches). */
uint64_t lzkp_kernel_launches(void);

/* Optional per-stage device timing (bench.py's roofline line): when enabled, every stage of the proving
 * pipeline is bracketed by two CUDA events on the stream it is launched on.  lzkp_profile_read waits for
 * the recorded events and returns accumulated milliseconds and bracket counts per region. */
#define LZKP_REGION_WITGEN 0
#define LZKP_REGION_WITNESS_MAP 1
#define LZKP_REGION_DIGITS 2
#define LZKP_REGION_MSM_G1 3
#define LZKP_REGION_MSM_G2 4
#define LZKP_REGION_ASSEMBLE 5
#define LZKP_PROFILE_REGIONS 8
int lzkp_profile_enable(int on);
int lzkp_profile_read(lzkp_pk *pk, double ms[LZKP_PROFILE_REGIONS], uint64_t count[LZKP_PROFILE_REGIONS], int reset);

/* Parse an ark-serialize uncompressed ProvingKey<Bn254> (exactly the bytes snark.rs:97-101 writes),
 * upload it, and build the resident fixed-base window tables.  validate != 0 adds the on-curve and
 * subgroup checks deserialize_uncompressed performs. */
int lzkp_pk_load(const uint8_t *pk_bytes, size_t len, int validate, lzkp_pk **out);
int lzkp_pk_load_ex(const uint8_t *pk_bytes, size_t len, int validate, const lzkp_pk_options *opt, lzkp_pk **out);
void lzkp_pk_free(lzkp_pk *pk);
/* info[0..8) = n_vars, n_inst, n_wit, domain n, window bits c, windows W, table bytes, max_chunk */
int lzkp_pk_info(const lzkp_pk *pk, uint64_t info[8]);
/* Work per proof on the batched path: work[0] / work[1] = (base, window) units of the G1 / G2 table MSMs, i.e. the
 * mixed additions one proof performs (identity points of the key are dropped at load and are not counted);
 * work[2] / work[3] = table rows (distinct bases).  Zeros for a large-domain key. */
int lzkp_pk_work(const lzkp_pk *pk, uint64_t work[4]);

/* R1CS matrices, once per circuit: CSR with m rows over z = instance || witness (column 0 = One);
 * coefficients 32 B canonical LE. */
int lzkp_circuit_load(lzkp_pk *pk, uint32_t m, uint32_t n_inst, uint32_t n_wit,
                      const uint32_t *a_rowptr, const uint32_t *a_col, const uint8_t *a_val,
                      const uint32_t *b_rowptr, const uint32_t *b_col, const uint8_t *b_val,
                      const uint32_t *c_rowptr, const uint32_t *c_col, const uint8_t *c_val);
/* The two libzkp circuits, synthesised natively (same rows/columns as generate_constraints). */
int lzkp_circuit_builtin(lzkp_pk *pk, int kind, uint32_t param);
/* Shape and CSR export of a builtin circuit without a pk (parity tests): shape = m, n_inst, n_wit,
 * nnzA, nnzB, nnzC.  Pass NULL arrays to query the shape only. */
int lzkp_builtin_circuit_csr(int kind, uint32_t param, uint64_t shape[6], uint32_t *rowptr[3], uint32_t *col[3],
                             uint8_t *val[3]);

/* Groth16 circuit-specific setup on the device.  toxic = alpha || beta || gamma || delta || tau, five
 * canonical non-zero 32 B scalars (the reference draws them from OsRng, snark.rs:310,331; the caller
 * must draw them from a CSPRNG and forget them).  Standard BN254 generators.  Outputs are ark-serialize
 * uncompressed ProvingKey<Bn254> / VerifyingKey<Bn254> (what snark.rs:97-112 persists); the buffers
 * must hold the sizes lzkp_key_sizes reports. */
int lzkp_key_sizes(uint32_t m, uint32_t n_inst, uint32_t n_wit, size_t *pk_len, size_t *vk_len);
int lzkp_setup(uint32_t m, uint32_t n_inst, uint32_t n_wit,
               const uint32_t *a_rowptr, const uint32_t *a_col, const uint8_t *a_val,
               const uint32_t *b_rowptr, const uint32_t *b_col, const uint8_t *b_val,
               const uint32_t *c_rowptr, const uint32_t *c_col, const uint8_t *c_val,
               const uint8_t toxic[160], uint8_t *pk_out, size_t pk_cap, uint8_t *vk_out, size_t vk_cap);
int lzkp_setup_builtin(int kind, uint32_t param, const uint8_t toxic[160], uint8_t *pk_out, size_t pk_cap,
                       uint8_t *vk_out, size_t vk_cap);

/* out[i] = scalars[i] * G for the standard generator of group 1 (G1, 64 B) or 2 (G2, 128 B): the fixed-base
 * primitive of the setup, also used to make synthetic MSM bases. */
int lzkp_generator_mul(int group, const uint8_t *scalars, size_t n, uint8_t *out_affine);

/* Full assignment z = instance || witness (n_vars x 32 B canonical) of a builtin circuit, computed on the host:
 * what generate_constraints assigns (snark.rs:263-290, 515-584).  Equality: value = a, other = b.  Membership:
 * value in set[0..set_len).  commitment may be NULL (then MiMC5(value) is used).  LZKP_E_INVALID when the
 * membership inputs are rejected (snark.rs:406,415-418). */
int lzkp_builtin_witness(int kind, uint32_t param, uint64_t value, uint64_t other, const uint64_t *set,
                         uint32_t set_len, const uint8_t *commitment, uint8_t *z_out, size_t z_cap);

/* n_proofs proofs from full assignments: z is n_proofs x n_vars x 32 B (z[0] = 1), r and s are
 * n_proofs x 32 B, proofs_out n_proofs x 256 B, status n_proofs ints (0 = ok). */
int lzkp_prove_batch(lzkp_pk *pk, size_t n_proofs, const uint8_t *z, const uint8_t *r, const uint8_t *s,
                     uint8_t *proofs_out, int32_t *status);
/* lzkp_prove_batch with every buffer in device memory, asynchronous on `stream`.
 * Contract of every *_device entry point: the call returns once the work is ENQUEUED on `stream`; caller buffers
 * must stay valid until `stream` has run it.  The key's internal workspaces are shared by all calls on that key:
 * the engine records a last-use event per workspace and makes the next user - any stream, any entry point,
 * host-buffer calls included - wait on it, so calls on one key from different (non-blocking) streams are ordered
 * on the device in the order they were issued and never overlap inside a workspace. */
int lzkp_prove_batch_device(lzkp_pk *pk, size_t n_proofs, const void *d_z, const void *d_r, const void *d_s,
                            void *d_proofs, void *d_status, void *stream);
/* Equality batch (prove_equality_zk x n): a, b u64; commitments n x 32 B or NULL (then MiMC5(a) is
 * computed on the device and, if commitments_out != NULL, returned).  status 1 = a != b (snark.rs:344). */
int lzkp_prove_equality_batch(lzkp_pk *pk, size_t n_proofs, const uint64_t *a, const uint64_t *b,
                              const uint8_t *commitments, const uint8_t *r, const uint8_t *s, uint8_t *proofs_out,
                              uint8_t *commitments_out, int32_t *status);
/* Membership batch (prove_membership_zk x n): sets is n x set_stride u64, set_len[i] entries used.
 * status 2 = empty / oversized set or value not in set (snark.rs:406,415-418). */
int lzkp_prove_membership_batch(lzkp_pk *pk, size_t n_proofs, const uint64_t *value, const uint64_t *sets,
                                const uint32_t *set_len, uint32_t set_stride, const uint8_t *commitments,
                                const uint8_t *r, const uint8_t *s, uint8_t *proofs_out, uint8_t *commitments_out,
                                int32_t *status);
/* The same batches with libzkp's proof envelope written on the device (SURVEY.md 8f-4), so the host shim does no
 * per-proof framing: Proof::to_bytes of src/proof/mod.rs:23-36 around the MiMC commitment computed on the device.
 *   equality   (equality_proof.rs:30-31, scheme 2): 298 B each, envelopes_out is n x 298
 *   membership (set_membership.rs:29-37, scheme 4): 10 + 4 + 8 * set_len + 256 + 32 B, rows envelope_stride apart
 * envelope_len[i] = bytes written, 0 for a failed proof (status[i] != 0). */
int lzkp_prove_equality_enveloped(lzkp_pk *pk, size_t n_proofs, const uint64_t *a, const uint64_t *b, const uint8_t *r,
                                  const uint8_t *s, uint8_t *envelopes_out, uint32_t *envelope_len, int32_t *status);
int lzkp_prove_membership_enveloped(lzkp_pk *pk, size_t n_proofs, const uint64_t *value, const uint64_t *sets,
                                    const uint32_t *set_len, uint32_t set_stride, const uint8_t *r, const uint8_t *s,
                                    uint8_t *envelopes_out, uint32_t envelope_stride, uint32_t *envelope_len,
                                    int32_t *status);
/* Same as lzkp_prove_equality_batch with every buffer already in device memory (a, b: u64[n];
 * r, s: n x 32 B; proofs: n x 256 B; status: int32[n]) on CUDA stream `stream` (cudaStream_t or NULL).
 * Asynchronous: returns after enqueueing.  Where status[i] != 0 the 256 bytes of proof i are unspecified (the
 * host-buffer calls zero them). */
int lzkp_prove_equality_batch_device(lzkp_pk *pk, size_t n_proofs, const void *d_a, const void *d_b, const void *d_r,
                                     const void *d_s, void *d_proofs, void *d_status, void *stream);

/* a3-a7 only: h_out is n_proofs x n x 32 B canonical. */
int lzkp_witness_map(lzkp_pk *pk, size_t n_proofs, const uint8_t *z, uint8_t *h_out);

/* Device-resident pieces of ONE large-domain proof, for splitting it across GPUs (one process per GPU):
 *   lzkp_witness_map_device    z -> h (for callers that want h itself)
 *   lzkp_prove_partial_device  every rank: the five MSMs over ITS point ranges -> LZKP_PARTIAL_BYTES.  phase 1 starts
 *                              the MSMs that only need z, phase 2 adds the H MSM and writes the partial sums; phase 0
 *                              or 3 = both in one call.  d_h == NULL: a shard that holds h_query points (the first
 *                              `map_ranks` shards, lzkp_pk_shard_info) runs the witness map itself from z - h is never
 *                              sent between GPUs - and needs lzkp_circuit_*; shards without h_query points skip it
 *   lzkp_prove_combine_device  one rank: add the gathered partial sums, convert A, B, C to affine and serialize
 * A partial is four G1 XYZZ sums and one G2 sum: A-range, s * A-range + r * B1-range (every shard scales its own sums
 * beside its remaining MSMs, shard 0 including alpha + a_0 and beta + b_0, so the combining rank runs no scalar
 * multiplication), L-range, H-range, B2-range.  All pointers are device pointers; calls are asynchronous on `stream`. */
int lzkp_witness_map_device(lzkp_pk *pk, const void *d_z, void *d_h, void *stream);
/* This shard's point range [first, first + count) of the queries a, b1, l, h, b2 (the +-delta extras included) and the
 * number of leading shards that run the witness map (and share the H query). */
int lzkp_pk_shard_info(const lzkp_pk *pk, uint32_t first[5], uint32_t count[5], uint32_t *map_ranks);
int lzkp_prove_partial_device(lzkp_pk *pk, const void *d_z, const void *d_r, const void *d_s, const void *d_h,
                              void *d_partial, void *d_status, void *stream, int phase);
int lzkp_prove_combine_device(lzkp_pk *pk, const void *d_partials, int n_partials, const void *d_r, const void *d_s,
                              void *d_proof, void *stream);

/* Variable-base MSM over arbitrary bases (ark affine uncompressed) and canonical scalars. */
int lzkp_msm_g1(const uint8_t *bases_affine, const uint8_t *scalars, size_t n, uint8_t *out_affine);
int lzkp_msm_g2(const uint8_t *bases_affine, const uint8_t *scalars, size_t n, uint8_t *out_affine);
/* MSM bases kept resident in HBM (what the prover does with the proving key's query vectors): upload once,
 * then run any number of MSMs against them.  group: 1 = G1 (64 B points), 2 = G2 (128 B).  window_bits in
 * [8,16], 0 = 16.  resident_windows != 0 also stores 2^(c*w) * P for every window w (W x the memory) so that
 * all windows share one bucket set.  validate != 0 checks that every point is on the curve. */
typedef struct lzkp_bases lzkp_bases;
int lzkp_bases_load(int group, const uint8_t *bases_affine, size_t n, int window_bits, int resident_windows,
                    int validate, lzkp_bases **out);
void lzkp_bases_free(lzkp_bases *b);
/* sum_{i<n} scalars[i] * base[i], n <= number of loaded bases; out_affine is 64 / 128 B. */
int lzkp_msm(lzkp_bases *b, const uint8_t *scalars, size_t n, uint8_t *out_affine);
/* Same with the scalars (n x 32 B canonical) and the output bytes in device memory; asynchronous on `stream`. */
int lzkp_msm_device(lzkp_bases *b, const void *d_scalars, size_t n, void *d_out_affine, void *stream);

/* In-place radix-2 (i)NTT over Fr on 2^log_n canonical elements, optionally on the coset 5*H. */
int lzkp_ntt(uint8_t *data, uint32_t log_n, int inverse, int coset);
/* Same transform on device buffers of 2^log_n x 32 B, asynchronous on `stream`: the result is written to
 * d_out; d_in is used as workspace (clobbered) when log_n > 11.  Elements keep the caller's representation
 * (canonical in -> canonical out, Montgomery in -> Montgomery out). */
int lzkp_ntt_device(void *d_in, void *d_out, uint32_t log_n, int inverse, int coset, void *stream);

/* Batched verification on the device (SURVEY.md 8f-3).  lzkp_vk_load parses an ark-serialize uncompressed
 * VerifyingKey<Bn254> (what snark.rs:103-112 persists) and computes e(alpha, beta) once - the reference recomputes
 * process_vk on every verify call (snark.rs:387,472).  lzkp_verify_batch decides, per proof, what
 * Proof::deserialize_uncompressed + Groth16::verify_with_processed_vk decide (snark.rs:378-400, 463-494):
 * proofs n x 256 B, public_inputs n x n_pub x 32 B canonical (equality: [commitment]; membership: [commitment,
 * set[64], is_real[64]], snark.rs:398,482-492); ok_out[i] = 1 accept, 0 reject (malformed, off-curve, outside the
 * subgroup, non-canonical, wrong input count, or failing the pairing equation).  lzkp_vk_load validates every point
 * of the key (curve and subgroup), as deserialize_uncompressed does, and prepares what ark-groth16 keeps in a
 * PreparedVerifyingKey (line coefficients of -gamma, -delta, beta) plus fixed-base byte-window tables for the
 * public-input combination: (n_pub + 2) x 522 240 B of device memory (0.52 MB per public input; 68.4 MB for membership's
 * 129 inputs, 1.07 GB for the 2049 of a 1024-slot set) plus 51 KB of prepared lines.  If they cannot be allocated the key
 * still loads; every call then runs one proof per lane, without the two forms below (lzkp_vk_info reports it).
 * Calls of up to three proofs per SM (LZKP_VERIFY_COOP_MAX, 444 on a B200) give every proof a CTA whose warps and lanes
 * share the pairing's arithmetic (one verification 1.8 ms).
 * Larger calls (LZKP_VERIFY_RLC_MIN) check groups of 64 proofs with one random linear combination
 * each (128-bit coefficients from the OS CSPRNG: one Miller loop per proof, one final exponentiation per group);
 * malformed proofs are reported individually and a failing group is re-verified proof by proof, so the decisions are
 * those of independent verification up to a soundness error of 2^-128 per group. */
typedef struct lzkp_vk lzkp_vk;
int lzkp_vk_load(const uint8_t *vk_bytes, size_t len, lzkp_vk **out);
void lzkp_vk_free(lzkp_vk *vk);
int lzkp_verify_batch(lzkp_vk *vk, size_t n, const uint8_t *proofs, const uint8_t *public_inputs, size_t n_pub,
                      uint8_t *ok_out);
/* lzkp_verify_batch with proofs, public inputs and ok in device memory of the key's device (the one it was loaded on),
 * asynchronous on `stream` (cudaStream_t or NULL): same layouts, same forms, same decisions.  Like every *_device entry
 * point it returns once the work is ENQUEUED, and the caller's buffers must stay valid until `stream` has run it; calls
 * on one key from several streams, host-buffer calls included, are ordered by the key's last-use event.  The combined
 * form's coefficients are a ChaCha20 expansion, on the device, of a 256-bit seed read from the OS at every call, and
 * groups whose combined check fails are re-verified on the device: nothing is copied to or from the host and the call
 * does not wait for the device, except when the call needs more scratch memory than the key holds - then it first waits
 * for the key's in-flight calls.
 *   LZKP_E_INVALID      a NULL buffer (n > 0), proofs or public inputs not 16-byte aligned, or a buffer that is host
 *                       memory or on another device
 *   LZKP_E_UNSUPPORTED  `stream` is being captured: the seed is drawn when the work is enqueued, so every replay of a
 *                       captured graph would reuse the same coefficients and the combined check would lose its soundness
 * A wrong n_pub enqueues a zeroing of ok (every proof rejected); n == 0 enqueues nothing. */
int lzkp_verify_batch_device(lzkp_vk *vk, size_t n, const void *d_proofs, const void *d_public_inputs, size_t n_pub,
                             void *d_ok, void *stream);
/* info[0..4) = n_pub, bytes of the byte-window tables on the device, latency form available (1/0), combined form with
 * the cooperative check available (1/0) */
int lzkp_vk_info(const lzkp_vk *vk, uint64_t info[4]);

/* ark-serialize's compressed form (Compress::Yes) next to the uncompressed one.  A compressed G1 point is x (32 B), a
 * compressed G2 point x.c0 || x.c1 (64 B), flags in the top two bits of the last byte: 0x40 = infinity, 0x80 = y is the
 * larger of y and -y (canonical integers; in Fq2 c1 first, then c0), both = invalid.  Objects keep the uncompressed
 * field order and u64 length prefixes: Proof = A(32) || B(64) || C(32) = 128 B; VerifyingKey = 232 + 32 (n_pub + 1) B.
 * Decoding takes one square root per point (Fq or Fq2), on the primary device, and checks no subgroup membership (ark's
 * deserialize_compressed_unchecked): the loaders with validation and every verifier form check the decoded points as they
 * check uncompressed ones, so decompress-then-load/verify decides what ark's validating compressed deserialization does.
 * Compressing recomputes each sign from y (the input's 0x80 bit is not read); it is format work and checks no curve.
 *
 * lzkp_pk_load_compressed / lzkp_vk_load_compressed decode the key on the device in chunks (bounded scratch, released
 * before the load) and pass the uncompressed bytes to lzkp_pk_load_ex / lzkp_vk_load: same options, validation, modes and
 * multi-GPU replicas.  LZKP_E_INVALID for a key that does not parse or has a point that does not decode.
 * lzkp_pk_compress / lzkp_vk_compress: uncompressed key bytes -> compressed; out == NULL sets *out_len only (from the
 * layout, without reading the points).  Host byte work, no device. */
int lzkp_pk_load_compressed(const uint8_t *pk_bytes, size_t len, int validate, const lzkp_pk_options *opt, lzkp_pk **out);
int lzkp_vk_load_compressed(const uint8_t *vk_bytes, size_t len, lzkp_vk **out);
int lzkp_pk_compress(const uint8_t *pk_bytes, size_t len, uint8_t *out, size_t cap, size_t *out_len);
int lzkp_vk_compress(const uint8_t *vk_bytes, size_t len, uint8_t *out, size_t cap, size_t *out_len);
/* Proofs n x 256 B <-> n x 128 B, ok_out[i] = 1 / 0.  Compressing: a row with a non-canonical coordinate or bad flags gets
 * ok 0 and 128 B of 0xFF (host, no device).  Decompressing (primary device): a row that does not decode (non-canonical x,
 * flags on x.c0, both flags, no point with that x) gets ok 0 and output bytes that every verifier form rejects as
 * malformed (0xFF over the failing point).  The *_device forms take device buffers of the primary device (any alignment)
 * and follow the contract of the other *_device entry points: enqueue-only on `stream`, LZKP_E_INVALID for a NULL buffer
 * or a buffer that is not device memory of that device when n > 0, nothing enqueued for n == 0.  They draw no randomness,
 * so a captured stream is accepted: lzkp_proofs_decompress_device then lzkp_verify_batch_device on one stream verifies
 * compressed proofs with nothing copied through the host. */
int lzkp_proofs_compress(size_t n, const uint8_t *proofs, uint8_t *out, uint8_t *ok_out);
int lzkp_proofs_decompress(size_t n, const uint8_t *in, uint8_t *proofs_out, uint8_t *ok_out);
int lzkp_proofs_compress_device(size_t n, const void *d_in, void *d_out, void *d_ok, void *stream);
int lzkp_proofs_decompress_device(size_t n, const void *d_in, void *d_proofs_out, void *d_ok, void *stream);

/* Groth16::<Bn254>::rerandomize_proof [ark-groth16, un-vendored], batched.  proofs / proofs_out n x 256 B,
 * r1 / r2 n x 32 B canonical non-zero, ok_out[i] = 1 / 0.  proofs_out may equal proofs (in place).
 * Per row, with the key's delta:  A' = r1^-1 A,  B' = r1 B + (r1 r2) delta,  C' = C + r2 A  - a fresh proof of the same
 * statement, statistically indistinguishable from a newly generated one (BKSV20, ePrint 2020/811, Thm. 3); the result is
 * written ark-serialize uncompressed (infinity flag when a point is the identity).  Like ark, the caller supplies the
 * randomness: draw r1, r2 uniformly from the non-zero residues mod r for unlinkable presentations.
 * A row gets ok 0 and 256 B of 0xFF (rejected as malformed by every verifier form), other rows unaffected, when
 *   - a coordinate is >= q, x carries a flag, or y carries both flags;
 *   - A, B or C is off its curve (the point at infinity is accepted);
 *   - B is outside the r-torsion subgroup;
 *   - r1 or r2 is 0 or >= r.
 * These are the checks of Proof::deserialize_uncompressed (validating).  The host form stages rows through device memory
 * in bounded chunks and blocks.  The *_device form takes device buffers of the key's device, proofs, factors and output
 * 16-byte aligned, and follows the contract of lzkp_verify_batch_device (enqueue-only on `stream`; LZKP_E_INVALID for a
 * NULL buffer, misalignment, host memory or another device's memory when n > 0; nothing enqueued for n == 0).  It only
 * reads the key's delta and draws no randomness: calls on one key from several streams need no ordering, and a captured
 * stream is accepted. */
int lzkp_proofs_rerandomize(lzkp_vk *vk, size_t n, const uint8_t *proofs, const uint8_t *r1, const uint8_t *r2,
                            uint8_t *proofs_out, uint8_t *ok_out);
int lzkp_proofs_rerandomize_device(lzkp_vk *vk, size_t n, const void *d_proofs, const void *d_r1, const void *d_r2,
                                   void *d_proofs_out, void *d_ok, void *stream);

/* MiMC-5 commitment of a u64 (commit_value_snark), 32 B canonical LE.  Host arithmetic, no device. */
int lzkp_commit_value_snark(uint64_t value, uint8_t out[32]);

#ifdef __cplusplus
}
#endif
#endif
