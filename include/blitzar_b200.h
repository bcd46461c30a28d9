/* blitzar_b200 — C ABI of the B200-native MSM / Pedersen-commitment backend.
 *
 * Part 1 ("sxt_*") is the drop-in boundary: the same 18 symbols, struct layouts and argument
 * meaning as the reference's cbindings/blitzar_api.h (line numbers of the reference declaration
 * each entry replaces are cited). A consumer that was linked against libblitzar (e.g. the
 * blitzar-sys crate, rust/blitzar-sys/build.rs:21-56) links against libblitzar_b200.so unchanged.
 * All pointers are caller-owned HOST memory; calls block until results are written.
 * Misuse aborts the process with a message on stderr (reference convention, blitzar_api.h:230-237).
 *
 * Part 2 ("b200_*") is an extension for callers that already hold inputs in HBM and for the
 * one-process-per-GPU multi-GPU layout (device-resident inputs, partial results, device events).
 */
#ifndef BLITZAR_B200_H
#define BLITZAR_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- constants (blitzar_api.h:25-34) ---- */
#define SXT_CPU_BACKEND 1
#define SXT_GPU_BACKEND 2
#define SXT_CURVE_RISTRETTO255 0
#define SXT_CURVE_BLS_381 1
#define SXT_CURVE_BN_254 2
#define SXT_CURVE_GRUMPKIN 3
#define SXT_FIELD_SCALAR255 0
#define SXT_FIELD_GRUMPKIN 1

/* ---- types (blitzar_api.h:37-131) ---- */
struct sxt_config { int backend; uint64_t num_precomputed_generators; };
struct sxt_ristretto255_compressed { uint8_t ristretto_bytes[32]; };
struct sxt_bls12_381_g1_compressed { uint8_t g1_bytes[48]; };
struct sxt_curve25519_scalar { uint8_t bytes[32]; };
struct sxt_transcript { uint8_t bytes[203]; };
/* ed25519 extended coordinates, radix-2^51 limbs (not necessarily reduced) */
struct sxt_ristretto255 { uint64_t X[5]; uint64_t Y[5]; uint64_t Z[5]; uint64_t T[5]; };
/* Montgomery-form limbs, R = 2^384. NOTE: arrays of generators passed to the bls12-381 commitment
 * entry point are read with a 104-byte stride ({X, Y, uint8 infinity} padded), exactly as the
 * reference does (cbindings/pedersen.cc:215-217); see INTEGRATION.md "ABI quirks". */
struct sxt_bls12_381_g1 { uint64_t X[6]; uint64_t Y[6]; };
struct sxt_bls12_381_g1_p2 { uint64_t X[6]; uint64_t Y[6]; uint64_t Z[6]; };
/* Montgomery-form limbs, R = 2^256 */
struct sxt_bn254_g1 { uint64_t X[4]; uint64_t Y[4]; uint8_t infinity; };
struct sxt_bn254_g1_p2 { uint64_t X[4]; uint64_t Y[4]; uint64_t Z[4]; };
struct sxt_grumpkin { uint64_t X[4]; uint64_t Y[4]; uint8_t infinity; };
struct sxt_grumpkin_p2 { uint64_t X[4]; uint64_t Y[4]; uint64_t Z[4]; };
/* one column of scalars: n little-endian integers of element_nbytes (1..32) bytes; signed columns
 * are two's complement with element_nbytes a power of two <= 16 */
struct sxt_sequence_descriptor {
  uint8_t element_nbytes;
  uint64_t n;
  const uint8_t* data;
  int is_signed;
};
/* blitzar_api.h:133-183. FIELD is the field of field_id: SXT_FIELD_SCALAR255, 32 little-endian
 * bytes of an integer < l in plain form (alignment 1); SXT_FIELD_GRUMPKIN, 4 x u64 Montgomery limbs
 * (R = 2^256) of a fully reduced residue mod the bn254 scalar field (alignment 8).
 *   mles:          n x num_mles FIELD, column-major (element i of MLE j at mles[j * n + i])
 *   product_table: num_products entries laid out as std::pair<FIELD, unsigned>, i.e. (multiplier,
 *                  product_length) with a stride of 36 bytes (scalar255) or 40 bytes (grumpkin);
 *                  the length is at byte offset 32 in both
 *   product_terms: the MLE indices of every product, concatenated (num_product_terms in all) */
struct sumcheck_descriptor {
  const void* mles;
  const void* product_table;
  const unsigned* product_terms;
  unsigned n;
  unsigned num_mles;
  unsigned num_products;
  unsigned num_product_terms;
  unsigned round_degree;
};
struct sxt_multiexp_handle; /* opaque: device-resident generators of one curve */

/* ---- Part 1: drop-in entry points ---- */

/* blitzar_api.h:200. 0 on success. Only SXT_GPU_BACKEND is provided (non-zero for anything else);
 * env BLITZAR_BACKEND=gpu|cpu overrides config->backend as in cbindings/backend.cc:72-89. */
int sxt_init(const struct sxt_config* config);

/* blitzar_api.h:243. commitments[i] = sum_j a_ij * g(offset_generators + j), built-in generators */
void sxt_curve25519_compute_pedersen_commitments(struct sxt_ristretto255_compressed* commitments,
                                                 uint32_t num_sequences,
                                                 const struct sxt_sequence_descriptor* descriptors,
                                                 uint64_t offset_generators);
/* blitzar_api.h:284 */
void sxt_curve25519_compute_pedersen_commitments_with_generators(
    struct sxt_ristretto255_compressed* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_ristretto255* generators);
/* blitzar_api.h:324 (generators: 104-byte stride, see above) */
void sxt_bls12_381_g1_compute_pedersen_commitments_with_generators(
    struct sxt_bls12_381_g1_compressed* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_bls12_381_g1* generators);
/* blitzar_api.h:364 (affine Montgomery outputs; identity = {0, R mod p, infinity = 1}) */
void sxt_bn254_g1_uncompressed_compute_pedersen_commitments_with_generators(
    struct sxt_bn254_g1* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_bn254_g1* generators);
/* blitzar_api.h:404 */
void sxt_grumpkin_uncompressed_compute_pedersen_commitments_with_generators(
    struct sxt_grumpkin* commitments, uint32_t num_sequences,
    const struct sxt_sequence_descriptor* descriptors, const struct sxt_grumpkin* generators);

/* blitzar_api.h:440. ABI quirk kept: the second argument is the COUNT and the third the OFFSET,
 * as implemented and tested by the reference (cbindings/get_generators.cc:32-33), although its
 * header names them the other way round. Returns 1 if generators == NULL and count > 0. */
int sxt_ristretto255_get_generators(struct sxt_ristretto255* generators, uint64_t num_generators,
                                    uint64_t offset_generators);
/* blitzar_api.h:477. one_commit = g(0) + ... + g(n-1) (identity for n = 0) */
int sxt_curve25519_get_one_commit(struct sxt_ristretto255* one_commit, uint64_t n);

/* blitzar_api.h:566 / :611. Inner-product argument over g(generators_offset ..) with Q = g[np],
 * np = 2^ceil(log2 n); `transcript` is the caller's Merlin transcript (203 bytes), advanced in
 * place exactly as the reference advances it. verify returns 1 / 0. */
void sxt_curve25519_prove_inner_product(struct sxt_ristretto255_compressed* l_vector,
                                        struct sxt_ristretto255_compressed* r_vector,
                                        struct sxt_curve25519_scalar* ap_value,
                                        struct sxt_transcript* transcript, uint64_t n,
                                        uint64_t generators_offset,
                                        const struct sxt_curve25519_scalar* a_vector,
                                        const struct sxt_curve25519_scalar* b_vector);
int sxt_curve25519_verify_inner_product(struct sxt_transcript* transcript, uint64_t n,
                                        uint64_t generators_offset,
                                        const struct sxt_curve25519_scalar* b_vector,
                                        const struct sxt_curve25519_scalar* product,
                                        const struct sxt_ristretto255* a_commit,
                                        const struct sxt_ristretto255_compressed* l_vector,
                                        const struct sxt_ristretto255_compressed* r_vector,
                                        const struct sxt_curve25519_scalar* ap_value);

/* blitzar_api.h:631-655. generators: sxt_ristretto255 / *_p2 arrays per curve_id; copied to HBM. */
struct sxt_multiexp_handle* sxt_multiexp_handle_new(unsigned curve_id, const void* generators,
                                                    unsigned n);
struct sxt_multiexp_handle* sxt_multiexp_handle_new_from_file(unsigned curve_id,
                                                              const char* filename);
void sxt_multiexp_handle_write_to_file(const struct sxt_multiexp_handle* handle,
                                       const char* filename);
void sxt_multiexp_handle_free(struct sxt_multiexp_handle* handle);

/* blitzar_api.h:685. scalars: n rows, row i = num_outputs x element_num_bytes bytes; res: projective
 * elements (sxt_ristretto255 / *_p2), one per output. */
void sxt_fixed_multiexponentiation(void* res, const struct sxt_multiexp_handle* handle,
                                   unsigned element_num_bytes, unsigned num_outputs, unsigned n,
                                   const uint8_t* scalars);
/* blitzar_api.h:712. bit-packed rows: output j owns output_bit_table[j] consecutive bits */
void sxt_fixed_packed_multiexponentiation(void* res, const struct sxt_multiexp_handle* handle,
                                          const unsigned* output_bit_table, unsigned num_outputs,
                                          unsigned n, const uint8_t* scalars);
/* blitzar_api.h:741. as packed, output j uses only the first output_lengths[j] rows */
void sxt_fixed_vlen_multiexponentiation(void* res, const struct sxt_multiexp_handle* handle,
                                        const unsigned* output_bit_table,
                                        const unsigned* output_lengths, unsigned num_outputs,
                                        const uint8_t* scalars);
/* blitzar_api.h:766. Sumcheck proof of sum_k mult_k prod_j f_j over num_variables =
 * max(ceil_log2(n), 1) rounds. polynomials: (round_degree + 1) x num_variables FIELD, column-major
 * (round k's coefficients in ascending powers at polynomials + k (round_degree + 1));
 * evaluation_point: num_variables FIELD. transcript_callback has the C type
 *   void (FIELD* r, void* transcript_context, const FIELD* polynomial, unsigned polynomial_len)
 * and is called once per round with that round's polynomial; it must store the round's challenge in
 * *r. The callback runs while the library's lock is held: it must not call into this library.
 * Aborts with a message unless 1 <= product_length <= min(round_degree, 5) for every product, the
 * lengths add up to num_product_terms, every term is < num_mles, field_id is 0 or 1, n > 0, and the
 * MLEs plus their first fold fit in free device memory. With BLITZAR_B200_DEVICES > 1 the proof runs
 * on the primary device. */
void sxt_prove_sumcheck(void* polynomials, void* evaluation_point, unsigned field_id,
                        const struct sumcheck_descriptor* descriptor, void* transcript_callback,
                        void* transcript_context);

/* ---- Part 2: device-resident extension ---- */

/* Bind the calling thread / library to a CUDA device before sxt_init (default: current device). */
void b200_set_device(int device);
/* Number of kernels this library has launched so far in this process. */
unsigned long long b200_launch_count(void);
/* sizeof of the internal accumulator point of a curve (for partial-result buffers). */
unsigned b200_point_bytes(unsigned curve_id);
/* Raw device buffers on the library's stream-ordered pool. */
void* b200_malloc(uint64_t bytes);
void b200_free(void* device_ptr);
void b200_memcpy_h2d(void* device_dst, const void* host_src, uint64_t bytes);
void b200_memcpy_d2h(void* host_dst, const void* device_src, uint64_t bytes);
void b200_synchronize(void);
/* The cudaStream_t every kernel of the engine is launched on (e.g. to wrap it as an external stream
 * of another runtime so that collectives can be ordered against it without host synchronisation). */
void* b200_stream(void);
/* CUDA events on the library's stream (the stream every kernel of the engine is launched on). */
void* b200_event_create(void);
void b200_event_record(void* event);
float b200_event_elapsed_ms(void* start, void* stop); /* synchronises on stop */
void b200_event_destroy(void* event);

/* Variable-base MSM with every input already in HBM, laid out exactly as the host ABI lays it out
 * (descriptors[i].data and generators are DEVICE pointers; generators == NULL selects the built-in
 * ristretto generators at offset_generators). Results:
 *   out_commitments (device or NULL): canonical commitments, as the sxt_*_commitments calls write
 *   out_partials    (device or NULL): internal accumulator points (b200_point_bytes each), to be
 *                                     combined across GPUs with b200_combine_partials_device
 * Enqueued on the library stream; returns without synchronising. */
void b200_commit_device(unsigned curve_id, void* out_commitments, void* out_partials,
                        uint32_t num_sequences, const struct sxt_sequence_descriptor* descriptors,
                        const void* generators, uint64_t offset_generators);
/* The host-pointer commitment call (same copy / compute pipeline as the sxt_*_commitments entry
 * points: descriptors[i].data and generators are HOST pointers) that leaves one internal accumulator
 * point per column in DEVICE memory instead of canonical commitments — the per-rank half of a
 * generator-range-sharded multi-GPU commitment. Synchronises before returning. */
void b200_commit_host_partials(unsigned curve_id, void* out_partials, uint32_t num_sequences,
                               const struct sxt_sequence_descriptor* descriptors,
                               const void* generators, uint64_t offset_generators);
/* as the three sxt_fixed_* calls (host scalars; mode 0 fixed width, 1 packed, 2 vlen), partial
 * accumulator points to device memory */
void b200_fixed_msm_host_partials(void* out_partials, const struct sxt_multiexp_handle* handle,
                                  int mode, unsigned element_num_bytes,
                                  const unsigned* output_bit_table, const unsigned* output_lengths,
                                  unsigned num_outputs, unsigned n, const uint8_t* scalars);
/* sxt_multiexp_handle_new over generators that already sit in HBM (projective ABI structs) */
struct sxt_multiexp_handle* b200_multiexp_handle_new_device(unsigned curve_id,
                                                            const void* generators_dev,
                                                            unsigned n);
/* out[j] = sum_r partials[r * count + j]; writes canonical commitments (device pointer). */
void b200_combine_partials_device(unsigned curve_id, void* out_commitments, const void* partials,
                                  uint32_t num_parts, uint32_t count);
/* Fixed-base MSM with the scalar table already in HBM (mode 0: fixed width; 1: packed; 2: vlen as
 * in the three sxt_fixed_* calls). out_res / out_partials as above (res = projective ABI structs). */
void b200_fixed_msm_device(void* out_res, void* out_partials,
                           const struct sxt_multiexp_handle* handle, int mode,
                           unsigned element_num_bytes, const unsigned* output_bit_table,
                           const unsigned* output_lengths, unsigned num_outputs, unsigned n,
                           const uint8_t* scalars);
/* as b200_combine_partials_device but writes projective ABI structs */
void b200_combine_partials_projective_device(unsigned curve_id, void* out_res,
                                             const void* partials, uint32_t num_parts,
                                             uint32_t count);
/* Synthetic benchmark / test inputs generated in HBM (device pointer out): the generators the
 * reference's own benchmarks use — ristretto255: built-in g(first + i) as sxt_ristretto255 structs;
 * other curves: generate_random_element with fast_random_number_generator{i + 1, i + 2}
 * (cbindings/pedersen.t.cc:81-123, benchmark/multi_exp_pip/benchmark.m.cc:84-95), as projective
 * *_p2 structs (projective != 0, handle input) or affine structs at the commitment stride. */
void b200_synthetic_generators_device(unsigned curve_id, void* out_generators, uint64_t n,
                                      uint64_t first, int projective);
/* sxt_prove_sumcheck with descriptor->mles a DEVICE pointer (same column-major ABI layout, read
 * only); the product table, terms, polynomials and evaluation point stay host memory. */
void b200_prove_sumcheck_device(void* polynomials, void* evaluation_point, unsigned field_id,
                                const struct sumcheck_descriptor* descriptor,
                                void* transcript_callback, void* transcript_context);
/* Self-test of the warp-cooperative (lane-sliced) field arithmetic of the tail kernels against the
 * per-thread arithmetic on `warps` warps of pseudo-random and edge-case operands: returns the number
 * of mismatching checks (0 = pass). */
unsigned b200_selftest_lane_arithmetic(unsigned warps, unsigned seed);
/* Per-launch CUDA-event timing of the dominant kernel (level-1 bucket accumulation) on the library
 * stream: enable, run, then read the total milliseconds and launch count since the last read. */
void b200_profile_accumulate(int enable);
void b200_profile_read(float* total_ms, unsigned* launches);
/* Engine tuning (0 keeps the default): window bits c, first-level and cascade chunk lengths. */
void b200_set_tuning(unsigned window_bits, unsigned chunk1, unsigned chunkn);
/* Bucket-reduction group sizes (powers of two; 0 keeps the default): first level, later levels. */
void b200_set_reduce_groups(unsigned g1, unsigned gn);

#ifdef __cplusplus
}
#endif
#endif /* BLITZAR_B200_H */
