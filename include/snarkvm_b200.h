/*
 * snarkvm_b200 — C ABI of the B200 (sm_100a) proving backend for snarkVM's two hot paths:
 *   VariableBase::msm over BLS12-377 G1 and the radix-2 EvaluationDomain NTT over Fr.
 *
 * PART 1 is the drop-in boundary: the three symbols the reference's Rust FFI binds
 * (declared at /root/reference/algorithms/cuda/src/lib.rs:42-69, defined by the reference at
 * algorithms/cuda/cuda/snarkvm_api.cu:52-84).  Same names, argument order, data layouts and
 * error convention, so `snarkvm-algorithms-cuda` links against this library unchanged
 * (see INTEGRATION.md).
 *
 * PART 2 is the extended, device-resident API (pointers already in HBM) used by the
 * host mirror, bench.py and multi-GPU sharding.
 *
 * Data layouts (identical to the reference's in-memory Rust types):
 *   Fr element   : 32 B, 4 x u64 little-endian limbs, Montgomery form  (fields/src/fp_256.rs:52)
 *   MSM scalar   : 32 B, canonical integer < r, NOT Montgomery         (BigInteger256; snarkvm.cu:275 mont=false)
 *   G1 affine    : x[48] y[48] (Montgomery Fq) infinity[1] pad -> 104-byte stride
 *                  (curves/src/templates/short_weierstrass_jacobian/affine.rs:41-46; lib.rs:161)
 *   G1 projective: X[48] Y[48] Z[48] Jacobian, infinity <=> Z == 0     (projective.rs:36-60)
 */
#ifndef SNARKVM_B200_H
#define SNARKVM_B200_H

#include <stddef.h>
#include <stdint.h>

#if defined(__GNUC__)
#define SNARKVM_API __attribute__((visibility("default")))
#else
#define SNARKVM_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

/* ------------------------------------------------------------------------------------------
 * PART 1 — drop-in replacements for the reference FFI
 * ---------------------------------------------------------------------------------------- */

/* #[repr(C)] enums of algorithms/cuda/src/lib.rs:22-40 */
typedef enum { SNARKVM_NTT_NN = 0, SNARKVM_NTT_NR = 1, SNARKVM_NTT_RN = 2, SNARKVM_NTT_RR = 3 } snarkvm_ntt_order_t;
typedef enum { SNARKVM_NTT_FORWARD = 0, SNARKVM_NTT_INVERSE = 1 } snarkvm_ntt_direction_t;
typedef enum { SNARKVM_NTT_STANDARD = 0, SNARKVM_NTT_COSET = 1 } snarkvm_ntt_type_t;

/* `cuda::Error` of sppark::cuda_error!() (lib.rs:19), returned BY VALUE.  The Rust side reads
 * .code (lib.rs:93,141,164; 0 = success, otherwise a cudaError_t) and frees .message, which is
 * therefore malloc()ed or NULL (shape evidenced at algorithms/cuda/cuda/snarkvm.cu:279). */
typedef struct {
    int code;
    char* message;
} snarkvm_error_t;

/* Replaces `snarkvm_ntt` (lib.rs:43-49 ; snarkvm_api.cu:53-62 ; called from
 * algorithms/src/fft/domain.rs:375-388, 404-417, 425-438).  In-place transform of 2^lg_domain_size
 * Fr elements in HOST memory.  NN (the only order any reference caller passes) is native; NR / RN / RR
 * add explicit bit-reversal passes (R = bit-reversed index order on that side).  On failure `inout` is
 * left untouched and a non-zero cudaError_t is returned, which makes the Rust caller fall back to CPU. */
SNARKVM_API snarkvm_error_t snarkvm_ntt(void* inout, uint32_t lg_domain_size, snarkvm_ntt_order_t ntt_order,
                            snarkvm_ntt_direction_t ntt_direction, snarkvm_ntt_type_t ntt_type);

/* Replaces `snarkvm_polymul` (lib.rs:51-60 ; snarkvm_api.cu:64-75 ; called from
 * algorithms/src/fft/polynomial/multiplier.rs:79-95).  out[2^lg] = iNTT( prod NTT(pad(poly_i)) * prod eval_j ).
 * polynomials: const Fr* [pcount] with lengths plens[] (<= 2^lg); evaluations: const Fr* [ecount] in natural
 * order with elens[] == 2^lg.  0 operands: success, out untouched. */
SNARKVM_API snarkvm_error_t snarkvm_polymul(void* out, size_t pcount, const void* polynomials, const void* plens, size_t ecount,
                                const void* evaluations, const void* elens, uint32_t lg_domain_size);

/* Replaces `snarkvm_msm` (lib.rs:62-68 ; snarkvm_api.cu:77-83 ; called from
 * algorithms/src/msm/variable_base/mod.rs:33-42).  out (144 B) = sum scalars[i] * points[i], i < npoints.
 * The result is written NORMALISED (Z = Montgomery one, or (0, R, 0) for infinity), i.e. the bytes of
 * `reference_result.to_affine().to_projective()`. */
SNARKVM_API snarkvm_error_t snarkvm_msm(void* out, const void* points_with_infinity, size_t npoints, const void* scalars,
                            size_t ffi_affine_sz);

/* ------------------------------------------------------------------------------------------
 * PART 2 — extended API.  `d_` pointers are device pointers on the CURRENT device; `stream` is a
 * cudaStream_t (NULL = legacy default stream).  All functions return 0 or a cudaError_t.
 * ---------------------------------------------------------------------------------------- */

SNARKVM_API const char* snarkvm_b200_version(void);
/* number of CUDA kernels this library has launched in this process (bench.py's gpu_launches) */
SNARKVM_API uint64_t snarkvm_b200_launch_count(void);

/* In-place transform of 2^lg Fr elements resident in HBM (any of the four orders).  d_scratch: 2^lg elements or NULL. */
SNARKVM_API int snarkvm_b200_ntt_device(void* d_inout, uint32_t lg, int ntt_order, int ntt_direction, int ntt_type,
                            void* d_scratch, void* stream);

/* Device-resident polymul: d_out[2^lg]; polys/evals are HOST arrays of device pointers. */
SNARKVM_API int snarkvm_b200_polymul_device(void* d_out, size_t pcount, const void* const* d_polys, const size_t* plens,
                                size_t ecount, const void* const* d_evals, const size_t* elens, uint32_t lg,
                                void* stream);

/* Window/bucket plan the MSM will use for npoints (signed c-bit digits). */
SNARKVM_API int snarkvm_b200_msm_plan(size_t npoints, int* c, int* nwin, uint32_t* cap);
/* batched-affine pair levels the plan for `npoints` runs before the XYZZ accumulation (0 = gather + XYZZ only) */
SNARKVM_API int snarkvm_b200_msm_plan_levels(size_t npoints);

/* Full MSM with bases and scalars resident in HBM; out144 is HOST memory (normalised projective). */
SNARKVM_API int snarkvm_b200_msm_device(void* out144, const void* d_points, size_t npoints, const void* d_scalars,
                            size_t stride, void* stream);

/* `count` MSMs over the SAME resident bases in ONE pass (all commitments of a prover round share powers_of_beta_g,
 * polycommit/sonic_pc/mod.rs:177-257): one digit/sort keyed by (vector, window, bucket), one set of pair levels, one D2H and one
 * synchronisation.  d_scalars / nscalars: HOST arrays of device pointers / lengths (canonical 32-byte integers);
 * out144s: count * 144 B of HOST memory.  Vector i uses the first nscalars[i] bases. */
SNARKVM_API int snarkvm_b200_msm_batch_device(void* out144s, const void* d_points, size_t stride, const void* const* d_scalars,
                                              const size_t* nscalars, size_t count, void* stream);

/* MSM pieces for multi-GPU sharding: per-window sums as XYZZ points (192 B each) in HBM ... */
SNARKVM_API int snarkvm_b200_msm_window_sums_device(void* d_window_sums /* nwin * 192 B */, const void* d_points, size_t npoints,
                                        const void* d_scalars, size_t stride, void* stream);
/* ... under the plan of `plan_npoints` >= npoints: every rank of a sharded MSM passes the size of the LARGEST shard, so all ranks
 * use the same window size and window count whatever their own shard length (snarkvm_b200_msm_plan(plan_npoints) gives nwin and c);
 * an empty shard (npoints = 0) contributes infinity sums.  d_flags: device u32 that receives bit 0 = "a scalar has bits 253..255
 * set" (the sums are then meaningless), or NULL to ignore. */
SNARKVM_API int snarkvm_b200_msm_window_sums_plan_device(void* d_window_sums, uint32_t* d_flags, size_t plan_npoints, const void* d_points,
                                                         size_t npoints, const void* d_scalars, size_t stride, void* stream);
/* ... the same from HOST buffers: uploads the shard (point ranges overlapped with the kernels of the previous range, pageable sources
 * staged through pinned buffers) and leaves its window sums in HBM without synchronising, so a collective can follow at once. */
SNARKVM_API int snarkvm_b200_msm_window_sums_host(void* d_window_sums, uint32_t* d_flags, size_t plan_npoints, const void* h_points,
                                                  size_t npoints, const void* h_scalars, size_t stride, void* stream);
/* ... summed across ranks after an all-gather: d_out[i] = sum_r d_in[r][i] ... */
SNARKVM_API int snarkvm_b200_xyzz_sum_ranks_device(void* d_out, const void* d_in, int nranks, int count, void* stream);
/* ... and folded on the host: out144 = sum_w 2^(c*w) * window_sums[w]  (h_window_sums in HOST memory). */
SNARKVM_API int snarkvm_b200_msm_finish(void* out144, const void* h_window_sums, int nwin, int c);

/* KZG10::commit core (algorithms/src/polycommit/kzg10/mod.rs:98-156): Montgomery coefficients ->
 * canonical (to_bigint, :455-474) -> MSM against resident powers.  out144 is HOST memory. */
SNARKVM_API int snarkvm_b200_kzg_commit_device(void* out144, const void* d_powers, size_t stride, const void* d_coeffs_mont,
                                   size_t ncoeffs, void* stream);

/* Fixed base sets (an SRS kept in HBM across many commitments): precompute the tables 2^(c*w) * P_i, w < nwin, once; every MSM
 * over those bases then uses ONE bucket set for all windows (c = 22, 12 windows at 2^24 points instead of 17 / 15).  The handle owns
 * npoints * nwin * 128 bytes of HBM (25.8 GB at 2^24).  nscalars <= npoints selects the prefix P_0..P_{nscalars-1}
 * (`&powers_of_beta_g[..len]`, polycommit/kzg10/mod.rs:121-135).  Results are the same group elements as snarkvm_b200_msm_device. */
SNARKVM_API int snarkvm_b200_msm_precompute_device(void** handle_out, const void* d_points, size_t npoints, size_t stride, void* stream);
SNARKVM_API int snarkvm_b200_msm_precomputed_free(void* handle);
SNARKVM_API int snarkvm_b200_msm_precomputed_info(const void* handle, size_t* npoints, int* c, int* nwin, size_t* table_bytes);
SNARKVM_API int snarkvm_b200_msm_precomputed_device(void* out144, const void* handle, const void* d_scalars, size_t nscalars, void* stream);
SNARKVM_API int snarkvm_b200_kzg_commit_precomputed_device(void* out144, const void* handle, const void* d_coeffs_mont, size_t ncoeffs,
                                                           void* stream);

/* KZG10::commit with hiding_bound = Some(_) (polycommit/kzg10/mod.rs:98-156): MSM(powers_of_beta_g, coeffs) +
 * MSM(powers_of_beta_times_gamma_g, blinding coefficients).  The caller samples the blinding polynomial; all coefficient arrays are
 * Montgomery Fr in HBM; nblinding = 0 gives the plain commitment. */
SNARKVM_API int snarkvm_b200_kzg_commit_hiding_device(void* out144, const void* d_powers, size_t stride, const void* d_coeffs_mont,
                                                      size_t ncoeffs, const void* d_gamma_powers, const void* d_blinding_mont,
                                                      size_t nblinding, void* stream);
/* `count` commitments against the same resident powers in ONE pass (one prover round, polycommit/sonic_pc/mod.rs:177-257).
 * d_coeffs_mont / ncoeffs: HOST arrays of device pointers / lengths; out144s: count * 144 B of HOST memory. */
SNARKVM_API int snarkvm_b200_kzg_commit_batch_device(void* out144s, const void* d_powers, size_t stride, const void* const* d_coeffs_mont,
                                                     const size_t* ncoeffs, size_t count, void* stream);
/* ... with hiding bounds: polynomial i also gets sum_j blinding_i[j] * gamma_powers[j] (nblinding[i] = 0: plain commitment);
 * the blinding terms ride in the same pass as a second scalar segment of the same sum. */
SNARKVM_API int snarkvm_b200_kzg_commit_batch_hiding_device(void* out144s, const void* d_powers, size_t stride,
                                                            const void* const* d_coeffs_mont, const size_t* ncoeffs,
                                                            const void* d_gamma_powers, const void* const* d_blinding_mont,
                                                            const size_t* nblinding, size_t count, void* stream);
/* ... over the precomputed tables of the resident powers (one bucket set per polynomial). */
SNARKVM_API int snarkvm_b200_kzg_commit_batch_precomputed_device(void* out144s, const void* handle, const void* const* d_coeffs_mont,
                                                                 const size_t* ncoeffs, size_t count, void* stream);

/* SonicKZG10::commit for all polynomials of a round (polycommit/sonic_pc/mod.rs:177-257) in one pass: polynomial i is committed
 * against d_bases[i] — the powers (ck.powers()), the powers advanced by max_degree - degree_bound points
 * (ck.shifted_powers_of_beta_g(degree_bound), sonic_pc/data_structures.rs:310-331) or a Lagrange basis (mod.rs:215-227) — plus, when
 * nblinding[i] > 0, sum_j blinding_i[j] * d_gamma_bases[i][j] (hiding_bound = Some(_), kzg10/mod.rs:129-150).  Base slices may
 * overlap (they are merged); all arrays share `stride`.  d_gamma_bases / d_blinding_mont / nblinding may be NULL (no hiding). */
SNARKVM_API int snarkvm_b200_sonic_commit_batch_device(void* out144s, size_t stride, const void* const* d_bases,
                                                       const void* const* d_coeffs_mont, const size_t* ncoeffs,
                                                       const void* const* d_gamma_bases, const void* const* d_blinding_mont,
                                                       const size_t* nblinding, size_t count, void* stream);

/* MSM scratch budget of the current device (bytes): the limit concurrent calls share (half the device unless
 * SNARKVM_B200_SCRATCH_LIMIT_GB is set; callers that do not fit wait instead of failing), what is in flight, and the high-water mark. */
SNARKVM_API int snarkvm_b200_msm_scratch_stats(size_t* limit_bytes, size_t* in_use_bytes, size_t* peak_bytes);
/* change the limit at run time (also resets the high-water mark) */
SNARKVM_API int snarkvm_b200_msm_set_scratch_limit(size_t limit_bytes);

/* FFT over G1 points (EvaluationDomain::{fft,ifft} with T = G1Projective, fft/domain.rs:169-221): 2^lg affine points in, affine
 * points out, natural order.  direction 1 = inverse, which is UniversalParams::lagrange_basis
 * (polycommit/kzg10/data_structures.rs:68-72): the commitment key for commit_lagrange (kzg10/mod.rs:159-206). */
SNARKVM_API int snarkvm_b200_g1_ntt_device(void* d_out, size_t out_stride, const void* d_in, size_t in_stride, uint32_t lg, int direction,
                                           void* stream);

/* batch_inversion_and_mul (fields/src/lib.rs:78-129): v_i <- coeff * v_i^{-1} in place, zeros stay zero.  coeff: 32 B HOST. */
SNARKVM_API int snarkvm_b200_fr_batch_inversion_and_mul_device(void* d_v, size_t n, const void* coeff_mont_host, void* stream);
/* DensePolynomial::divide_by_vanishing_poly (fft/polynomial/dense.rs:162-169): p (m coefficients) = q * (x^n - 1) + r;
 * d_q receives max(m - n, 0) coefficients, d_r receives min(m, n) (neither trimmed). */
SNARKVM_API int snarkvm_b200_poly_divide_by_vanishing_device(void* d_q, void* d_r, const void* d_p, size_t m, size_t n, void* stream);
/* KZG10::compute_witness_polynomial (polycommit/kzg10/mod.rs:220-241): quotient of p (m coefficients) / (x - point); d_q receives
 * m - 1 coefficients; the remainder p(point) is dropped as in the reference.  point: 32 B Montgomery, HOST. */
SNARKVM_API int snarkvm_b200_poly_divide_by_linear_device(void* d_q, const void* d_p, size_t m, const void* point_mont_host, void* stream);
/* z_M = M * (public || private) for a sparse R1CS matrix (inner_product, snark/varuna/ahp/prover/round_functions/mod.rs:169-189,
 * called per row of A, B, C at :128-152).  CSR in HBM: row_ptr = nrows + 1 u32, cols = u32 indices into d_x (nvars Montgomery Fr),
 * vals = Montgomery Fr.  A column >= nvars makes the call return cudaErrorInvalidValue. */
SNARKVM_API int snarkvm_b200_sparse_matvec_device(void* d_out, const void* d_row_ptr, const void* d_cols, const void* d_vals, size_t nrows,
                                                  const void* d_x, size_t nvars, void* stream);
/* Elementwise Fr arithmetic on HBM vectors (the zip loops between transforms, e.g. polycommit/kzg10/mod.rs:292-297,
 * fft/evaluations.rs:49-74): op 0 = a + b, 1 = a - b, 2 = a * b; out may alias an input; the scalar form takes a 32-byte HOST scalar. */
SNARKVM_API int snarkvm_b200_fr_vec_op_device(void* d_out, const void* d_a, const void* d_b, size_t n, int op, void* stream);
SNARKVM_API int snarkvm_b200_fr_vec_scalar_op_device(void* d_out, const void* d_a, const void* scalar_mont_host, size_t n, int op, void* stream);
/* EvaluationDomain::elements (fft/domain.rs:307-309): d_out[i] = group_gen^i, i < 2^lg, Montgomery. */
SNARKVM_API int snarkvm_b200_domain_elements_device(void* d_out, uint32_t lg, void* stream);
/* The indexer's arithmetization of A, B, C (matrix_evals, snark/varuna/ahp/matrices.rs:138-190) in one launch.  Matrix m (0 = A,
 * 1 = B, 2 = C) is CSR in HBM: d_row_ptr[m] = num_constraints + 1 u32 offsets, d_cols[m] = nnz[m] u32 variable indices (public
 * first), d_vals[m] = nnz[m] Montgomery Fr; its non-zero domain K_m has 2^lg_k[m] >= nnz[m] elements.  The constraint and variable
 * domains are the next powers of two of num_constraints and num_variables; num_public (a power of two, smaller than the variable
 * domain) is the input domain columns are reindexed by (fft/domain.rs:322-344).  Slots past nnz[m] are the padding (1, 1, 1, 0).
 *   mode 0 (materialise): d_io[4m + j] (K_m Montgomery Fr each) receives row, col, row_col, row_col_val for j = 0..3.
 *   mode 1 (evaluate):    d_io[m] holds the Lagrange coefficients of K_m at a point (evaluate_all_lagrange_coefficients);
 *                         sums_mont_host (HOST, 12 x 32 B) receives sum_k L_k * e_j(k) at index 4m + j, the verifier's
 *                         evaluate_index_polynomials (ahp/indexer/indexer.rs:232-260), without storing the evaluations.
 * A malformed row_ptr, a column >= num_variables or nnz[m] > 2^lg_k[m] returns cudaErrorInvalidValue.  Synchronises the stream. */
SNARKVM_API int snarkvm_b200_index_arithmetize_device(int mode, const void* const* d_row_ptr, const void* const* d_cols,
                                                      const void* const* d_vals, const size_t* nnz, const uint32_t* lg_k,
                                                      size_t num_constraints, size_t num_variables, size_t num_public, void* const* d_io,
                                                      void* sums_mont_host, void* stream);
/* DensePolynomial::evaluate (fft/polynomial/dense.rs:98-114): out = sum c_i * point^i; out and point are 32-byte HOST buffers. */
SNARKVM_API int snarkvm_b200_poly_evaluate_device(void* out_mont_host, const void* d_coeffs, size_t m, const void* point_mont_host,
                                                  void* stream);

/* Fr Montgomery <-> canonical, n elements in HBM (to_bigint / from_bigint, fields/src/fp_256.rs:362-413). */
SNARKVM_API int snarkvm_b200_fr_from_mont_device(void* d_out, const void* d_in, size_t n, void* stream);
SNARKVM_API int snarkvm_b200_fr_to_mont_device(void* d_out, const void* d_in, size_t n, void* stream);

/* SRS ingest: npoints uncompressed canonical G1 points as stored in a `.usrs` file after its 8-byte count (x LE 48 B, y LE 48 B,
 * bit 6 of the last byte = infinity; parameters/src/mainnet/powers.rs, utilities/src/serialize/flags.rs:72-98) -> the reference's
 * Affine images (Montgomery, `stride` bytes apart) in HBM.  *d_invalid (device u32) receives the number of points that are
 * out of range, off the curve y^2 = x^3 + 1 or badly flagged.  d_in96 must be 4-byte aligned. */
SNARKVM_API int snarkvm_b200_srs_decode_device(void* d_out, size_t stride, const void* d_in96, size_t npoints, uint32_t* d_invalid, void* stream);

/* Resident bases for the drop-in snarkvm_msm: upload `host_points` (npoints x stride bytes) to the current device once;
 * later snarkvm_msm calls whose `points_with_infinity` is this same pointer (same stride, npoints <= registered) skip the
 * upload.  The SRS powers of a proving key are constant (polycommit/sonic_pc/data_structures.rs:41-63) and the reference
 * passes the same slice to every commitment.  The caller must not mutate the slice while it is registered. */
SNARKVM_API int snarkvm_b200_register_bases(const void* host_points, size_t npoints, size_t stride);
SNARKVM_API int snarkvm_b200_unregister_bases(const void* host_points);
/* As snarkvm_b200_register_bases, and also builds the fixed-base tables (snarkvm_b200_msm_precompute_device) of the uploaded copy:
 * snarkvm_msm calls on this slice then run over the tables (npoints * nwin * 128 B of HBM, seconds of one-off set-up). */
SNARKVM_API int snarkvm_b200_register_bases_precomputed(const void* host_points, size_t npoints, size_t stride);

/* Per-kernel CUDA-event timing on the launching stream (off by default).  kind: 0 = MSM bucket sort
 * (digit histogram + scatter), 1 = MSM bucket accumulation, 2 = MSM bucket reduction, 3 = NTT passes.
 * collect() waits for the recorded launches of that kind, returns their summed milliseconds and count, and
 * clears them. */
SNARKVM_API int snarkvm_b200_profile_enable(int on);
SNARKVM_API int snarkvm_b200_profile_collect(int kind, double* total_ms, uint64_t* count);

/* Device self-test of the warp-cooperative Fq multiplication / inversion used by the CTA-shared inversions: nwarps pseudo-random cases
 * (plus 0, 1, q - 1 and a long-carry value) checked against the per-thread multiplier; *mismatches (HOST) = failing cases. */
SNARKVM_API int snarkvm_b200_selftest_coop(uint32_t nwarps, uint64_t seed, uint32_t* mismatches, void* stream);
/* host-only self-test of the pageable-memory staging copies (copy-thread pool, non-temporal stores); needs no GPU */
SNARKVM_API int snarkvm_b200_selftest_host_copy(size_t max_bytes, uint64_t seed, uint32_t* mismatches);

/* Deterministic synthetic bases P_i = h(seed, i) * G written in the reference affine layout. */
/* ---- G2 (points over Fq2) ----------------------------------------------------------------------------------------------
 * VariableBase::msm for Affine<G2> — the type the reference dispatches to standard::msm
 * (algorithms/src/msm/variable_base/mod.rs:44-47, standard.rs:79-118).  Point layout: x.c0 x.c1 y.c0 y.c1 (4 × 48 B Montgomery
 * Fq), infinity flag, padding: stride ≥ 200 (curves/src/templates/short_weierstrass_jacobian/affine.rs:41-46 over Fq2);
 * scalars: canonical 32-byte integers.  Result: 288 bytes, Projective<G2> X Y Z over Fq2, normalised (Z = 1, or (0, 1, 0)). */
SNARKVM_API snarkvm_error_t snarkvm_b200_msm_g2(void* out288, const void* points, size_t npoints, const void* scalars, size_t ffi_affine_sz);
SNARKVM_API int snarkvm_b200_msm_g2_device(void* out288, const void* d_points, size_t npoints, const void* d_scalars, size_t stride, void* stream);
/* test / bench input: P_i = h(seed, i)·G2 with the multipliers of snarkvm_b200_generate_bases_device */
SNARKVM_API int snarkvm_b200_generate_bases_g2_device(void* d_points, size_t npoints, size_t stride, uint64_t seed, void* stream);

SNARKVM_API int snarkvm_b200_generate_bases_device(void* d_points, size_t npoints, size_t stride, uint64_t seed, void* stream);
/* P_i = s_i * G for npoints canonical scalars (32 B each) in HBM, written in the reference Affine layout: s_i = beta^i gives the
 * powers_of_beta_g of a universal setup with a KNOWN trapdoor (kzg10/data_structures.rs UniversalParams) for tests and benches. */
SNARKVM_API int snarkvm_b200_generator_mul_device(void* d_points, size_t stride, const void* d_scalars, size_t npoints, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SNARKVM_B200_H */
