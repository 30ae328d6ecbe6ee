// Device-resident polynomial / field-vector helpers (see poly.cu for the reference map).
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace b200 {

// v_i ← coeff · v_i^{-1} in place on n Montgomery Fr elements in HBM; zeros stay zero.  coeff: 32 B Montgomery, HOST memory.
int fr_batch_inversion_and_mul_device(void* d_v, size_t n, const void* coeff_mont_host, cudaStream_t stream);

// p (m coefficients) = q·(x^n − 1) + r:  d_q gets max(m − n, 0) coefficients, d_r gets min(m, n).
int poly_divide_by_vanishing_device(void* d_q, void* d_r, const void* d_p, size_t m, size_t n, cudaStream_t stream);

// quotient of p (m coefficients) / (x − point): d_q gets m − 1 coefficients (the KZG witness polynomial, kzg10/mod.rs:220-241)
int poly_divide_by_linear_device(void* d_q, const void* d_p, size_t m, const void* point_mont_host, cudaStream_t stream);

// out = Σ c_i·point^i (Montgomery in and out; out and point are 32-byte HOST buffers; synchronises the stream)
int poly_evaluate_device(void* out_mont_host, const void* d_coeffs, size_t m, const void* point_mont_host, cudaStream_t stream);

// out[r] = Σ_e vals[e]·x[cols[e]] over e ∈ [row_ptr[r], row_ptr[r+1]) — CSR sparse matrix × vector over Fr (Montgomery);
// row_ptr: nrows + 1 u32, cols: u32.  A column ≥ nvars returns cudaErrorInvalidValue.  Synchronises the stream.
int sparse_matvec_device(void* d_out, const void* d_row_ptr, const void* d_cols, const void* d_vals, size_t nrows, const void* d_x,
                         size_t nvars, cudaStream_t stream);

// elementwise on n Montgomery Fr in HBM: op 0 = a + b, 1 = a − b, 2 = a·b; the scalar form takes a 32-byte HOST scalar
int fr_vec_op_device(void* d_out, const void* d_a, const void* d_b, size_t n, int op, cudaStream_t stream);
int fr_vec_scalar_op_device(void* d_out, const void* d_a, const void* scalar_mont_host, size_t n, int op, cudaStream_t stream);
// out[i] = ω_n^i, i < n = 2^lg (EvaluationDomain::elements, fft/domain.rs:307-309)
int domain_elements_device(void* d_out, uint32_t lg, cudaStream_t stream);

// The indexer's arithmetization of A, B, C (ahp/matrices.rs:138-190) in one launch.  Per matrix m: CSR row_ptr (num_constraints + 1
// u32), cols (nnz[m] u32 variable indices, public first), vals (nnz[m] Montgomery Fr), K_m = 2^lg_k[m] ≥ nnz[m].  The constraint
// and variable domains are the next powers of two of num_constraints and num_variables; num_public (a power of two, smaller than
// the variable domain) is the input domain columns are reindexed by.
//   INDEX_MATERIALISE: d_io[4m + j] receives vector j ∈ (row, col, row_col, row_col_val) of matrix m, K_m Montgomery Fr.
//   INDEX_EVALUATE:    d_io[m] holds the Lagrange coefficients of K_m at a point (K_m Montgomery Fr); sums_mont_host (HOST,
//                      12 × 32 B) receives Σ_κ L_κ·e_j(κ) in the order 4m + j.
// A malformed row_ptr or a column ≥ num_variables returns cudaErrorInvalidValue.  Synchronises the stream.
enum { INDEX_MATERIALISE = 0, INDEX_EVALUATE = 1 };
int index_arithmetize_device(int mode, const void* const* d_row_ptr, const void* const* d_cols, const void* const* d_vals, const size_t* nnz,
                             const uint32_t* lg_k, size_t num_constraints, size_t num_variables, size_t num_public, void* const* d_io,
                             void* sums_mont_host, cudaStream_t stream);

// Group FFT over G1 (DomainCoeff = G1Projective, fft/domain.rs:169-221 generic path): n = 2^lg affine points in, affine points
// out (natural order both sides).  direction 1 = inverse (includes n^{-1}): UniversalParams::lagrange_basis
// (polycommit/kzg10/data_structures.rs:68-72).
int g1_ntt_device(void* d_out, size_t out_stride, const void* d_in, size_t in_stride, uint32_t lg, int direction, cudaStream_t stream);

// ntt.cu: the cached table ω_N^j (j < N/2, Montgomery), N = 2^lgN ≥ 2^lg
int ntt_get_twiddles(int lg, const void** tw, int* lgN);

}  // namespace b200
