// Device-resident polynomial helpers around the NTT (SURVEY §8 f2/f3): the pieces of the Varuna prover that sit between
// transforms and would otherwise force a PCIe round trip per polynomial.
//
//   fr_batch_inversion_and_mul_device  — fields/src/lib.rs:78-129 (batch_inversion_and_mul; used by
//                                        snark/varuna/ahp/prover/round_functions/fourth.rs:203-211)
//   poly_divide_by_vanishing_device    — fft/polynomial/dense.rs:162-169 → fft/polynomial/mod.rs:222-256 with the
//                                        divisor x^n − 1
//   poly_evaluate_device               — DensePolynomial::evaluate (fft/polynomial/dense.rs:98-114)
//
// Every result is a canonical Fr value, so any correct evaluation order is bit-identical to the reference's.
#include "poly.cuh"

#include "ff.cuh"
#include "msm.cuh"   // count_launch, ensure_pool_configured

namespace b200 {

struct FrArg { uint32_t v[8]; };
FF_DEV Fr fr_from_arg(const FrArg& a) { Fr r;
#pragma unroll
    for (int i = 0; i < 8; i++) r.v[i] = a.v[i]; return r; }

// ---------------------------------------------------------------------------------------------------------------------
// v_i ← coeff · v_i^{-1}; zeros are skipped and stay zero (lib.rs:107, 121).  Montgomery's trick per thread over K
// elements taken with a grid stride (coalesced), one Fermat inversion per K: ≈ 3 + 380/K multiplications per element.
// ---------------------------------------------------------------------------------------------------------------------
static constexpr int BINV_K = 8;
__global__ void __launch_bounds__(128) k_fr_batch_inverse(uint32_t* __restrict__ v, size_t n, FrArg coeff_arg) {
    const size_t T = (size_t)gridDim.x * blockDim.x, t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    Fr x[BINV_K], pre[BINV_K];
    Fr run = Fr::one();
#pragma unroll
    for (int k = 0; k < BINV_K; k++) {
        size_t i = (size_t)k * T + t;
        x[k] = i < n ? Fr::load(v + i * 8) : Fr::zero();
        pre[k] = run;                                      // product of the non-zero elements before k
        if (!x[k].is_zero()) run = run * x[k];
    }
    Fr inv = run.inverse() * fr_from_arg(coeff_arg);       // run ≠ 0 (one if everything was zero)
#pragma unroll
    for (int k = BINV_K - 1; k >= 0; k--) {
        size_t i = (size_t)k * T + t;
        if (i < n && !x[k].is_zero()) {
            (inv * pre[k]).store(v + i * 8);
            inv = inv * x[k];
        }
    }
}

int fr_batch_inversion_and_mul_device(void* d_v, size_t n, const void* coeff_mont_host, cudaStream_t stream) {
    if (n == 0) return 0;
    if (!d_v || !coeff_mont_host) return (int)cudaErrorInvalidValue;
    FrArg c;
    memcpy(c.v, coeff_mont_host, 32);
    size_t threads = (n + BINV_K - 1) / BINV_K;
    k_fr_batch_inverse<<<(unsigned)((threads + 127) / 128), 128, 0, stream>>>((uint32_t*)d_v, n, c);
    count_launch();
    return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------------------
// p = q·(x^n − 1) + r  ⇒  q_i = Σ_{k ≥ 1} p_{i + k·n},  r_i = p_i + q_i  (q_i = 0 past its end).
// ---------------------------------------------------------------------------------------------------------------------
__global__ void k_divide_by_vanishing(const uint32_t* __restrict__ p, size_t m, size_t n, uint32_t* __restrict__ q,
                                      uint32_t* __restrict__ r) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t qlen = m > n ? m - n : 0, rlen = m < n ? m : n;
    if (i >= qlen && i >= rlen) return;
    Fr acc = Fr::zero();
    for (size_t j = i + n; j < m; j += n) acc = acc + Fr::load_ldg(p + j * 8);
    if (i < qlen) acc.store(q + i * 8);
    if (i < rlen) (acc + Fr::load_ldg(p + i * 8)).store(r + i * 8);
}

// The loop above costs m/n additions per output: fine for the quotient by a large domain (m/n ≤ a few), quadratic for a SMALL
// one — Varuna's first round divides a |C|-coefficient polynomial by the vanishing polynomial of the input domain (n = 4 … 64),
// 2.7·10^11 additions at |C| = 2^20.  View p as rows of n coefficients: q is the exclusive suffix sum DOWN each column.  Blocks of
// RB rows: (1) per-block column sums, (2) a suffix scan over the blocks of each column, (3) every block walks its rows once more
// with its offset — 2m additions, depth RB + #blocks ≈ 2·sqrt(m/n).
__global__ void k_dbv_block_sums(const uint32_t* __restrict__ p, size_t m, size_t n, size_t rb, size_t nblocks, uint32_t* __restrict__ S) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nblocks * n) return;
    const size_t b = t / n, c = t % n;
    Fr acc = Fr::zero();
    for (size_t k = b * rb; k < (b + 1) * rb; k++) { const size_t j = k * n + c; if (j < m) acc = acc + Fr::load_ldg(p + j * 8); }
    acc.store(S + t * 8);
}
__global__ void k_dbv_block_scan(uint32_t* __restrict__ S, size_t n, size_t nblocks) {     // in place: S[b][c] ← Σ_{b' > b} S[b'][c]
    const size_t c = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n) return;
    Fr run = Fr::zero();
    for (size_t b = nblocks; b-- > 0;) {
        const Fr v = Fr::load(S + (b * n + c) * 8);
        run.store(S + (b * n + c) * 8);
        run = run + v;
    }
}
__global__ void k_dbv_finish(const uint32_t* __restrict__ p, size_t m, size_t n, size_t rb, size_t nblocks, const uint32_t* __restrict__ T,
                             uint32_t* __restrict__ q, uint32_t* __restrict__ r) {
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nblocks * n) return;
    const size_t b = t / n, c = t % n, qlen = m > n ? m - n : 0, rlen = m < n ? m : n;
    Fr run = Fr::load(T + t * 8);                                                          // Σ of the rows below this block
    for (size_t k = (b + 1) * rb; k-- > b * rb;) {
        const size_t j = k * n + c;
        if (j >= m) continue;
        const Fr v = Fr::load_ldg(p + j * 8);
        if (j < qlen) run.store(q + j * 8);
        if (j < rlen) (run + v).store(r + j * 8);
        run = run + v;
    }
}

int poly_divide_by_vanishing_device(void* d_q, void* d_r, const void* d_p, size_t m, size_t n, cudaStream_t stream) {
    if (n == 0) return (int)cudaErrorInvalidValue;
    if (m == 0) return 0;
    const size_t qlen = m > n ? m - n : 0, rlen = m < n ? m : n, work = qlen > rlen ? qlen : rlen;
    if (!d_p || !d_r || (qlen && !d_q)) return (int)cudaErrorInvalidValue;
    const size_t rows = (m + n - 1) / n;
    if (rows <= 64) {
        k_divide_by_vanishing<<<(unsigned)((work + 255) / 256), 256, 0, stream>>>((const uint32_t*)d_p, m, n, (uint32_t*)d_q, (uint32_t*)d_r);
        count_launch();
        return (int)cudaGetLastError();
    }
    size_t rb = 1;
    while (rb * rb < rows) rb <<= 1;                                                       // ≈ sqrt(rows), a power of two
    const size_t nblocks = (rows + rb - 1) / rb, cells = nblocks * n;
    uint32_t* S = nullptr;
    cudaError_t e = pool_alloc(&S, cells * 32, stream);
    if (e != cudaSuccess) return (int)e;
    k_dbv_block_sums<<<(unsigned)((cells + 127) / 128), 128, 0, stream>>>((const uint32_t*)d_p, m, n, rb, nblocks, S);
    k_dbv_block_scan<<<(unsigned)((n + 127) / 128), 128, 0, stream>>>(S, n, nblocks);
    k_dbv_finish<<<(unsigned)((cells + 127) / 128), 128, 0, stream>>>((const uint32_t*)d_p, m, n, rb, nblocks, S, (uint32_t*)d_q, (uint32_t*)d_r);
    count_launch(3);
    int rc = (int)cudaGetLastError();
    cudaFreeAsync(S, stream);
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// Σ c_i z^i: a thread runs Horner over EVAL_K consecutive coefficients and shifts its partial by z^{first index}; the
// CTA adds its 256 partials in shared memory; a second single-CTA launch adds the per-CTA sums.
// ---------------------------------------------------------------------------------------------------------------------
static constexpr int EVAL_K = 64, EVAL_THREADS = 256;
FF_DEV Fr fr_pow_u64(Fr base, uint64_t e) {
    Fr acc = Fr::one();
    while (e) { if (e & 1) acc = acc * base; base = base.sqr(); e >>= 1; }
    return acc;
}
FF_DEV Fr cta_sum(Fr mine, uint32_t* sh) {
    mine.store(sh + threadIdx.x * 8);
    __syncthreads();
    for (int s = EVAL_THREADS / 2; s > 0; s >>= 1) {
        if ((int)threadIdx.x < s) (Fr::load(sh + threadIdx.x * 8) + Fr::load(sh + (threadIdx.x + s) * 8)).store(sh + threadIdx.x * 8);
        __syncthreads();
    }
    return Fr::load(sh);
}
__global__ void __launch_bounds__(EVAL_THREADS) k_poly_eval_partial(const uint32_t* __restrict__ c, size_t m, FrArg z_arg,
                                                                     uint32_t* __restrict__ partial) {
    __shared__ uint4 sh4[EVAL_THREADS * 2];
    const Fr z = fr_from_arg(z_arg);
    const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x, i0 = t * EVAL_K;
    Fr acc = Fr::zero();
    if (i0 < m) {
        const size_t i1 = i0 + EVAL_K < m ? i0 + EVAL_K : m;
        for (size_t i = i1; i-- > i0;) acc = acc * z + Fr::load_ldg(c + i * 8);
        acc = acc * fr_pow_u64(z, (uint64_t)i0);
    }
    Fr s = cta_sum(acc, reinterpret_cast<uint32_t*>(sh4));
    if (threadIdx.x == 0) s.store(partial + (size_t)blockIdx.x * 8);
}
__global__ void __launch_bounds__(EVAL_THREADS) k_fr_sum(const uint32_t* __restrict__ in, size_t count, uint32_t* __restrict__ out) {
    __shared__ uint4 sh4[EVAL_THREADS * 2];
    Fr acc = Fr::zero();
    for (size_t i = threadIdx.x; i < count; i += EVAL_THREADS) acc = acc + Fr::load_ldg(in + i * 8);
    Fr s = cta_sum(acc, reinterpret_cast<uint32_t*>(sh4));
    if (threadIdx.x == 0) s.store(out);
}

int poly_evaluate_device(void* out_mont_host, const void* d_coeffs, size_t m, const void* point_mont_host, cudaStream_t stream) {
    if (!out_mont_host || !point_mont_host) return (int)cudaErrorInvalidValue;
    if (m == 0) { memset(out_mont_host, 0, 32); return 0; }
    if (!d_coeffs) return (int)cudaErrorInvalidValue;
    FrArg z;
    memcpy(z.v, point_mont_host, 32);
    const size_t threads = (m + EVAL_K - 1) / EVAL_K, blocks = (threads + EVAL_THREADS - 1) / EVAL_THREADS;
    uint32_t* scratch = nullptr;
    cudaError_t e = pool_alloc(&scratch, (blocks + 1) * 32, stream);
    if (e != cudaSuccess) return (int)e;
    k_poly_eval_partial<<<(unsigned)blocks, EVAL_THREADS, 0, stream>>>((const uint32_t*)d_coeffs, m, z, scratch);
    k_fr_sum<<<1, EVAL_THREADS, 0, stream>>>(scratch, blocks, scratch + blocks * 8);
    count_launch(2);
    int rc = (int)cudaGetLastError();
    if (rc == 0) rc = (int)cudaMemcpyAsync(out_mont_host, scratch + blocks * 8, 32, cudaMemcpyDeviceToHost, stream);
    cudaFreeAsync(scratch, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// Quotient of p / (x − z) — the KZG witness polynomial (polycommit/kzg10/mod.rs:220-241).  q_{L−1} = p_L, q_{i−1} = p_i + z·q_i
// (L = m − 1) is a first-order linear recurrence; it is cut into chunks of LIN_K coefficients:
//   pass 1: each chunk's value at its low end assuming a zero carry-in (A_k),
//   pass 2: one CTA chains the chunks, C_k = A_k + z^{len_k}·C_{k+1}, two levels deep, and leaves every chunk's carry-in,
//   pass 3: each chunk reruns its recurrence from the true carry-in and writes q.
// 2 Fr multiplications per coefficient.
// ---------------------------------------------------------------------------------------------------------------------
static constexpr int LIN_K = 64, LIN_THREADS = 256;
__global__ void k_lin_local(const uint32_t* __restrict__ p, size_t L, FrArg z_arg, uint32_t* __restrict__ A) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x, bot = k * LIN_K;
    if (bot >= L) return;
    const size_t top = bot + LIN_K < L ? bot + LIN_K : L;
    const Fr z = fr_from_arg(z_arg);
    Fr acc = Fr::zero();
    for (size_t i = top; i-- > bot;) acc = acc * z + Fr::load_ldg(p + (i + 1) * 8);
    acc.store(A + k * 8);
}
__global__ void __launch_bounds__(LIN_THREADS) k_lin_carry(const uint32_t* __restrict__ A, size_t nchunks, size_t L, FrArg z_arg,
                                                            uint32_t* __restrict__ cin) {
    __shared__ uint4 shB4[LIN_THREADS * 2], shW4[LIN_THREADS * 2];
    uint32_t* shB = reinterpret_cast<uint32_t*>(shB4);
    uint32_t* shW = reinterpret_cast<uint32_t*>(shW4);
    const Fr z = fr_from_arg(z_arg);
    const Fr zK = fr_pow_u64(z, LIN_K);
    const Fr zlast = fr_pow_u64(z, (uint64_t)(L - (nchunks - 1) * LIN_K));      // the highest chunk may be short
    const size_t per = (nchunks + LIN_THREADS - 1) / LIN_THREADS;
    const size_t k0 = (size_t)threadIdx.x * per, k1 = k0 + per < nchunks ? k0 + per : nchunks;
    Fr B = Fr::zero(), W = Fr::one();
    for (size_t k = k1; k-- > k0 && k0 < nchunks;) {
        const Fr zl = (k == nchunks - 1) ? zlast : zK;
        B = Fr::load_ldg(A + k * 8) + zl * B;
        W = W * zl;
    }
    B.store(shB + threadIdx.x * 8);
    W.store(shW + threadIdx.x * 8);
    __syncthreads();
    if (threadIdx.x == 0) {                                  // D_t = value entering super-chunk t from above
        Fr D = Fr::zero();
        for (int t = LIN_THREADS - 1; t >= 0; t--) {
            Fr Bt = Fr::load(shB + t * 8), Wt = Fr::load(shW + t * 8);
            D.store(shB + t * 8);                            // carry-in of super-chunk t
            D = Bt + Wt * D;
        }
    }
    __syncthreads();
    Fr C = Fr::load(shB + threadIdx.x * 8);
    for (size_t k = k1; k-- > k0 && k0 < nchunks;) {
        C.store(cin + k * 8);
        const Fr zl = (k == nchunks - 1) ? zlast : zK;
        C = Fr::load_ldg(A + k * 8) + zl * C;
    }
}
__global__ void k_lin_final(const uint32_t* __restrict__ p, size_t L, FrArg z_arg, const uint32_t* __restrict__ cin, uint32_t* __restrict__ q) {
    const size_t k = (size_t)blockIdx.x * blockDim.x + threadIdx.x, bot = k * LIN_K;
    if (bot >= L) return;
    const size_t top = bot + LIN_K < L ? bot + LIN_K : L;
    const Fr z = fr_from_arg(z_arg);
    Fr acc = Fr::load_ldg(cin + k * 8);
    for (size_t i = top; i-- > bot;) { acc = acc * z + Fr::load_ldg(p + (i + 1) * 8); acc.store(q + i * 8); }
}

int poly_divide_by_linear_device(void* d_q, const void* d_p, size_t m, const void* point_mont_host, cudaStream_t stream) {
    if (m <= 1) return 0;
    if (!d_q || !d_p || !point_mont_host) return (int)cudaErrorInvalidValue;
    FrArg z;
    memcpy(z.v, point_mont_host, 32);
    const size_t L = m - 1, nchunks = (L + LIN_K - 1) / LIN_K;
    uint32_t* scratch = nullptr;                             // A[nchunks] then cin[nchunks]
    cudaError_t e = pool_alloc(&scratch, nchunks * 64, stream);
    if (e != cudaSuccess) return (int)e;
    const unsigned grid = (unsigned)((nchunks + 127) / 128);
    k_lin_local<<<grid, 128, 0, stream>>>((const uint32_t*)d_p, L, z, scratch);
    k_lin_carry<<<1, LIN_THREADS, 0, stream>>>(scratch, nchunks, L, z, scratch + nchunks * 8);
    k_lin_final<<<grid, 128, 0, stream>>>((const uint32_t*)d_p, L, z, scratch + nchunks * 8, (uint32_t*)d_q);
    count_launch(3);
    int rc = (int)cudaGetLastError();
    cudaFreeAsync(scratch, stream);
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// z_M = M·z for a sparse R1CS matrix in CSR form — inner_product (snark/varuna/ahp/prover/round_functions/mod.rs:169-189),
// the per-row loop the prover runs for A, B and C (:128-152).  One thread per row (rows hold a handful of entries).
// ---------------------------------------------------------------------------------------------------------------------
// Rows longer than SPMV_LONG entries (a hot variable: the constant one, or — transposed — a variable every constraint uses;
// the reference's TestCircuit puts 2^20 entries of B in ONE column) would serialise a thread: 2.6 s for M(α, ·) of a
// 2^20-constraint circuit.  They leave the thread-per-row kernel through a device-side work list — no host round trip —
// and are cut into segments of SPMV_SEG entries, one CTA per segment, then one CTA per long row adds its segments.
static constexpr uint32_t SPMV_LONG = 256, SPMV_SEG = 2048;
struct SpmvLong { uint32_t row, base, nseg; };
__global__ void k_sparse_matvec(const uint32_t* __restrict__ row_ptr, const uint32_t* __restrict__ cols, const uint32_t* __restrict__ vals,
                                size_t nrows, const uint32_t* __restrict__ x, size_t nvars, uint32_t* __restrict__ out, int* __restrict__ bad,
                                uint32_t* __restrict__ ctr /* [0] long rows, [1] work items */, SpmvLong* __restrict__ long_rows,
                                uint2* __restrict__ items) {
    const size_t r = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    const uint32_t e0 = row_ptr[r], e1 = row_ptr[r + 1];
    if (e1 - e0 > SPMV_LONG) {
        const uint32_t nseg = (e1 - e0 + SPMV_SEG - 1) / SPMV_SEG;
        const uint32_t base = atomicAdd(&ctr[1], nseg), slot = atomicAdd(&ctr[0], 1u);
        long_rows[slot] = SpmvLong{(uint32_t)r, base, nseg};
        for (uint32_t j = 0; j < nseg; j++) items[base + j] = make_uint2((uint32_t)r, j);
        return;
    }
    Fr acc = Fr::zero();
    for (uint32_t e = e0; e < e1; e++) {
        const uint32_t c = cols[e];
        if (c >= nvars) { *bad = 1; continue; }              // out-of-range column: reported, never read
        acc = acc + Fr::load_ldg(x + (size_t)c * 8) * Fr::load_ldg(vals + (size_t)e * 8);
    }
    acc.store(out + r * 8);
}
// Σ over the 256 threads of a CTA (shared memory tree); the result is valid in thread 0
FF_DEV Fr cta_sum_fr(Fr v, uint4* sh) {
    const uint32_t t = threadIdx.x;
    sh[2 * t] = make_uint4(v.v[0], v.v[1], v.v[2], v.v[3]); sh[2 * t + 1] = make_uint4(v.v[4], v.v[5], v.v[6], v.v[7]);
    __syncthreads();
    for (uint32_t d = 128; d >= 1; d >>= 1) {
        if (t < d) {
            Fr a = Fr::load(sh + 2 * t), b = Fr::load(sh + 2 * (t + d));
            a = a + b;
            a.store(sh + 2 * t);
        }
        __syncthreads();
    }
    return Fr::load(sh);
}
__global__ void __launch_bounds__(256) k_spmv_segments(const uint32_t* __restrict__ row_ptr, const uint32_t* __restrict__ cols,
                                                       const uint32_t* __restrict__ vals, const uint32_t* __restrict__ x, size_t nvars,
                                                       const uint32_t* __restrict__ ctr, const uint2* __restrict__ items,
                                                       uint32_t* __restrict__ partial, int* __restrict__ bad) {
    __shared__ uint4 sh[512];
    const uint32_t nitems = ctr[1];
    for (uint32_t it = blockIdx.x; it < nitems; it += gridDim.x) {
        const uint2 w = items[it];
        const uint32_t e0 = row_ptr[w.x] + w.y * SPMV_SEG, rend = row_ptr[w.x + 1], e1 = e0 + SPMV_SEG < rend ? e0 + SPMV_SEG : rend;
        Fr acc = Fr::zero();
        for (uint32_t e = e0 + threadIdx.x; e < e1; e += 256) {
            const uint32_t c = cols[e];
            if (c >= nvars) { *bad = 1; continue; }
            acc = acc + Fr::load_ldg(x + (size_t)c * 8) * Fr::load_ldg(vals + (size_t)e * 8);
        }
        const Fr tot = cta_sum_fr(acc, sh);
        if (threadIdx.x == 0) tot.store(partial + (size_t)it * 8);
        __syncthreads();
    }
}
__global__ void __launch_bounds__(256) k_spmv_long_rows(const uint32_t* __restrict__ ctr, const SpmvLong* __restrict__ long_rows,
                                                        const uint32_t* __restrict__ partial, uint32_t* __restrict__ out) {
    __shared__ uint4 sh[512];
    const uint32_t nlong = ctr[0];
    for (uint32_t k = blockIdx.x; k < nlong; k += gridDim.x) {
        const SpmvLong L = long_rows[k];
        Fr acc = Fr::zero();
        for (uint32_t j = threadIdx.x; j < L.nseg; j += 256) acc = acc + Fr::load(partial + (size_t)(L.base + j) * 8);
        const Fr tot = cta_sum_fr(acc, sh);
        if (threadIdx.x == 0) tot.store(out + (size_t)L.row * 8);
        __syncthreads();
    }
}

int sparse_matvec_device(void* d_out, const void* d_row_ptr, const void* d_cols, const void* d_vals, size_t nrows, const void* d_x,
                         size_t nvars, cudaStream_t stream) {
    if (nrows == 0) return 0;
    if (!d_out || !d_row_ptr || !d_x) return (int)cudaErrorInvalidValue;
    // the number of entries sizes the work lists of the long rows
    uint32_t nnz = 0;
    int rc = (int)cudaMemcpyAsync(&nnz, (const uint32_t*)d_row_ptr + nrows, 4, cudaMemcpyDeviceToHost, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc != 0) return rc;
    const size_t max_long = (size_t)nnz / SPMV_LONG + 1, max_items = (size_t)nnz / SPMV_SEG + max_long + 1;
    uint8_t* scratch = nullptr;
    const size_t off_long = 256, off_items = off_long + ((max_long * sizeof(SpmvLong) + 255) & ~(size_t)255),
                 off_partial = off_items + ((max_items * sizeof(uint2) + 255) & ~(size_t)255), total = off_partial + max_items * 32;
    cudaError_t e = pool_alloc(&scratch, total, stream);
    if (e != cudaSuccess) return (int)e;
    int* bad = (int*)scratch;                                     // [0] bad flag, [1..2] counters
    uint32_t* ctr = (uint32_t*)scratch + 1;
    rc = (int)cudaMemsetAsync(scratch, 0, 256, stream);
    k_sparse_matvec<<<(unsigned)((nrows + 127) / 128), 128, 0, stream>>>((const uint32_t*)d_row_ptr, (const uint32_t*)d_cols, (const uint32_t*)d_vals,
                                                                         nrows, (const uint32_t*)d_x, nvars, (uint32_t*)d_out, bad, ctr,
                                                                         (SpmvLong*)(scratch + off_long), (uint2*)(scratch + off_items));
    k_spmv_segments<<<592, 256, 0, stream>>>((const uint32_t*)d_row_ptr, (const uint32_t*)d_cols, (const uint32_t*)d_vals, (const uint32_t*)d_x, nvars,
                                             ctr, (const uint2*)(scratch + off_items), (uint32_t*)(scratch + off_partial), bad);
    k_spmv_long_rows<<<148, 256, 0, stream>>>(ctr, (const SpmvLong*)(scratch + off_long), (const uint32_t*)(scratch + off_partial), (uint32_t*)d_out);
    count_launch(3);
    if (rc == 0) rc = (int)cudaGetLastError();
    int h_bad = 0;
    if (rc == 0) rc = (int)cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, stream);
    cudaFreeAsync(scratch, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc == 0 && h_bad) rc = (int)cudaErrorInvalidValue;
    return rc;
}

// ---------------------------------------------------------------------------------------------------------------------
// Elementwise Fr arithmetic on HBM vectors (the `cfg_iter_mut!(..).zip(..)` loops between transforms, e.g.
// polycommit/kzg10/mod.rs:292-297, fft/evaluations.rs:49-74) and the domain's elements (fft/domain.rs:307-309, 980-988).
// op: 0 = a + b, 1 = a − b, 2 = a · b.  out may alias a or b.
// ---------------------------------------------------------------------------------------------------------------------
FF_DEV Fr fr_apply(int op, const Fr& a, const Fr& b) { return op == 0 ? a + b : op == 1 ? a - b : a * b; }
__global__ void k_fr_vec_op(uint32_t* out, const uint32_t* a, const uint32_t* b, size_t n, int op) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) fr_apply(op, Fr::load(a + i * 8), Fr::load(b + i * 8)).store(out + i * 8);
}
__global__ void k_fr_vec_scalar_op(uint32_t* out, const uint32_t* a, FrArg s_arg, size_t n, int op) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) fr_apply(op, Fr::load(a + i * 8), fr_from_arg(s_arg)).store(out + i * 8);
}
// out[i] = ω_n^i from the NTT's table ω_N^j (j < N/2): ω_n^i = ω_N^{i·N/n}, and ω^{i} = −ω^{i − n/2} in the upper half
__global__ void k_domain_elements(uint32_t* __restrict__ out, int lg, const uint32_t* __restrict__ tw, int lgN) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x, n = (size_t)1 << lg, half = n >> 1;
    if (i >= n) return;
    if (lg == 0) { Fr::one().store(out); return; }
    const size_t j = i < half ? i : i - half;
    Fr w = Fr::load_ldg(tw + (j << (lgN - lg)) * 8);
    (i < half ? w : w.neg()).store(out + i * 8);
}

// ---------------------------------------------------------------------------------------------------------------------
// The indexer's arithmetization of A, B, C (matrix_evals, snark/varuna/ahp/matrices.rs:138-190) in one launch: thread κ of
// matrix m (blockIdx.y) finds its entry's row by a binary search in row_ptr, remaps the column with reindex_by_subdomain
// (fft/domain.rs:322-344) and reads ω_R^row, ω_C^col from the NTT twiddle table, so no per-entry index array and no |R| or
// |C| element table exists.  Slots κ ≥ nnz_m are the padding (1, 1, 1, 0).
//   INDEX_MATERIALISE: the four evaluation vectors row, col, row_col = row·col, row_col_val = val·row_col on K_m.
//   INDEX_EVALUATE:    Σ_κ L_κ(z)·e(κ) for the four vectors (MatrixEvals::evaluate with the Lagrange coefficients of K_m at z,
//                      ahp/indexer/indexer.rs:232-260): CTA partial sums, then one CTA per sum adds the partials.
// A row_ptr that is not a CSR offset array over nnz_m entries, or a column ≥ num_variables, sets *bad; the entry is skipped.
// ---------------------------------------------------------------------------------------------------------------------
struct IndexMatrix {
    const uint32_t* row_ptr;     // nrows + 1
    const uint32_t* cols;        // nnz
    const uint32_t* vals;        // nnz Montgomery Fr
    uint32_t* out[4];            // INDEX_MATERIALISE: row, col, row_col, row_col_val [K]
    const uint32_t* lagrange;    // INDEX_EVALUATE: L_κ(z) [K]
    uint32_t nnz, lg_k;
};
struct IndexArgs {
    IndexMatrix m[3];
    const uint32_t* tw;          // ω_N^j, j < N/2
    uint32_t nrows, num_variables, num_public;
    int lg_r, lg_c, lgN;
};
FF_DEV Fr domain_element(const uint32_t* tw, int lgN, int lg, uint64_t i) {     // ω_n^i, n = 2^lg (as k_domain_elements)
    if (lg == 0) return Fr::one();
    const uint64_t half = (uint64_t)1 << (lg - 1), j = i < half ? i : i - half;
    const Fr w = Fr::load_ldg(tw + (j << (lgN - lg)) * 8);
    return i < half ? w : w.neg();
}
template <int MODE>
__global__ void __launch_bounds__(EVAL_THREADS) k_index_arith(IndexArgs a, uint32_t* __restrict__ partial, uint32_t max_blocks,
                                                               int* __restrict__ bad) {
    const IndexMatrix& M = a.m[blockIdx.y];
    const uint64_t k = (uint64_t)blockIdx.x * EVAL_THREADS + threadIdx.x, K = (uint64_t)1 << M.lg_k;
    Fr e[4] = {Fr::one(), Fr::one(), Fr::one(), Fr::zero()};
    if (k < M.nnz) {
        uint32_t lo = 0, hi = a.nrows;                                  // largest r < nrows with row_ptr[r] ≤ κ
        while (hi - lo > 1) {
            const uint32_t mid = lo + (hi - lo) / 2;
            if (M.row_ptr[mid] <= k) lo = mid; else hi = mid;
        }
        const uint32_t c = M.cols[k];
        if (M.row_ptr[lo] > k || M.row_ptr[lo + 1] <= k || c >= a.num_variables) {
            *bad = 1;
        } else {
            const uint64_t period = ((uint64_t)1 << a.lg_c) / a.num_public;
            uint64_t ci;
            if (c < a.num_public) {
                ci = (uint64_t)c * period;
            } else {
                const uint64_t i = c - a.num_public;
                ci = i + i / (period - 1) + 1;
            }
            e[0] = domain_element(a.tw, a.lgN, a.lg_r, lo);
            e[1] = domain_element(a.tw, a.lgN, a.lg_c, ci);
            e[2] = e[0] * e[1];
            e[3] = Fr::load_ldg(M.vals + k * 8) * e[2];
        }
    }
    if (k == 0 && M.row_ptr[a.nrows] != M.nnz) *bad = 1;
    if constexpr (MODE == INDEX_MATERIALISE) {
        if (k < K) {
#pragma unroll
            for (int j = 0; j < 4; j++) e[j].store(M.out[j] + k * 8);
        }
    } else {
        __shared__ uint4 sh4[EVAL_THREADS * 2];
        const Fr l = k < K ? Fr::load_ldg(M.lagrange + k * 8) : Fr::zero();
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const Fr s = cta_sum(e[j] * l, reinterpret_cast<uint32_t*>(sh4));
            if (threadIdx.x == 0) s.store(partial + (((size_t)blockIdx.y * max_blocks + blockIdx.x) * 4 + j) * 8);
            __syncthreads();
        }
    }
}
// CTA (m, j) adds the partial sums of vector j of matrix m
__global__ void __launch_bounds__(EVAL_THREADS) k_index_sums(const uint32_t* __restrict__ partial, uint32_t max_blocks, uint3 nblocks,
                                                             uint32_t* __restrict__ out) {
    __shared__ uint4 sh4[EVAL_THREADS * 2];
    const uint32_t m = blockIdx.x / 4, j = blockIdx.x % 4, nb = m == 0 ? nblocks.x : m == 1 ? nblocks.y : nblocks.z;
    Fr acc = Fr::zero();
    for (uint32_t b = threadIdx.x; b < nb; b += EVAL_THREADS) acc = acc + Fr::load_ldg(partial + (((size_t)m * max_blocks + b) * 4 + j) * 8);
    const Fr s = cta_sum(acc, reinterpret_cast<uint32_t*>(sh4));
    if (threadIdx.x == 0) s.store(out + blockIdx.x * 8);
}

int index_arithmetize_device(int mode, const void* const* d_row_ptr, const void* const* d_cols, const void* const* d_vals, const size_t* nnz,
                             const uint32_t* lg_k, size_t num_constraints, size_t num_variables, size_t num_public, void* const* d_io,
                             void* sums_mont_host, cudaStream_t stream) {
    if ((mode != INDEX_MATERIALISE && mode != INDEX_EVALUATE) || !d_row_ptr || !d_cols || !d_vals || !nnz || !lg_k || !d_io)
        return (int)cudaErrorInvalidValue;
    if (mode == INDEX_EVALUATE && !sums_mont_host) return (int)cudaErrorInvalidValue;
    // the three domains: R ⊇ rows, C ⊇ variables, X = the padded public variables, a proper subgroup of C (domain.rs:323)
    int lg_r = 0, lg_c = 0;
    while (((size_t)1 << lg_r) < num_constraints) lg_r++;
    while (((size_t)1 << lg_c) < num_variables) lg_c++;
    if (num_constraints == 0 || num_constraints > ((size_t)1 << 31) || num_variables > ((size_t)1 << 31) || lg_r > 30 || lg_c > 30)
        return (int)cudaErrorInvalidValue;
    if (num_public == 0 || (num_public & (num_public - 1)) || num_public >= ((size_t)1 << lg_c)) return (int)cudaErrorInvalidValue;
    IndexArgs a{};
    uint32_t max_blocks = 1;
    for (int m = 0; m < 3; m++) {
        if (lg_k[m] > 30 || nnz[m] > ((size_t)1 << lg_k[m]) || !d_row_ptr[m] || (nnz[m] && (!d_cols[m] || !d_vals[m]))) return (int)cudaErrorInvalidValue;
        IndexMatrix& M = a.m[m];
        M.row_ptr = (const uint32_t*)d_row_ptr[m]; M.cols = (const uint32_t*)d_cols[m]; M.vals = (const uint32_t*)d_vals[m];
        M.nnz = (uint32_t)nnz[m]; M.lg_k = lg_k[m];
        if (mode == INDEX_MATERIALISE) {
            for (int j = 0; j < 4; j++) {
                if (!d_io[m * 4 + j]) return (int)cudaErrorInvalidValue;
                M.out[j] = (uint32_t*)d_io[m * 4 + j];
            }
        } else {
            if (!d_io[m]) return (int)cudaErrorInvalidValue;
            M.lagrange = (const uint32_t*)d_io[m];
        }
        const uint32_t blocks = (uint32_t)((((size_t)1 << lg_k[m]) + EVAL_THREADS - 1) / EVAL_THREADS);
        if (blocks > max_blocks) max_blocks = blocks;
    }
    const void* tw = nullptr;
    int lgN = 0, rc = 0;
    if ((rc = ntt_get_twiddles(lg_r > lg_c ? lg_r : lg_c > 0 ? lg_c : 1, &tw, &lgN)) != 0) return rc;
    a.tw = (const uint32_t*)tw; a.lgN = lgN; a.lg_r = lg_r; a.lg_c = lg_c;
    a.nrows = (uint32_t)num_constraints; a.num_variables = (uint32_t)num_variables; a.num_public = (uint32_t)num_public;
    // scratch: [0] bad flag, then (EVALUATE) 3 × max_blocks × 4 partial sums and the 12 results
    const size_t off_partial = 256, off_sums = off_partial + (size_t)3 * max_blocks * 4 * 32;
    uint8_t* scratch = nullptr;
    cudaError_t e = pool_alloc(&scratch, mode == INDEX_EVALUATE ? off_sums + 12 * 32 : off_partial, stream);
    if (e != cudaSuccess) return (int)e;
    int* bad = (int*)scratch;
    uint32_t* partial = (uint32_t*)(scratch + off_partial);
    rc = (int)cudaMemsetAsync(scratch, 0, 256, stream);
    const dim3 grid(max_blocks, 3);
    if (rc != 0) {
        // the flag could not be cleared: launch nothing
    } else if (mode == INDEX_MATERIALISE) {
        k_index_arith<INDEX_MATERIALISE><<<grid, EVAL_THREADS, 0, stream>>>(a, partial, max_blocks, bad);
        count_launch();
    } else {
        uint3 nb;
        nb.x = (uint32_t)((((size_t)1 << lg_k[0]) + EVAL_THREADS - 1) / EVAL_THREADS);
        nb.y = (uint32_t)((((size_t)1 << lg_k[1]) + EVAL_THREADS - 1) / EVAL_THREADS);
        nb.z = (uint32_t)((((size_t)1 << lg_k[2]) + EVAL_THREADS - 1) / EVAL_THREADS);
        k_index_arith<INDEX_EVALUATE><<<grid, EVAL_THREADS, 0, stream>>>(a, partial, max_blocks, bad);
        k_index_sums<<<12, EVAL_THREADS, 0, stream>>>(partial, max_blocks, nb, (uint32_t*)(scratch + off_sums));
        count_launch(2);
    }
    if (rc == 0) rc = (int)cudaGetLastError();
    int h_bad = 0;
    if (rc == 0) rc = (int)cudaMemcpyAsync(&h_bad, bad, sizeof(int), cudaMemcpyDeviceToHost, stream);
    if (rc == 0 && mode == INDEX_EVALUATE) rc = (int)cudaMemcpyAsync(sums_mont_host, scratch + off_sums, 12 * 32, cudaMemcpyDeviceToHost, stream);
    cudaFreeAsync(scratch, stream);
    if (rc == 0) rc = (int)cudaStreamSynchronize(stream);
    if (rc == 0 && h_bad) rc = (int)cudaErrorInvalidValue;
    return rc;
}

int fr_vec_op_device(void* d_out, const void* d_a, const void* d_b, size_t n, int op, cudaStream_t stream) {
    if (n == 0) return 0;
    if (!d_out || !d_a || !d_b || op < 0 || op > 2) return (int)cudaErrorInvalidValue;
    k_fr_vec_op<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>((uint32_t*)d_out, (const uint32_t*)d_a, (const uint32_t*)d_b, n, op);
    count_launch();
    return (int)cudaGetLastError();
}
int fr_vec_scalar_op_device(void* d_out, const void* d_a, const void* scalar_mont_host, size_t n, int op, cudaStream_t stream) {
    if (n == 0) return 0;
    if (!d_out || !d_a || !scalar_mont_host || op < 0 || op > 2) return (int)cudaErrorInvalidValue;
    FrArg sc;
    memcpy(sc.v, scalar_mont_host, 32);
    k_fr_vec_scalar_op<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>((uint32_t*)d_out, (const uint32_t*)d_a, sc, n, op);
    count_launch();
    return (int)cudaGetLastError();
}
int domain_elements_device(void* d_out, uint32_t lg, cudaStream_t stream) {
    if (!d_out || lg > 30) return (int)cudaErrorInvalidValue;
    const void* tw = nullptr;
    int lgN = 0, rc = 0;
    if (lg > 0 && (rc = ntt_get_twiddles((int)lg, &tw, &lgN)) != 0) return rc;
    const size_t n = (size_t)1 << lg;
    k_domain_elements<<<(unsigned)((n + 255) / 256), 256, 0, stream>>>((uint32_t*)d_out, (int)lg, (const uint32_t*)tw, lgN);
    count_launch();
    return (int)cudaGetLastError();
}

}  // namespace b200
