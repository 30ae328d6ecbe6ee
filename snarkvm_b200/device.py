"""Device-resident entry points (PART 2 of include/snarkvm_b200.h) on torch CUDA tensors.

PyTorch is plumbing only: it owns the HBM allocations and the stream; every kernel that runs
is one of this repository's hand-written sm_100a kernels inside libsnarkvm_b200.so.
Tensor conventions: any dtype, contiguous, interpreted as raw bytes in the reference layouts
(Fr: 32 B/elt; scalar: 32 B; affine: `stride` B/point, stride ≥ 104 and a multiple of 8).
"""
from __future__ import annotations

import ctypes

import numpy as np
import torch

from . import _lib
from .cuda import NTTDirection, NTTInputOutputOrder, NTTType

XYZZ_BYTES = 192
AFFINE_STRIDE = 104


def _check(t: torch.Tensor, name: str) -> int:
    if not (isinstance(t, torch.Tensor) and t.is_cuda and t.is_contiguous()):
        raise TypeError(f"{name} must be a contiguous CUDA tensor")
    return t.data_ptr()


def _nbytes(t: torch.Tensor) -> int:
    return t.numel() * t.element_size()


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def ntt_(x: torch.Tensor, direction: NTTDirection = NTTDirection.Forward, ntt_type: NTTType = NTTType.Standard,
         scratch: torch.Tensor | None = None) -> torch.Tensor:
    """In-place natural-order NTT of the 2^lg Fr elements in `x` (32 B each)."""
    n = _nbytes(x) // 32
    if n <= 0 or n & (n - 1) or n * 32 != _nbytes(x):
        raise ValueError("domain_size is not power of 2")
    lg = n.bit_length() - 1
    sp = 0
    if scratch is not None:
        if _nbytes(scratch) < _nbytes(x):
            raise ValueError("scratch too small")
        sp = _check(scratch, "scratch")
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().snarkvm_b200_ntt_device(_check(x, "x"), lg, int(NTTInputOutputOrder.NN), int(direction),
                                                       int(ntt_type), sp, _stream()))
    return x


def polymul(polys: list, evals: list, lg: int) -> torch.Tensor:
    dev = (polys + evals)[0].device
    n = 1 << lg
    out = torch.zeros((n, 4), dtype=torch.int64, device=dev)
    pp = (ctypes.c_void_p * max(1, len(polys)))(*[_check(p, "poly") for p in polys])
    pl = (ctypes.c_size_t * max(1, len(polys)))(*[_nbytes(p) // 32 for p in polys])
    ep = (ctypes.c_void_p * max(1, len(evals)))(*[_check(e, "eval") for e in evals])
    el = (ctypes.c_size_t * max(1, len(evals)))(*[_nbytes(e) // 32 for e in evals])
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().snarkvm_b200_polymul_device(out.data_ptr(), len(polys), ctypes.cast(pp, ctypes.c_void_p),
                                                           ctypes.cast(pl, ctypes.c_void_p), len(evals),
                                                           ctypes.cast(ep, ctypes.c_void_p), ctypes.cast(el, ctypes.c_void_p),
                                                           lg, _stream()))
    return out


def msm_plan(npoints: int) -> dict:
    c, nwin, cap = ctypes.c_int(), ctypes.c_int(), ctypes.c_uint32()
    _lib.check(_lib.lib().snarkvm_b200_msm_plan(npoints, ctypes.byref(c), ctypes.byref(nwin), ctypes.byref(cap)))
    return {"c": c.value, "nwin": nwin.value, "cap": cap.value, "levels": int(_lib.lib().snarkvm_b200_msm_plan_levels(npoints))}


def _msm_args(bases: torch.Tensor, scalars: torch.Tensor, stride: int):
    npoints = _nbytes(scalars) // 32
    if npoints * 32 != _nbytes(scalars):
        raise ValueError("scalars must be a whole number of 32-byte integers")
    if npoints * stride > _nbytes(bases):
        raise ValueError(f"length mismatch {_nbytes(bases) // stride} points < {npoints} scalars")
    return npoints


def msm(bases: torch.Tensor, scalars: torch.Tensor, stride: int = AFFINE_STRIDE) -> np.ndarray:
    """VariableBase::msm with bases and scalars resident in HBM → normalised projective uint64[18]."""
    npoints = _msm_args(bases, scalars, stride)
    out = np.zeros(18, dtype=np.uint64)
    with torch.cuda.device(bases.device):
        _lib.check(_lib.lib().snarkvm_b200_msm_device(out.ctypes.data, _check(bases, "bases"), npoints,
                                                       _check(scalars, "scalars"), stride, _stream()))
    return out


G2_AFFINE_STRIDE = 200       # Affine<G2>: x.c0 x.c1 y.c0 y.c1 (4 × 48 B) infinity pad


def msm_g2(bases: torch.Tensor, scalars: torch.Tensor, stride: int = G2_AFFINE_STRIDE) -> np.ndarray:
    """VariableBase::msm over G2 (standard::msm semantics) with bases and scalars resident in HBM → normalised Projective<G2>
    image uint64[36] (X, Y, Z over Fq2)."""
    npoints = _msm_args(bases, scalars, stride)
    out = np.zeros(36, dtype=np.uint64)
    with torch.cuda.device(bases.device):
        _lib.check(_lib.lib().snarkvm_b200_msm_g2_device(out.ctypes.data, _check(bases, "bases"), npoints,
                                                          _check(scalars, "scalars"), stride, _stream()))
    return out


def generate_bases_g2(npoints: int, seed: int, device="cuda", stride: int = G2_AFFINE_STRIDE) -> torch.Tensor:
    """Synthetic G2 bases P_i = h(seed, i)·G2 in the reference Affine<G2> layout, generated in HBM."""
    t = torch.empty((npoints, stride), dtype=torch.uint8, device=device)
    with torch.cuda.device(t.device):
        _lib.check(_lib.lib().snarkvm_b200_generate_bases_g2_device(t.data_ptr(), npoints, stride, seed & (2**64 - 1), _stream()))
    return t


def msm_window_sums(bases: torch.Tensor, scalars: torch.Tensor, stride: int = AFFINE_STRIDE, plan_npoints: int | None = None,
                    flags: torch.Tensor | None = None, out: torch.Tensor | None = None) -> torch.Tensor:
    """Per-window XYZZ sums [nwin, 24] (int64 view of 192-byte points), left in HBM.  `plan_npoints` (≥ the number of
    scalars) fixes the window plan — all ranks of a sharded MSM pass the largest shard size; an empty shard gives infinity
    sums.  `flags`: optional int32 CUDA tensor [1] that receives bit 0 = "a scalar ≥ 2^253 was seen"."""
    npoints = _msm_args(bases, scalars, stride)
    pn = npoints if plan_npoints is None else int(plan_npoints)
    if pn < max(npoints, 1):
        raise ValueError("plan_npoints must be at least the shard size and positive")
    plan = msm_plan(pn)
    dev = bases.device if bases.is_cuda else scalars.device
    sums = torch.empty((plan["nwin"], XYZZ_BYTES // 8), dtype=torch.int64, device=dev) if out is None else out
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().snarkvm_b200_msm_window_sums_plan_device(
            _check(sums, "out"), flags.data_ptr() if flags is not None else None, pn, _check(bases, "bases") if npoints else None, npoints,
            _check(scalars, "scalars") if npoints else None, stride, _stream()))
    return sums


def msm_window_sums_host(out: torch.Tensor, flags: torch.Tensor | None, plan_npoints: int, points: np.ndarray, scalars: np.ndarray,
                         stride: int = AFFINE_STRIDE) -> torch.Tensor:
    """msm_window_sums from HOST buffers (numpy uint8 [n, stride] points, uint64 [n, 4] canonical scalars): the library uploads
    them (ranges overlapped with the kernels, pageable memory staged through pinned buffers) and leaves the sums in `out`
    (CUDA, [nwin, 24] int64) without synchronising."""
    npoints = scalars.shape[0]
    if npoints > points.shape[0]:
        raise ValueError(f"length mismatch {points.shape[0]} points < {npoints} scalars")
    with torch.cuda.device(out.device):
        _lib.check(_lib.lib().snarkvm_b200_msm_window_sums_host(
            _check(out, "out"), flags.data_ptr() if flags is not None else None, int(plan_npoints), points.ctypes.data if npoints else None,
            npoints, scalars.ctypes.data if npoints else None, stride, _stream()))
    return out


def msm_batch(bases: torch.Tensor, scalar_vectors: list, stride: int = AFFINE_STRIDE) -> np.ndarray:
    """`len(scalar_vectors)` MSMs over the same resident bases in ONE pass → [count, 18] u64 (normalised projective each)."""
    count = len(scalar_vectors)
    out = np.zeros((count, 18), dtype=np.uint64)
    if count == 0:
        return out
    lens = [_msm_args(bases, v, stride) for v in scalar_vectors]
    ptrs = (ctypes.c_void_p * count)(*[(_check(v, "scalars") if n else None) for v, n in zip(scalar_vectors, lens)])
    szs = (ctypes.c_size_t * count)(*lens)
    with torch.cuda.device(bases.device):
        _lib.check(_lib.lib().snarkvm_b200_msm_batch_device(out.ctypes.data, _check(bases, "bases"), stride, ptrs, szs, count, _stream()))
    return out


def msm_set_scratch_limit(nbytes: int) -> None:
    """bytes of MSM scratch concurrent calls on the current device may hold together (callers beyond it wait)"""
    _lib.check(_lib.lib().snarkvm_b200_msm_set_scratch_limit(int(nbytes)))


def msm_scratch_stats() -> dict:
    """MSM scratch budget of the current device: {'limit', 'in_use', 'peak'} in bytes."""
    a, b, c = ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_size_t()
    _lib.check(_lib.lib().snarkvm_b200_msm_scratch_stats(ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)))
    return {"limit": a.value, "in_use": b.value, "peak": c.value}


def xyzz_sum_ranks(gathered: torch.Tensor, nranks: int, count: int) -> torch.Tensor:
    out = torch.empty((count, XYZZ_BYTES // 8), dtype=torch.int64, device=gathered.device)
    with torch.cuda.device(gathered.device):
        _lib.check(_lib.lib().snarkvm_b200_xyzz_sum_ranks_device(out.data_ptr(), _check(gathered, "gathered"), nranks, count,
                                                                  _stream()))
    return out


def msm_finish(window_sums_host: np.ndarray, c: int) -> np.ndarray:
    """Host fold Σ_w 2^{c·w}·S_w of XYZZ window sums (c = 0: plain sum) → normalised projective."""
    ws = np.ascontiguousarray(window_sums_host).view(np.uint8).reshape(-1, XYZZ_BYTES)
    out = np.zeros(18, dtype=np.uint64)
    _lib.check(_lib.lib().snarkvm_b200_msm_finish(out.ctypes.data, ws.ctypes.data, ws.shape[0], c))
    return out


def kzg_commit(powers: torch.Tensor, coeffs_mont: torch.Tensor, stride: int = AFFINE_STRIDE) -> np.ndarray:
    """KZG10::commit core: Σ to_bigint(coeff_i)·powers_i (kzg10/mod.rs:98-156), all operands in HBM."""
    n = _msm_args(powers, coeffs_mont, stride)
    out = np.zeros(18, dtype=np.uint64)
    with torch.cuda.device(powers.device):
        _lib.check(_lib.lib().snarkvm_b200_kzg_commit_device(out.ctypes.data, _check(powers, "powers"), stride,
                                                              _check(coeffs_mont, "coeffs"), n, _stream()))
    return out


def kzg_commit_hiding(powers: torch.Tensor, coeffs_mont: torch.Tensor, gamma_powers: torch.Tensor, blinding_mont: torch.Tensor,
                      stride: int = AFFINE_STRIDE) -> np.ndarray:
    """KZG10::commit with hiding_bound = Some(_) (kzg10/mod.rs:98-156): Σ to_bigint(c_i)·powers_i + Σ to_bigint(b_j)·gamma_powers_j;
    the caller samples the blinding polynomial b (KZGRandomness::rand)."""
    n = _msm_args(powers, coeffs_mont, stride)
    nb = _nbytes(blinding_mont) // 32
    if nb > _nbytes(gamma_powers) // stride:
        raise ValueError("hiding bound exceeds powers_of_beta_times_gamma_g")      # check_hiding_bound, mod.rs:134-137
    out = np.zeros(18, dtype=np.uint64)
    with torch.cuda.device(powers.device):
        _lib.check(_lib.lib().snarkvm_b200_kzg_commit_hiding_device(
            out.ctypes.data, _check(powers, "powers"), stride, _check(coeffs_mont, "coeffs"), n,
            _check(gamma_powers, "gamma_powers"), _check(blinding_mont, "blinding"), nb, _stream()))
    return out


def kzg_commit_batch(powers: torch.Tensor, polys_mont: list, stride: int = AFFINE_STRIDE, gamma_powers: torch.Tensor | None = None,
                     blindings_mont: list | None = None) -> np.ndarray:
    """All commitments of a round against the same resident powers in ONE pass (sonic_pc/mod.rs:177-257) → [count, 18] u64.
    With `gamma_powers` and `blindings_mont` (one Montgomery coefficient tensor or None per polynomial) the hiding terms
    Σ_j blinding_i[j]·gamma_powers[j] (kzg10/mod.rs:129-150) ride in the same pass."""
    count = len(polys_mont)
    out = np.zeros((count, 18), dtype=np.uint64)
    if count == 0:
        return out
    nb = _nbytes(powers) // stride
    lens = [_nbytes(p) // 32 for p in polys_mont]
    if max(lens) > nb:
        raise ValueError("polynomial degree exceeds the number of powers")         # check_degree_is_too_large, mod.rs:105
    ptrs = (ctypes.c_void_p * count)(*[(_check(p, "poly") if n else None) for p, n in zip(polys_mont, lens)])
    szs = (ctypes.c_size_t * count)(*lens)
    with torch.cuda.device(powers.device):
        if blindings_mont is None:
            _lib.check(_lib.lib().snarkvm_b200_kzg_commit_batch_device(out.ctypes.data, _check(powers, "powers"), stride, ptrs, szs, count, _stream()))
        else:
            if len(blindings_mont) != count:
                raise ValueError("one blinding polynomial (or None) per polynomial")
            blens = [0 if b is None else _nbytes(b) // 32 for b in blindings_mont]
            if max(blens) > _nbytes(gamma_powers) // stride:
                raise ValueError("hiding bound exceeds powers_of_beta_times_gamma_g")          # check_hiding_bound, mod.rs:134-137
            bptrs = (ctypes.c_void_p * count)(*[(_check(b, "blinding") if n else None) for b, n in zip(blindings_mont, blens)])
            bszs = (ctypes.c_size_t * count)(*blens)
            _lib.check(_lib.lib().snarkvm_b200_kzg_commit_batch_hiding_device(
                out.ctypes.data, _check(powers, "powers"), stride, ptrs, szs, _check(gamma_powers, "gamma_powers"), bptrs, bszs, count, _stream()))
    return out


def generator_mul(scalars: torch.Tensor, stride: int = AFFINE_STRIDE) -> torch.Tensor:
    """P_i = s_i·G for canonical scalars [n, 4] in HBM → affine points [n, stride] (set-up helper, not a hot path)"""
    n = _nbytes(scalars) // 32
    out = torch.empty((n, stride), dtype=torch.uint8, device=scalars.device)
    with torch.cuda.device(scalars.device):
        _lib.check(_lib.lib().snarkvm_b200_generator_mul_device(out.data_ptr(), stride, _check(scalars, "scalars") if n else None, n, _stream()))
    return out


def generate_powers(n: int, beta: int, scale: int = 1, device="cuda", stride: int = AFFINE_STRIDE) -> torch.Tensor:
    """scale·β^i·G for i < n: powers_of_beta_g (scale = 1) or powers_of_beta_times_gamma_g (scale = γ) of a universal setup whose
    trapdoor the caller knows.  The scalars are built by doubling (v[m:2m] = β^m·v[0:m]), then one fixed-base pass."""
    from .algorithms import _fr_int_to_mont, _R_MOD
    s = torch.zeros((n, 4), dtype=torch.int64, device=device)
    if n == 0:
        return torch.empty((0, stride), dtype=torch.uint8, device=device)
    s[0] = torch.from_numpy(_fr_int_to_mont(scale % _R_MOD).view(np.int64)).to(s.device)
    m = 1
    while m < n:
        k = min(m, n - m)
        fr_vec_op(s[:k], _fr_int_to_mont(pow(beta, m, _R_MOD)), FR_MUL, out=s[m:m + k])
        m *= 2
    return generator_mul(fr_from_mont(s), stride)


def sonic_commit_batch(bases: list, polys_mont: list, gamma_bases: list | None = None, blindings_mont: list | None = None,
                       stride: int = AFFINE_STRIDE) -> np.ndarray:
    """SonicKZG10::commit of a round in ONE pass (sonic_pc/mod.rs:177-257) → [count, 18] u64.  `bases[i]` is the CUDA tensor (or a
    row slice of one: shifted powers are suffixes of the SRS) polynomial i is committed against; `gamma_bases[i]` / `blindings_mont[i]`
    (or None) its hiding terms (kzg10/mod.rs:129-150)."""
    count = len(polys_mont)
    out = np.zeros((count, 18), dtype=np.uint64)
    if count == 0:
        return out
    if len(bases) != count:
        raise ValueError("one base array per polynomial")
    lens = [_nbytes(p) // 32 for p in polys_mont]
    for b, n in zip(bases, lens):
        if n > _nbytes(b) // stride:
            raise ValueError("polynomial degree exceeds the number of powers")             # check_degree_is_too_large, kzg10/mod.rs:105
    bptr = (ctypes.c_void_p * count)(*[(_check(b, "bases") if n else None) for b, n in zip(bases, lens)])
    cptr = (ctypes.c_void_p * count)(*[(_check(p, "poly") if n else None) for p, n in zip(polys_mont, lens)])
    szs = (ctypes.c_size_t * count)(*lens)
    gptr = rptr = rszs = None
    if blindings_mont is not None:
        if gamma_bases is None or len(blindings_mont) != count or len(gamma_bases) != count:
            raise ValueError("one (gamma powers, blinding polynomial) pair (or None) per polynomial")
        blens = [0 if r is None else _nbytes(r) // 32 for r in blindings_mont]
        for g, n in zip(gamma_bases, blens):
            if n and (g is None or n > _nbytes(g) // stride):
                raise ValueError("hiding bound exceeds powers_of_beta_times_gamma_g")      # check_hiding_bound, kzg10/mod.rs:134-137
        gptr = (ctypes.c_void_p * count)(*[(_check(g, "gamma") if n else None) for g, n in zip(gamma_bases, blens)])
        rptr = (ctypes.c_void_p * count)(*[(_check(r, "blinding") if n else None) for r, n in zip(blindings_mont, blens)])
        rszs = (ctypes.c_size_t * count)(*blens)
    dev = next(b.device for b in bases if b is not None)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().snarkvm_b200_sonic_commit_batch_device(out.ctypes.data, stride, bptr, cptr, szs, gptr, rptr, rszs, count, _stream()))
    return out


def g1_ntt(points: torch.Tensor, inverse: bool, stride: int = AFFINE_STRIDE) -> torch.Tensor:
    """FFT / iFFT over 2^k G1 points (EvaluationDomain with T = G1Projective, fft/domain.rs:169-221) → affine points, same stride."""
    n = _nbytes(points) // stride
    if n == 0 or n & (n - 1):
        raise ValueError("domain size must be a power of two")
    out = torch.empty_like(points)
    with torch.cuda.device(points.device):
        _lib.check(_lib.lib().snarkvm_b200_g1_ntt_device(out.data_ptr(), stride, _check(points, "points"), stride, n.bit_length() - 1,
                                                          1 if inverse else 0, _stream()))
    return out


def lagrange_basis(powers_of_beta_g: torch.Tensor, stride: int = AFFINE_STRIDE) -> torch.Tensor:
    """UniversalParams::lagrange_basis (kzg10/data_structures.rs:68-72): ifft of the first n powers, normalised to affine."""
    return g1_ntt(powers_of_beta_g, True, stride)


def _fr_host(x) -> np.ndarray:
    a = np.ascontiguousarray(x, dtype=np.uint64).reshape(4)
    return a


def fr_batch_inversion_and_mul(v: torch.Tensor, coeff_mont) -> torch.Tensor:
    """fields/src/lib.rs:78-129, in place on a CUDA tensor of Montgomery Fr: v_i ← coeff·v_i^{-1}; zeros stay zero."""
    c = _fr_host(coeff_mont)
    with torch.cuda.device(v.device):
        _lib.check(_lib.lib().snarkvm_b200_fr_batch_inversion_and_mul_device(_check(v, "v"), _nbytes(v) // 32, c.ctypes.data, _stream()))
    return v


def poly_divide_by_vanishing(p: torch.Tensor, domain_size: int):
    """DensePolynomial::divide_by_vanishing_poly (fft/polynomial/dense.rs:162-169) → (quotient, remainder) CUDA tensors [.., 4] i64,
    max(m − n, 0) and min(m, n) coefficients, not trimmed."""
    m = _nbytes(p) // 32
    q = torch.empty((max(m - domain_size, 0), 4), dtype=torch.int64, device=p.device)
    r = torch.empty((min(m, domain_size), 4), dtype=torch.int64, device=p.device)
    if m:
        with torch.cuda.device(p.device):
            _lib.check(_lib.lib().snarkvm_b200_poly_divide_by_vanishing_device(q.data_ptr() if q.numel() else None, r.data_ptr(),
                                                                                _check(p, "p"), m, domain_size, _stream()))
    return q, r


FR_ADD, FR_SUB, FR_MUL = 0, 1, 2


def fr_vec_op(a: torch.Tensor, b, op: int, out: torch.Tensor | None = None) -> torch.Tensor:
    """Elementwise a (op) b on Montgomery Fr vectors in HBM; b is a tensor of the same length or one 32-byte host scalar."""
    out = torch.empty_like(a) if out is None else out
    n = _nbytes(a) // 32
    with torch.cuda.device(a.device):
        if isinstance(b, torch.Tensor):
            if _nbytes(b) != _nbytes(a):
                raise ValueError("length mismatch")
            _lib.check(_lib.lib().snarkvm_b200_fr_vec_op_device(out.data_ptr(), _check(a, "a"), _check(b, "b"), n, op, _stream()))
        else:
            s = _fr_host(b)
            _lib.check(_lib.lib().snarkvm_b200_fr_vec_scalar_op_device(out.data_ptr(), _check(a, "a"), s.ctypes.data, n, op, _stream()))
    return out


def domain_elements(lg: int, device="cuda") -> torch.Tensor:
    """EvaluationDomain::elements (fft/domain.rs:307-309): [2^lg, 4] i64, element i = group_gen^i (Montgomery)."""
    out = torch.empty((1 << lg, 4), dtype=torch.int64, device=device)
    with torch.cuda.device(out.device):
        _lib.check(_lib.lib().snarkvm_b200_domain_elements_device(out.data_ptr(), lg, _stream()))
    return out


INDEX_MATERIALISE, INDEX_EVALUATE = 0, 1


def index_arithmetize(matrices: list, k_sizes: list, num_variables: int, num_public: int, lagrange: list | None = None):
    """The indexer's arithmetization of A, B, C (matrix_evals, ahp/matrices.rs:138-190) in one launch.
    `matrices`: three (row_ptr int32 [nrows + 1], cols int32 [nnz], vals [nnz, 4] i64 Montgomery) CUDA tensors with the same nrows;
    `k_sizes`: the three non-zero domain sizes (powers of two ≥ nnz); `num_public`: the input domain size (a power of two below the
    variable domain's size).
    Without `lagrange`: → per matrix the CUDA tensors (row, col, row_col, row_col_val) [K, 4] i64 Montgomery.
    With `lagrange` (per matrix the Lagrange coefficients of K at a point, [K, 4] Montgomery): → the twelve sums Σ_κ L_κ·e(κ) as
    Montgomery uint64 [3, 4, 4] on the host (matrix, vector), without storing the evaluations (indexer.rs:232-260)."""
    if len(matrices) != 3 or len(k_sizes) != 3:
        raise ValueError("three matrices (A, B, C) and three non-zero domain sizes")
    nrows = matrices[0][0].numel() - 1
    if nrows < 1:
        raise ValueError("a circuit needs at least one constraint")
    if num_public < 1 or num_public & (num_public - 1):
        raise ValueError("the number of public variables must be a power of two")
    if num_public >= 1 << max(num_variables - 1, 0).bit_length():
        raise ValueError("the input domain must be smaller than the variable domain")
    lg_k, nnz = [], []
    for (row_ptr, cols, vals), k in zip(matrices, k_sizes):
        if row_ptr.dtype != torch.int32 or cols.dtype != torch.int32:
            raise TypeError("row_ptr and cols must be int32 tensors")
        if row_ptr.numel() - 1 != nrows:
            raise ValueError("A, B and C must have the same number of rows")
        n = cols.numel()
        if _nbytes(vals) != 32 * n:
            raise ValueError("one value per column index")
        if k < 1 or k & (k - 1) or n > k:
            raise ValueError(f"non-zero domain of size {k} cannot hold {n} entries")
        lg_k.append(k.bit_length() - 1)
        nnz.append(n)
    dev = matrices[0][0].device
    rp = (ctypes.c_void_p * 3)(*[_check(m[0], "row_ptr") for m in matrices])
    cp = (ctypes.c_void_p * 3)(*[(_check(m[1], "cols") if n else None) for m, n in zip(matrices, nnz)])
    vp = (ctypes.c_void_p * 3)(*[(_check(m[2], "vals") if n else None) for m, n in zip(matrices, nnz)])
    nz = (ctypes.c_size_t * 3)(*nnz)
    lk = (ctypes.c_uint32 * 3)(*lg_k)
    if lagrange is None:
        outs = [tuple(torch.empty((k, 4), dtype=torch.int64, device=dev) for _ in range(4)) for k in k_sizes]
        io = (ctypes.c_void_p * 12)(*[t.data_ptr() for o in outs for t in o])
        sums = None
    else:
        if len(lagrange) != 3 or any(_nbytes(l) != 32 * k for l, k in zip(lagrange, k_sizes)):
            raise ValueError("one Lagrange coefficient vector of |K| elements per matrix")
        io = (ctypes.c_void_p * 3)(*[_check(l, "lagrange") for l in lagrange])
        sums = np.zeros((3, 4, 4), dtype=np.uint64)
    with torch.cuda.device(dev):
        _lib.check(_lib.lib().snarkvm_b200_index_arithmetize_device(
            INDEX_MATERIALISE if lagrange is None else INDEX_EVALUATE, rp, cp, vp, nz, lk, nrows, num_variables, num_public, io,
            sums.ctypes.data if sums is not None else None, _stream()))
    return outs if lagrange is None else sums


def sparse_matvec(row_ptr: torch.Tensor, cols: torch.Tensor, vals: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """z_M = M·x for a CSR matrix over Fr (inner_product per row, varuna/ahp/prover/round_functions/mod.rs:130-189).
    row_ptr: int32 [nrows + 1], cols: int32 [nnz], vals: [nnz, 4] i64 Montgomery, x: [nvars, 4] i64 Montgomery → [nrows, 4] i64."""
    if row_ptr.dtype != torch.int32 or cols.dtype != torch.int32:
        raise TypeError("row_ptr and cols must be int32 tensors")
    nrows = row_ptr.numel() - 1
    out = torch.empty((max(nrows, 0), 4), dtype=torch.int64, device=x.device)
    if nrows > 0:
        with torch.cuda.device(x.device):
            _lib.check(_lib.lib().snarkvm_b200_sparse_matvec_device(out.data_ptr(), _check(row_ptr, "row_ptr"),
                                                                     _check(cols, "cols") if cols.numel() else None,
                                                                     _check(vals, "vals") if vals.numel() else None, nrows, _check(x, "x"),
                                                                     _nbytes(x) // 32, _stream()))
    return out


def poly_divide_by_linear(p: torch.Tensor, point_mont) -> torch.Tensor:
    """Quotient of p / (x − point), the KZG witness polynomial (kzg10/mod.rs:220-241) → CUDA tensor [m − 1, 4] i64, not trimmed."""
    z = _fr_host(point_mont)
    m = _nbytes(p) // 32
    q = torch.empty((max(m - 1, 0), 4), dtype=torch.int64, device=p.device)
    if m > 1:
        with torch.cuda.device(p.device):
            _lib.check(_lib.lib().snarkvm_b200_poly_divide_by_linear_device(q.data_ptr(), _check(p, "p"), m, z.ctypes.data, _stream()))
    return q


def poly_evaluate(coeffs: torch.Tensor, point_mont) -> np.ndarray:
    """DensePolynomial::evaluate (fft/polynomial/dense.rs:98-114) → Montgomery Fr as uint64[4] on the host."""
    z = _fr_host(point_mont)
    out = np.zeros(4, dtype=np.uint64)
    m = _nbytes(coeffs) // 32
    with torch.cuda.device(coeffs.device):
        _lib.check(_lib.lib().snarkvm_b200_poly_evaluate_device(out.ctypes.data, _check(coeffs, "coeffs") if m else None, m, z.ctypes.data, _stream()))
    return out


class PrecomputedBases:
    """A fixed base set with its tables 2^{c·w}·P_i resident in HBM (snarkvm_b200_msm_precompute_device): MSMs over it use one
    bucket set for all windows.  `msm(scalars)` / `kzg_commit(coeffs_mont)` take the first len(scalars) bases, like
    `&powers_of_beta_g[..len]` in KZG10::commit (kzg10/mod.rs:121-135)."""

    def __init__(self, bases: torch.Tensor, stride: int = AFFINE_STRIDE):
        npoints = _nbytes(bases) // stride
        self.device = bases.device
        h = ctypes.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().snarkvm_b200_msm_precompute_device(ctypes.byref(h), _check(bases, "bases"), npoints, stride, _stream()))
        self._h = h
        n, c, nwin, tb = ctypes.c_size_t(), ctypes.c_int(), ctypes.c_int(), ctypes.c_size_t()
        _lib.check(_lib.lib().snarkvm_b200_msm_precomputed_info(h, ctypes.byref(n), ctypes.byref(c), ctypes.byref(nwin), ctypes.byref(tb)))
        self.npoints, self.c, self.nwin, self.table_bytes = n.value, c.value, nwin.value, tb.value

    def _run(self, fn, scalars: torch.Tensor) -> np.ndarray:
        if self._h is None:
            raise ValueError("PrecomputedBases was freed")
        n = _nbytes(scalars) // 32
        if n > self.npoints:
            raise ValueError("more scalars than bases")
        out = np.zeros(18, dtype=np.uint64)
        with torch.cuda.device(self.device):
            _lib.check(fn(out.ctypes.data, self._h, _check(scalars, "scalars") if n else None, n, _stream()))
        return out

    def msm(self, scalars: torch.Tensor) -> np.ndarray:
        return self._run(_lib.lib().snarkvm_b200_msm_precomputed_device, scalars)

    def kzg_commit(self, coeffs_mont: torch.Tensor) -> np.ndarray:
        return self._run(_lib.lib().snarkvm_b200_kzg_commit_precomputed_device, coeffs_mont)

    def kzg_commit_batch(self, polys_mont: list) -> np.ndarray:
        """all commitments of a round over the tables, one pass → [count, 18] u64"""
        if self._h is None:
            raise ValueError("PrecomputedBases was freed")
        count = len(polys_mont)
        out = np.zeros((count, 18), dtype=np.uint64)
        if count == 0:
            return out
        lens = [_nbytes(p) // 32 for p in polys_mont]
        if max(lens) > self.npoints:
            raise ValueError("more coefficients than bases")
        ptrs = (ctypes.c_void_p * count)(*[(_check(p, "poly") if n else None) for p, n in zip(polys_mont, lens)])
        szs = (ctypes.c_size_t * count)(*lens)
        with torch.cuda.device(self.device):
            _lib.check(_lib.lib().snarkvm_b200_kzg_commit_batch_precomputed_device(out.ctypes.data, self._h, ptrs, szs, count, _stream()))
        return out

    def free(self) -> None:
        if self._h is not None:
            _lib.check(_lib.lib().snarkvm_b200_msm_precomputed_free(self._h))
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def fr_from_mont(x: torch.Tensor) -> torch.Tensor:
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().snarkvm_b200_fr_from_mont_device(out.data_ptr(), _check(x, "x"), _nbytes(x) // 32, _stream()))
    return out


def fr_to_mont(x: torch.Tensor) -> torch.Tensor:
    out = torch.empty_like(x)
    with torch.cuda.device(x.device):
        _lib.check(_lib.lib().snarkvm_b200_fr_to_mont_device(out.data_ptr(), _check(x, "x"), _nbytes(x) // 32, _stream()))
    return out


def generate_bases(npoints: int, seed: int, device="cuda", stride: int = AFFINE_STRIDE) -> torch.Tensor:
    """Synthetic G1 bases P_i = h(seed, i)·G in the reference affine layout, generated in HBM."""
    t = torch.empty((npoints, stride), dtype=torch.uint8, device=device)
    with torch.cuda.device(t.device):
        _lib.check(_lib.lib().snarkvm_b200_generate_bases_device(t.data_ptr(), npoints, stride, seed & (2**64 - 1), _stream()))
    return t


def srs_decode(usrs_points: torch.Tensor, stride: int = AFFINE_STRIDE):
    """`.usrs` payload in HBM (uint8, 96 B per uncompressed canonical point, count header already stripped) →
    (bases in the reference affine layout, number of invalid points).  parameters/src/mainnet/powers.rs."""
    nbytes = _nbytes(usrs_points)
    if nbytes % 96:
        raise ValueError("payload must be a whole number of 96-byte points")
    n = nbytes // 96
    out = torch.empty((n, stride), dtype=torch.uint8, device=usrs_points.device)
    invalid = torch.zeros(1, dtype=torch.int32, device=usrs_points.device)
    with torch.cuda.device(usrs_points.device):
        _lib.check(_lib.lib().snarkvm_b200_srs_decode_device(out.data_ptr(), stride, _check(usrs_points, "usrs_points"), n,
                                                              invalid.data_ptr(), _stream()))
    return out, int(invalid.item())
