"""Varuna AHP prover rounds with every polynomial resident in HBM (SURVEY §8 f3).

Device-side mirror of /root/reference/algorithms/src/snark/varuna for the part of `prove_batch` (varuna.rs:336-620) that is
bulk field arithmetic — the five `AHPForR1CS::prover_*_round` functions and the indexer's arithmetization:

    ahp/indexer/indexer.rs:121-200, ahp/matrices.rs:138-190, 239-254   Circuit            (domains, row / col / row_col / row_col_val on K, transposes)
    ahp/indexer/circuit.rs:109-148, varuna.rs:72-134, 236-331           circuit setup      (info, id, index polynomials, batch_circuit_setup, prove_vk,
                                                                                         evaluate_index_polynomials)
    ahp/prover/round_functions/mod.rs:43-192, ahp/prover/state.rs:107-178   init_prover   (z_A, z_B, z_C by sparse mat-vec, x_poly)
    ahp/prover/round_functions/first.rs:129-160    prover_first_round   (w)
    ahp/prover/round_functions/third.rs:207-234    calculate_assignments (z)
    ahp/prover/round_functions/second.rs:77-146    prover_second_round  (h_0)
    ahp/prover/round_functions/third.rs:126-326    prover_third_round   (g_1, h_1, lineval sums)
    ahp/prover/round_functions/fourth.rs:151-245   prover_fourth_round  (g_a, g_b, g_c, sums)
    ahp/prover/round_functions/fifth.rs:41-67      prover_fifth_round   (h_2)
    ahp/selectors.rs:70-123                        apply_randomized_selector

for the NON-HIDING mode (VarunaNonHidingMode), one circuit, any batch of instances.  Everything O(n) runs in this library's
kernels (NTT passes, PolyMultiplier pipeline, divide_by_vanishing_poly, batch inversion, sparse mat-vec, elementwise Fr ops);
torch only owns the buffers and does index plumbing (gathers, concatenation).  Challenges are host scalars: the Fiat-Shamir
sponge (Poseidon) is sequential and stays on the CPU (SURVEY §8 f3), so callers pass α, η, β, δ in.
Polynomials are CUDA tensors [m, 4] int64 (Montgomery Fr, low degree first, NOT trimmed: trailing zero coefficients may be present;
`trimmed()` gives the reference's canonical form on the host).
"""
from __future__ import annotations

import hashlib
import struct
from dataclasses import astuple, dataclass

import numpy as np
import torch

from . import device
from .algorithms import EvaluationDomain, _fr_int_to_mont, _fr_mont_to_int
from .sonic_pc import CommitterKey, LabeledPolynomial, Randomness, SonicKZG10

R_MOD = 8444461749428370424248824938781546531375899335154063827935233455917409239041   # curves/src/bls12_377/fr.rs:138-145


def _mont(v: int) -> np.ndarray:
    return _fr_int_to_mont(v % R_MOD)


def _zeros(n: int, dev) -> torch.Tensor:
    return torch.zeros((n, 4), dtype=torch.int64, device=dev)


def _pad(x: torch.Tensor, n: int) -> torch.Tensor:
    if x.shape[0] == n:
        return x
    out = _zeros(n, x.device)
    out[: x.shape[0]] = x[:n]
    return out


def _scale(x: torch.Tensor, k: int) -> torch.Tensor:
    if x.shape[0] == 0 or k % R_MOD == 1:
        return x
    return device.fr_vec_op(x, _mont(k), device.FR_MUL)


def _add(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """a + b for polynomials of different lengths"""
    if a.shape[0] < b.shape[0]:
        a, b = b, a
    if b.shape[0] == 0:
        return a
    out = a.clone()
    device.fr_vec_op(out[: b.shape[0]], b, device.FR_ADD, out=out[: b.shape[0]])
    return out


def _sub(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    n = max(a.shape[0], b.shape[0])
    out = _pad(a, n).clone() if a.shape[0] == n else _pad(a, n)
    if b.shape[0]:
        device.fr_vec_op(out[: b.shape[0]], b, device.FR_SUB, out=out[: b.shape[0]])
    return out


def trimmed(poly: torch.Tensor) -> list:
    """host copy as canonical integers with trailing zeros removed (DensePolynomial::from_coefficients_vec, dense.rs:61-66)"""
    h = device.fr_from_mont(poly).cpu().numpy().view(np.uint64) if poly.shape[0] else np.zeros((0, 4), dtype=np.uint64)
    vals = [sum(int(v) << (64 * i) for i, v in enumerate(row)) for row in h]
    while vals and vals[-1] == 0:
        vals.pop()
    return vals


def polymul(a: torch.Tensor, b: torch.Tensor) -> torch.Tensor:
    """PolyMultiplier::multiply of two coefficient vectors (fft/polynomial/multiplier.rs:70-134)"""
    if a.shape[0] == 0 or b.shape[0] == 0:
        return _zeros(0, a.device)
    dom = EvaluationDomain.new(a.shape[0] + b.shape[0] - 1)
    return device.polymul([a.contiguous(), b.contiguous()], [], dom.log_size_of_group)


def divide_by_vanishing(p: torch.Tensor, domain: EvaluationDomain):
    return device.poly_divide_by_vanishing(p.contiguous(), domain.size)


def mul_by_vanishing(p: torch.Tensor, domain: EvaluationDomain) -> torch.Tensor:
    """DensePolynomial::mul_by_vanishing_poly (dense.rs:153-158): p·(x^n − 1)"""
    n, m = domain.size, p.shape[0]
    out = _zeros(n + m, p.device)
    out[n:] = p
    device.fr_vec_op(out[:m], p, device.FR_SUB, out=out[:m])       # out[:m] −= p (for m > n the shifted copy is already there)
    return out


def apply_randomized_selector(poly: torch.Tensor, combiner: int, target: EvaluationDomain, src: EvaluationDomain, remainder_witness: bool):
    """ahp/selectors.rs:70-123"""
    multiplier = combiner * src.size % R_MOD * pow(target.size, -1, R_MOD) % R_MOD
    if not remainder_witness:
        h, _rem = divide_by_vanishing(poly, src)               # the reference asserts a zero remainder; parity tests check the result
        return _scale(h, multiplier), None
    poly = _scale(poly, multiplier)
    h, xg = divide_by_vanishing(poly, src)
    if target.size != src.size:
        xg = mul_by_vanishing(xg, target)
        xg, _rem = divide_by_vanishing(xg, src)
    return h, xg


def reindex_by_subdomain(variable_size: int, input_size: int, index: np.ndarray) -> np.ndarray:
    """EvaluationDomain::reindex_by_subdomain (fft/domain.rs:322-344), vectorised"""
    if variable_size <= input_size:
        raise ValueError("other.size() must be smaller than self.size()")
    period = variable_size // input_size
    index = np.asarray(index, dtype=np.int64)
    i = index - input_size
    x = period - 1
    return np.where(index < input_size, index * period, i + i // x + 1)


class Matrix:
    """A sparse R1CS matrix in CSR form on the device: row_ptr int32 [nrows + 1], cols int32 [nnz] (variable indices: public first,
    then private — into_matrix_helper, ahp/matrices.rs:39-63), vals [nnz, 4] int64 Montgomery."""

    def __init__(self, row_ptr: np.ndarray, cols: np.ndarray, vals_mont: np.ndarray, dev):
        self.row_ptr_h = np.ascontiguousarray(row_ptr, dtype=np.int64)
        self.cols_h = np.ascontiguousarray(cols, dtype=np.int64)
        self.nrows, self.nnz = len(row_ptr) - 1, len(cols)
        self.row_ptr = torch.from_numpy(self.row_ptr_h.astype(np.int32)).to(dev)
        self.cols = torch.from_numpy(self.cols_h.astype(np.int32)).to(dev)
        self.vals = torch.from_numpy(np.ascontiguousarray(vals_mont, dtype=np.uint64).reshape(-1, 4).view(np.int64)).to(dev)


class MatrixEvals:
    """ahp/matrices.rs:102-136: row, col, row_col, row_col_val evaluations on the non-zero domain K"""

    def __init__(self, row, col, row_col, row_col_val, domain):
        self.row, self.col, self.row_col, self.row_col_val, self.domain = row, col, row_col, row_col_val, domain

    def vectors(self) -> tuple:
        return self.row, self.col, self.row_col, self.row_col_val


@dataclass(frozen=True)
class CircuitInfo:
    """ahp/indexer/circuit_info.rs:25-38"""
    num_public_inputs: int
    num_public_and_private_variables: int
    num_constraints: int
    num_non_zero_a: int
    num_non_zero_b: int
    num_non_zero_c: int

    def to_bytes(self) -> bytes:
        """the uncompressed serialisation (derive(CanonicalSerialize)): six u64, little-endian"""
        return struct.pack("<6Q", *astuple(self))

    def max_degree(self, hiding: bool) -> int:
        """AHPForR1CS::max_degree (ahp/ahp.rs:85-108) with zk_bound 1 in the hiding mode"""
        zk = 1 if hiding else 0
        size = EvaluationDomain.compute_size_of_domain
        r, v = size(self.num_constraints), size(self.num_public_and_private_variables)
        k = size(max(self.num_non_zero_a, self.num_non_zero_b, self.num_non_zero_c))
        return max(2 * r + 2 * zk - 2, 2 * v + 2 * zk - 2, v + 3 if hiding else 0, v, r, k - 1)

    def degree_bounds(self) -> list:
        """AHPForR1CS::get_degree_bounds (ahp/ahp.rs:110-121): |C| − 2 and |K_M| − 2"""
        size = EvaluationDomain.compute_size_of_domain
        bounds = [size(n) - 2 for n in (self.num_public_and_private_variables, self.num_non_zero_a, self.num_non_zero_b, self.num_non_zero_c)]
        if min(bounds) < 0:
            raise ValueError("every non-zero domain needs at least two elements to bound the degree of its g polynomial")
        return bounds


def _matrix_bytes(m: Matrix) -> bytes:
    """Matrix<F> = Vec<Vec<(F, usize)>> serialised uncompressed (utilities/src/serialize/impls.rs:151-160, 392-420, 524-550 and
    fields/src/macros.rs:191-): u64 row count; per row a u64 entry count, then per entry the value as 32 canonical little-endian
    bytes and its column as u64."""
    entries = np.zeros((m.nnz, 40), dtype=np.uint8)
    if m.nnz:
        entries[:, :32] = device.fr_from_mont(m.vals).cpu().numpy().view(np.uint8).reshape(m.nnz, 32)
        entries[:, 32:] = m.cols_h.astype("<u8").view(np.uint8).reshape(m.nnz, 8)
    body = np.empty(m.nrows * 8 + m.nnz * 40, dtype=np.uint8)
    header = np.zeros(body.size, dtype=bool)                          # row r's count sits after r counts and row_ptr[r] entries
    header[((np.arange(m.nrows) * 8 + m.row_ptr_h[:-1] * 40)[:, None] + np.arange(8)).ravel()] = True
    body[header] = np.diff(m.row_ptr_h).astype("<u8").view(np.uint8)
    body[~header] = entries.ravel()
    return struct.pack("<Q", m.nrows) + body.tobytes()


def index_polynomial_labels(circuit_id) -> list:
    """AHPForR1CS::index_polynomial_labels (ahp/indexer/indexer.rs:104-122) for matrices a, b, c, in the indexer's order; the id is
    printed as lowercase hex (ahp/indexer/circuit.rs:42-48)"""
    cid = circuit_id.hex() if isinstance(circuit_id, (bytes, bytearray)) else str(circuit_id)
    return [f"circuit_{cid}_{poly}_{m}" for m in "abc" for poly in ("row", "col", "row_col", "row_col_val")]


class Circuit:
    """AHPForR1CS::index_helper (ahp/indexer/indexer.rs:121-200): the caller has already padded the public variables to a power of
    two (pad_input_for_indexer_and_prover, ahp/matrices.rs:85-100) and, for the hiding mode, added the randomizing variables and
    their constraint before that (add_randomizing_variables, ahp/matrices.rs:64-82).  The arithmetization of A, B, C is one
    device launch (device.index_arithmetize)."""

    def __init__(self, a: Matrix, b: Matrix, c: Matrix, num_public: int, num_variables: int):
        dev = a.vals.device
        self.a, self.b, self.c = a, b, c
        self.num_public, self.num_variables, self.num_constraints = num_public, num_variables, a.nrows
        if num_public & (num_public - 1):
            raise ValueError("public variables must be padded to a power of two")
        self.constraint_domain = EvaluationDomain.new(self.num_constraints)
        self.variable_domain = EvaluationDomain.new(num_variables)
        self.input_domain = EvaluationDomain.new(num_public)
        self.non_zero_domains = [EvaluationDomain.new(m.nnz) for m in (a, b, c)]
        self.max_non_zero_domain = max(self.non_zero_domains, key=lambda d: d.size)
        self._id = None
        self.ariths, self.transposes = [], []
        evals = device.index_arithmetize(self._csr(), [K.size for K in self.non_zero_domains], num_variables, num_public)
        for m, K, e in zip((a, b, c), self.non_zero_domains, evals):
            self.ariths.append(MatrixEvals(*e, K))                                              # matrix_evals (ahp/matrices.rs:138-190)
            entry_rows = np.repeat(np.arange(m.nrows, dtype=np.int64), np.diff(m.row_ptr_h))
            entry_cols = reindex_by_subdomain(self.variable_domain.size, self.input_domain.size, m.cols_h)
            # transpose (ahp/matrices.rs:239-254) as CSR over the variable domain's indices; entries keep the row-major order
            order = np.argsort(entry_cols, kind="stable")
            counts = np.bincount(entry_cols, minlength=self.variable_domain.size)
            t_ptr = np.concatenate([[0], np.cumsum(counts)])
            t_vals = m.vals[torch.from_numpy(order).to(dev)] if m.nnz else m.vals
            tm = Matrix.__new__(Matrix)
            tm.nrows, tm.nnz = self.variable_domain.size, m.nnz
            tm.row_ptr = torch.from_numpy(t_ptr.astype(np.int32)).to(dev)
            tm.cols = torch.from_numpy(entry_rows[order].astype(np.int32)).to(dev)
            tm.vals = t_vals.contiguous()
            self.transposes.append(tm)

    def _csr(self) -> list:
        return [(m.row_ptr, m.cols, m.vals) for m in (self.a, self.b, self.c)]

    def info(self) -> CircuitInfo:
        """CircuitInfo of the index (ahp/indexer/indexer.rs:169-176)"""
        return CircuitInfo(self.num_public, self.num_variables, self.num_constraints, self.a.nnz, self.b.nnz, self.c.nnz)

    def id(self) -> bytes:
        """Circuit::hash (ahp/indexer/circuit.rs:109-121): Blake2s-256 over the uncompressed serialisation of the info and of A, B, C"""
        if self._id is None:
            h = hashlib.blake2s(digest_size=32)
            h.update(self.info().to_bytes())
            for m in (self.a, self.b, self.c):
                h.update(_matrix_bytes(m))
            self._id = h.digest()
        return self._id

    def interpolate_matrix_evals(self) -> list:
        """Circuit::interpolate_matrix_evals (ahp/indexer/circuit.rs:142-148, MatrixArithmetization::new, ahp/matrices.rs:213-240): the
        twelve index polynomials — the iFFT over K_M of row, col, row_col, row_col_val for M = A, B, C — with no degree or hiding
        bound, in the indexer's label order"""
        polys = []
        for arith in self.ariths:
            for v in arith.vectors():
                polys.append(v.clone() if arith.domain.size == 1 else arith.domain.ifft(v))      # a one-point iFFT is the identity
        return [LabeledPolynomial(label, p) for label, p in zip(index_polynomial_labels(self.id()), polys)]


class Prover:
    """init_prover + State::initialize (round_functions/mod.rs:43-170, state.rs:107-178) and the five rounds.
    `assignments`: one CUDA tensor [num_variables, 4] per instance — padded public variables (first one is One) then private."""

    def __init__(self, circuit: Circuit, assignments: list):
        self.circuit = c = circuit
        self.batch = len(assignments)
        self.z = [z.contiguous() for z in assignments]
        for z in self.z:
            if z.shape[0] != c.num_variables:
                raise ValueError("instance does not match the index")                       # AHPError::InstanceDoesNotMatchIndex
        self.z_a = [device.sparse_matvec(c.a.row_ptr, c.a.cols, c.a.vals, z) for z in self.z]
        self.z_b = [device.sparse_matvec(c.b.row_ptr, c.b.cols, c.b.vals, z) for z in self.z]
        self.z_c = [device.sparse_matvec(c.c.row_ptr, c.c.cols, c.c.vals, z) for z in self.z]
        self.x_polys = [c.input_domain.ifft(z[: c.num_public]) for z in self.z]                 # state.rs:137-139

    # ---- round 1: calculate_w (first.rs:129-160) ----
    def first_round(self):
        c = self.circuit
        V, I = c.variable_domain, c.input_domain
        dev = self.z[0].device
        # the index plumbing of calculate_w depends only on the two domain sizes: built once per circuit and device, on the device
        # (building it with numpy and uploading it every proof was 15 of the round's 21 ms at 2^20 constraints)
        cache = c.__dict__.setdefault("_w_index", {})
        if dev not in cache:
            ratio = V.size // I.size
            k = torch.arange(V.size, dtype=torch.int64, device=dev)
            mask = (k % ratio) != 0
            cache[dev] = (k[mask].contiguous(), (k - torch.div(k, ratio, rounding_mode="floor") - 1)[mask].contiguous())
        keep, src = cache[dev]
        self.w_polys = []
        for z, x_poly in zip(self.z, self.x_polys):
            w_ext = _zeros(V.size - I.size, dev)
            prv = z[c.num_public:]
            w_ext[: prv.shape[0]] = prv
            x_evals = V.fft_in_place(_pad(x_poly, V.size).clone())
            evals = _zeros(V.size, dev)
            evals[keep] = device.fr_vec_op(w_ext[src].contiguous(), x_evals[keep].contiguous(), device.FR_SUB)
            w_poly, _rem = divide_by_vanishing(V.ifft_in_place(evals), I)
            self.w_polys.append(w_poly)
        return self.w_polys

    # ---- calculate_assignments (third.rs:207-234): z = w·v_I + x ----
    def assignments(self):
        I = self.circuit.input_domain
        self.z_polys = [_add(mul_by_vanishing(w, I), x) for w, x in zip(self.w_polys, self.x_polys)]
        return self.z_polys

    # ---- round 2: calculate_rowcheck_witness (second.rs:77-146) ----
    def second_round(self, circuit_combiner: int = 1, instance_combiners=None):
        c = self.circuit
        Rd = c.constraint_domain
        instance_combiners = instance_combiners or [1] * self.batch
        h_0 = _zeros(0, self.z[0].device)
        for comb, za, zb, zc in zip(instance_combiners, self.z_a, self.z_b, self.z_c):
            pa, pb, pc = (Rd.ifft_in_place(_pad(e, Rd.size).clone()) for e in (za, zb, zc))
            rowcheck = _sub(polymul(pa, pb), pc)
            h_i, _ = apply_randomized_selector(_scale(rowcheck, comb), circuit_combiner, Rd, Rd, False)
            h_0 = _add(h_0, h_i)
        self.h_0 = h_0
        return h_0

    # ---- evaluate_all_lagrange_coefficients (fft/domain.rs:258-292) on the device ----
    @staticmethod
    def lagrange_coefficients(domain: EvaluationDomain, tau: int, dev) -> torch.Tensor:
        return domain.evaluate_all_lagrange_coefficients(tau, dev)

    # ---- round 3: lineval sumcheck (third.rs:126-205, 266-326) ----
    def third_round(self, alpha: int, eta_b: int, eta_c: int, circuit_combiner: int = 1, instance_combiners=None):
        c = self.circuit
        Rd, V = c.constraint_domain, c.variable_domain
        dev = self.z[0].device
        instance_combiners = instance_combiners or [1] * self.batch
        l_at_alpha = self.lagrange_coefficients(Rd, alpha, dev)
        h_1, xg_1, sums = _zeros(0, dev), _zeros(0, dev), []
        m_polys = []
        for tm in c.transposes:
            m_evals = device.sparse_matvec(tm.row_ptr, tm.cols, tm.vals, l_at_alpha)            # M(α, c) for every c ∈ C
            m_polys.append(V.ifft_in_place(m_evals))
        for inst_comb, z_poly in zip(instance_combiners, self.z_polys):
            inst_sums = []
            for m_at_alpha, m_comb in zip(m_polys, (1, eta_b % R_MOD, eta_c % R_MOD)):
                z_m = polymul(m_at_alpha, z_poly)
                # Σ_{c ∈ C} z_m(c) = |C| · Σ_j coefficient_{j·|C|}
                picks = device.fr_from_mont(z_m[:: V.size].contiguous()).cpu().numpy().view(np.uint64)
                inst_sums.append(V.size * sum(sum(int(v) << (64 * i) for i, v in enumerate(row)) for row in picks) % R_MOD)
                combiner = circuit_combiner * inst_comb % R_MOD * m_comb % R_MOD
                h_i, xg_i = apply_randomized_selector(z_m, combiner, V, V, True)
                h_1, xg_1 = _add(h_1, h_i), _add(xg_1, xg_i)
            sums.append(inst_sums)
        if self.mask_poly is not None:                                  # third.rs:207-213 (hiding mode)
            h_mask, xg_mask = divide_by_vanishing(self.mask_poly, V)
            h_1, xg_1 = _add(h_1, h_mask), _add(xg_1, xg_mask)
        self.h_1, self.g_1, self.third_sums = h_1, xg_1[1:].contiguous(), sums
        return self.g_1, self.h_1

    # ---- AHPForR1CS::construct_linear_combinations (ahp/ahp.rs:172-389) + verifier_query_set, one circuit ----
    def polynomials(self) -> dict:
        """label → device polynomial, everything prove_batch hands to open_combinations (varuna.rs:509-517)"""
        out = {f"w_{j}": w for j, w in enumerate(self.w_polys)}
        if self.mask_poly is not None:
            out["mask_poly"] = self.mask_poly
        out.update({"h_0": self.h_0, "g_1": self.g_1, "h_1": self.h_1, "h_2": self.h_2})
        for m, g, a, b in zip("abc", self.gs, self.a_polys, self.b_polys):
            out[f"g_{m}"], out[f"a_poly_{m}"], out[f"b_poly_{m}"] = g, a, b
        return out

    @staticmethod
    def _eval(poly: torch.Tensor, point: int) -> int:
        return _fr_mont_to_int(device.poly_evaluate(poly.contiguous(), _mont(point))) if poly.shape[0] else 0

    def linear_combinations(self, alpha, eta_b, eta_c, beta, deltas, gamma, circuit_combiner: int = 1, instance_combiners=None):
        """→ (lcs, query_set) exactly as oracle/varuna.py Prover.linear_combinations: the coefficients are host integers (a few dozen
        field operations), the three evaluations they need — g_1(β), g_M(γ), x_j(β) — are device Horner passes."""
        c = self.circuit
        Rd, V, I, K = c.constraint_domain, c.variable_domain, c.input_domain, c.max_non_zero_domain
        vanish = lambda d, x: (pow(x, d.size, R_MOD) - 1) % R_MOD       # noqa: E731
        instance_combiners = instance_combiners or [1] * self.batch
        lcs = {}
        const = 0
        for comb, sums in zip(instance_combiners, self.third_sums):
            const = (const + comb * (sums[0] * sums[1] - sums[2])) % R_MOD
        lcs["rowcheck_zerocheck"] = [(circuit_combiner * const % R_MOD, None), ((-vanish(Rd, alpha)) % R_MOD, "h_0")]
        lcs["g_1"] = [(1, "g_1")]
        v_c_beta, v_x_beta = vanish(V, beta), vanish(I, beta)
        g_1_at_beta = self._eval(self.g_1, beta)
        doms = [a.domain for a in c.ariths]
        sums4 = [s * d.size % R_MOD for s, d in zip(self.fourth_sums, doms)]
        weight = (sums4[0] + sums4[1] * eta_b + sums4[2] * eta_c) % R_MOD
        lineval = [(1, "mask_poly")] if self.mask_poly is not None else []
        for j, comb in enumerate(instance_combiners):
            x_at_beta = self._eval(self.x_polys[j], beta)
            k = circuit_combiner * comb % R_MOD
            lineval.append((k * weight % R_MOD * x_at_beta % R_MOD, None))
            lineval.append((k * weight % R_MOD * v_x_beta % R_MOD, f"w_{j}"))
        batch_lineval_sum = circuit_combiner * sum(comb * (s[0] + eta_b * s[1] + eta_c * s[2]) for comb, s in zip(instance_combiners, self.third_sums)) % R_MOD \
            * pow(V.size, -1, R_MOD) % R_MOD
        lineval += [((-v_c_beta) % R_MOD, "h_1"), ((-beta * g_1_at_beta) % R_MOD, None), ((-batch_lineval_sum) % R_MOD, None)]
        lcs["lineval_sumcheck"] = lineval
        v_k_gamma = vanish(K, gamma)
        matrix = []
        for m, g, s, delta, dom in zip("abc", self.gs, self.fourth_sums, deltas, doms):
            lcs[f"g_{m}"] = [(1, f"g_{m}")]
            selector = v_k_gamma * dom.size % R_MOD * pow(vanish(dom, gamma) * K.size % R_MOD, -1, R_MOD) % R_MOD
            b_term = (gamma * self._eval(g, gamma) + s) % R_MOD
            matrix.append((delta * selector % R_MOD, f"a_poly_{m}"))
            matrix.append(((-delta * selector % R_MOD * b_term) % R_MOD, f"b_poly_{m}"))
        matrix.append(((-v_k_gamma) % R_MOD, "h_2"))
        lcs["matrix_sumcheck"] = matrix
        points = {"rowcheck_zerocheck": ("alpha", alpha), "g_1": ("beta", beta), "lineval_sumcheck": ("beta", beta),
                  "g_a": ("gamma", gamma), "g_b": ("gamma", gamma), "g_c": ("gamma", gamma), "matrix_sumcheck": ("gamma", gamma)}
        order = sorted(lcs)
        return [(k, lcs[k]) for k in order], [(k, points[k]) for k in order]

    mask_poly = None

    def set_mask_poly(self, h_1_mask_rand, g_1_mask_rand):
        """calculate_mask_poly (first.rs:102-127) for the hiding mode: rand(degree 3)·v_H on the variable domain plus rand(degree 5)
        with a zero constant term; the random coefficients (ints) are arguments.  The mask is a first-round oracle (committed without a
        degree or hiding bound, first.rs:54-56) and enters h_1 / g_1 in the third round."""
        assert len(h_1_mask_rand) == 4 and len(g_1_mask_rand) == 6
        n = self.circuit.variable_domain.size
        mask = [0] * (n + 4)
        for i, c in enumerate(h_1_mask_rand):
            mask[n + i] = (mask[n + i] + c) % R_MOD
            mask[i] = (mask[i] - c) % R_MOD
        for i, c in enumerate(g_1_mask_rand):
            if i:
                mask[i] = (mask[i] + c) % R_MOD
        dev = self.z[0].device
        idx = sorted(set(range(6)) | set(range(n, n + 4)))              # the (at most ten) non-zero coefficients
        vals = np.array([_mont(mask[i]) for i in idx], dtype=np.uint64).reshape(-1, 4)
        self.mask_poly = _zeros(n + 4, dev)
        self.mask_poly[torch.tensor(idx, dtype=torch.int64, device=dev)] = torch.from_numpy(vals.view(np.int64)).to(dev)
        return self.mask_poly

    # ---- round 4: matrix sumchecks (fourth.rs:151-245) ----
    def fourth_round(self, alpha: int, beta: int):
        c = self.circuit
        Rd, V = c.constraint_domain, c.variable_domain
        v_rc = (pow(alpha, Rd.size, R_MOD) - 1) * (pow(beta, V.size, R_MOD) - 1) % R_MOD
        rc_size = Rd.size * V.size % R_MOD
        consts = v_rc * pow(Rd.size, -1, R_MOD) % R_MOD * pow(V.size, -1, R_MOD) % R_MOD
        self.gs, self.lhs, self.fourth_sums, self.a_polys, self.b_polys = [], [], [], [], []
        for arith in c.ariths:
            K = arith.domain
            a_poly = K.ifft_in_place(_scale(arith.row_col_val, v_rc).clone())
            # (α − r)(β − c) = (r − α)(c − β): the common factor of b's evaluations and of the denominators
            ra = device.fr_vec_op(arith.row, _mont(alpha), device.FR_SUB)
            cb = device.fr_vec_op(arith.col, _mont(beta), device.FR_SUB)
            prod = device.fr_vec_op(ra, cb, device.FR_MUL)
            b_poly = K.ifft_in_place(_scale(prod, rc_size).clone())                          # |R||C|(αβ − βr − αc + rc)
            device.fr_batch_inversion_and_mul(prod, _mont(consts))                            # fields/src/lib.rs:78-129
            f = K.ifft_in_place(device.fr_vec_op(prod, arith.row_col_val, device.FR_MUL))
            h = _sub(a_poly, polymul(b_poly, f))
            lhs, _ = apply_randomized_selector(h, 1, c.max_non_zero_domain, K, False)
            self.gs.append(f[1:].contiguous()); self.lhs.append(lhs)
            self.fourth_sums.append(_fr_mont_to_int(f[0].cpu().numpy().view(np.uint64)))
            self.a_polys.append(a_poly); self.b_polys.append(b_poly)
        return self.gs

    # ---- round 5 (fifth.rs:41-67) ----
    def fifth_round(self, deltas):
        h_2 = _zeros(0, self.z[0].device)
        for d, lhs in zip(deltas, self.lhs):
            h_2 = _add(h_2, _scale(lhs, d % R_MOD))
        self.h_2 = h_2
        return h_2

    def oracles(self) -> dict:
        """every polynomial the prover commits to, by round (varuna.rs:387-506)"""
        first = list(self.w_polys) + ([self.mask_poly] if self.mask_poly is not None else [])
        return {1: first, 2: [self.h_0], 3: [self.g_1, self.h_1], 4: list(self.gs), 5: [self.h_2]}


def test_circuit_csr(a: int, b: int, mul_depth: int, num_constraints: int, num_variables: int, dev):
    """TestCircuit (data_structures/test_circuit.rs:42-139) laid out directly as CSR matrices and one assignment, with the public
    variables padded to a power of two: every A, B, C row has a single unit entry.  Returns (Circuit, assignment tensor)."""
    num_public = 1 + mul_depth
    padded = 1 << (num_public - 1).bit_length() if num_public > 1 else 1
    num_private = num_variables - num_public
    nv = padded + num_private
    va, vb = padded + 0, padded + 1                                   # private variables a, b
    mul = [1 + i for i in range(mul_depth)]                            # public mul_var i
    mul_constraints = mul_depth - 1
    plain = num_constraints - mul_constraints
    a_cols = np.array([va] * plain + [mul[i] for i in range(mul_constraints)], dtype=np.int64)
    b_cols = np.full(num_constraints, vb, dtype=np.int64)
    c_cols = np.array([mul[0]] * plain + [mul[i + 1] for i in range(mul_constraints)], dtype=np.int64)
    row_ptr = np.arange(num_constraints + 1, dtype=np.int64)
    ones = np.tile(_mont(1), (num_constraints, 1))
    mats = [Matrix(row_ptr, cols, ones, dev) for cols in (a_cols, b_cols, c_cols)]
    circuit = Circuit(mats[0], mats[1], mats[2], padded, nv)
    z = np.zeros((nv, 4), dtype=np.uint64)
    z[0] = _mont(1)
    v = a % R_MOD
    for i in range(mul_depth):
        v = v * b % R_MOD
        z[1 + i] = _mont(v)
    z[padded:] = _mont(a)
    z[vb] = _mont(b)
    return circuit, torch.from_numpy(z.view(np.int64)).to(dev)


# ---- circuit setup and the key certificate (varuna.rs:72-134, 236-331) ----
@dataclass
class VerifyingKey:
    """CircuitVerifyingKey: the circuit info, the twelve index commitments (uint64 [12, 18], normalised projective) sorted by label,
    and the circuit id"""
    circuit_info: CircuitInfo
    circuit_commitments: np.ndarray
    id: bytes


@dataclass
class ProvingKey:
    """CircuitProvingKey: the verifying key, the indexed circuit and the committer key trimmed for it"""
    circuit_verifying_key: VerifyingKey
    circuit: Circuit
    committer_key: CommitterKey


def batch_circuit_setup(pp_powers_of_beta_g: torch.Tensor, pp_powers_of_beta_times_gamma_g: torch.Tensor, circuits: list,
                        hiding: bool = False) -> list:
    """Varuna::batch_circuit_setup (varuna.rs:72-134) → [(ProvingKey, VerifyingKey)] per circuit.  Each circuit's committer key is
    trimmed as the reference does (max_degree, hiding bound 1, the AHP's degree bounds); the index polynomials of ALL circuits are
    then committed in one device pass (the reference commits circuit by circuit: the commitments are the same).  The commitments
    are not blinded.  An SRS with fewer powers than a circuit's max_degree raises ValueError."""
    srs_degree = pp_powers_of_beta_g.shape[0] - 1
    keyed, bases, polys = [], [], []
    for c in circuits:
        info = c.info()
        max_degree = info.max_degree(hiding)
        if max_degree > srs_degree:
            raise ValueError(f"the universal SRS supports degree {srs_degree}, the circuit needs {max_degree}")
        ck = CommitterKey.trim(pp_powers_of_beta_g, pp_powers_of_beta_times_gamma_g, max_degree, (), 1, info.degree_bounds())
        labeled = c.interpolate_matrix_evals()
        keyed.append((c, info, ck, labeled))
        bases += [ck.powers_of_beta_g] * len(labeled)
        polys += [p.polynomial for p in labeled]
    comms = device.sonic_commit_batch(bases, polys)
    out = []
    for i, (c, info, ck, labeled) in enumerate(keyed):
        rows = comms[12 * i: 12 * i + 12]
        order = sorted(range(12), key=lambda j: labeled[j].label)
        vk = VerifyingKey(info, rows[order].copy(), c.id())
        out.append((ProvingKey(vk, c, ck), vk))
    return out


def circuit_setup(pp_powers_of_beta_g: torch.Tensor, pp_powers_of_beta_times_gamma_g: torch.Tensor, circuit: Circuit, hiding: bool = False):
    """Varuna::circuit_setup (varuna.rs:223-233) → (ProvingKey, VerifyingKey)"""
    return batch_circuit_setup(pp_powers_of_beta_g, pp_powers_of_beta_times_gamma_g, [circuit], hiding)[0]


def _certificate_challenges(challenges, count: int):
    """the squeezed values of the certificate sponge: the last is the point, the combiners are 1 and the others (varuna.rs:245-251)"""
    challenges = [int(x) % R_MOD for x in challenges]
    if len(challenges) != count:
        raise ValueError(f"{count} challenges expected, one per index commitment")
    return challenges[-1], [1] + challenges[:-1]


def prove_vk(pk: ProvingKey, vk: VerifyingKey, challenges, opening_challenges):
    """Varuna::prove_vk (varuna.rs:236-276): opens Σ c_i·p_i over the sorted labels at the point (LC `circuit_check`) with
    SonicKZG10.open_combinations.  `challenges`: the twelve squeezed values; `opening_challenges`: what open_combinations squeezes
    (one combiner, then the discarded randomizer).  → the BatchLCProof's [(w, random_v)]."""
    point, combiners = _certificate_challenges(challenges, len(vk.circuit_commitments))
    labeled = pk.circuit.interpolate_matrix_evals()
    lc = [("circuit_check", list(zip(combiners, sorted(p.label for p in labeled))))]
    query_set = [("circuit_check", ("challenge", point))]
    return SonicKZG10.open_combinations(pk.committer_key, lc, labeled, [Randomness() for _ in labeled], query_set, iter(opening_challenges))


def evaluate_index_polynomials(circuit: Circuit, point: int, combiners):
    """AHPForR1CS::evaluate_index_polynomials (ahp/indexer/indexer.rs:232-260): the twelve evaluations at `point` through the
    Lagrange coefficients of each K_M, summed in one device pass without interpolating → (("circuit_check", [(combiner, label)]),
    Σ combiner·evaluation) over the sorted labels."""
    combiners = [int(x) % R_MOD for x in combiners]
    if len(combiners) != 12:
        raise ValueError("one combiner per index polynomial")
    dev = circuit.a.vals.device
    lagrange = [K.evaluate_all_lagrange_coefficients(point, dev) for K in circuit.non_zero_domains]
    sums = device.index_arithmetize(circuit._csr(), [K.size for K in circuit.non_zero_domains], circuit.num_variables,
                                    circuit.num_public, lagrange)
    evals = dict(zip(index_polynomial_labels(circuit.id()), (_fr_mont_to_int(v) for v in sums.reshape(12, 4))))
    terms, total = [], 0
    for comb, label in zip(combiners, sorted(evals)):
        terms.append((comb, label))
        total += comb * evals[label]
    return ("circuit_check", terms), total % R_MOD


def verify_vk_evaluation(circuit: Circuit, vk: VerifyingKey, challenges):
    """The half of Varuna::verify_vk (varuna.rs:280-311) that precedes check_combinations: the re-indexed circuit must have the key's
    info and id (else ValueError, SNARKError::CircuitNotFound), then → (lc, point, evaluation)."""
    if circuit.info() != vk.circuit_info or circuit.id() != vk.id:
        raise ValueError("CircuitNotFound: the circuit does not match the verifying key")
    point, combiners = _certificate_challenges(challenges, len(vk.circuit_commitments))
    lc, evaluation = evaluate_index_polynomials(circuit, point, combiners)
    return lc, point, evaluation
