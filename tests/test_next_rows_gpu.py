"""GPU parity for the rows after the hot path (SURVEY §8 f1–f4): hiding / batched / Lagrange KZG commitments, the group FFT behind
UniversalParams::lagrange_basis, batch_inversion_and_mul, divide_by_vanishing_poly, DensePolynomial::evaluate — each against the
oracle's restatement of the reference CPU code, bit-exact."""
import os

import numpy as np
import pytest

from oracle import bls12_377 as py

from helpers import affine_array, fr_ints_to_mont_array, mont_array_to_fr_ints, oracle_bases, random_canonical_fr, random_fr_mont

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))


def _dev(x):
    import torch
    if x.dtype == np.uint64:
        x = x.view(np.int64)
    return torch.from_numpy(x.copy()).cuda()


def _host_u64(t):
    return t.cpu().numpy().view(np.uint64)


@pytest.mark.parametrize("lg", [0, 1, 2, 3, 6, 7, 8, 9, 12])
def test_g1_ifft_vs_oracle(oracle_cpu, lg):
    from snarkvm_b200 import device
    n = 1 << lg
    bases = oracle_bases(oracle_cpu, max(n, 4), seed=20 + lg)[:n].copy()
    if n >= 8:
        bases[5, 96] = 1                                       # an ∞ input
        bases[6] = bases[2]                                    # a repeated point (sum doubles, difference cancels)
    got = device.g1_ntt(_dev(bases), inverse=True).cpu().numpy()
    assert (got == oracle_cpu.g1_ifft(bases)).all()
    # forward transform undoes it (fft ∘ ifft = id on the group elements); ∞ comes back in the canonical (0, 1, ∞) image
    back = device.g1_ntt(_dev(got), inverse=False).cpu().numpy()
    want = bases.copy()
    if n >= 8:
        want[5] = affine_array([None])[0]
    assert (back == want).all()


def test_lagrange_basis_real_srs_and_commit_lagrange(oracle_cpu):
    """lagrange_basis of the real powers-of-beta (kzg10/data_structures.rs:68-72); then commit_lagrange(evals) == commit(ifft(evals)):
    the two commitment keys commit to the same polynomial (kzg10/mod.rs:98-206)."""
    from snarkvm_b200.algorithms import KZG10, EvaluationDomain, UniversalParams
    n = 512                                                    # every point of the committed excerpt of the mainnet file
    blob = open(os.path.join(HERE, "golden", "powers_of_beta_15_first512.usrs"), "rb").read()
    powers = affine_array(py.parse_usrs_points(blob, n))
    dpowers = _dev(powers)
    domain = EvaluationDomain.new(n)
    basis = UniversalParams(dpowers).lagrange_basis(domain)
    assert (basis.cpu().numpy().reshape(n, 104) == oracle_cpu.g1_ifft(powers)).all()
    evals = random_fr_mont(n, seed=77)
    c_lagrange = KZG10.commit_lagrange(basis, _dev(evals))
    coeffs = oracle_cpu.ntt(evals, oracle_cpu.INVERSE)
    assert (c_lagrange == oracle_cpu.msm(powers, oracle_cpu.fr_from_mont(coeffs), 0)).all()
    assert (c_lagrange == KZG10.commit(dpowers, _dev(coeffs))).all()
    with pytest.raises(ValueError):
        KZG10.commit_lagrange(basis, _dev(evals[:100]))       # next_power_of_two(100) != 256


def _powers_of_tau_usrs(cpu, n, tau):
    """A .usrs file in the layout of the mainnet powers-of-beta files (u64-LE count, then per point x and y as 48-byte LE canonical
    integers, flag bits clear) holding P_i = τ^i·G for i < n, built with the oracle's scalar multiplication."""
    g = np.frombuffer(py.affine_bytes(py.G1_GENERATOR), dtype=np.uint8)
    proj = np.empty((n, 18), dtype=np.uint64)
    k = 1
    for i in range(n):
        proj[i] = cpu.g1_mul(g, np.array(py.to_limbs(k, 4), dtype=np.uint64))    # normalised: Z = 1, X and Y affine
        k = k * tau % py.R_MOD
    xy = np.concatenate([cpu.fq_from_mont(proj[:, 0:6]), cpu.fq_from_mont(proj[:, 6:12])], axis=1)
    return n.to_bytes(8, "little") + xy.tobytes()


def test_lagrange_basis_of_a_2_15_point_srs(oracle_cpu):
    """UniversalParams::lagrange_basis (kzg10/data_structures.rs:68-72) at the size of the mainnet powers-of-beta-15 file, on a
    seeded powers-of-τ SRS in the same file layout (the real points are covered by the 512-point excerpt above): decoded on the
    device, every basis point equal to the oracle's group iFFT, Σ_i L_i(τ)·G = powers[0] = G, and a few basis points equal to
    their closed form L_i(τ)·G = (τ^n − 1)·ω^i / (n·(τ − ω^i))·G."""
    import torch
    from snarkvm_b200 import device
    n = 1 << 15
    tau = py.from_limbs(random_canonical_fr(1, seed=15)[0])
    blob = _powers_of_tau_usrs(oracle_cpu, n, tau)
    powers = affine_array(py.parse_usrs_points(blob, n))
    raw = torch.from_numpy(np.frombuffer(blob[8:], dtype=np.uint8).copy()).cuda()
    decoded, invalid = device.srs_decode(raw)
    assert invalid == 0 and (decoded.cpu().numpy() == powers).all()
    basis = device.lagrange_basis(decoded).cpu().numpy().reshape(n, 104)
    assert (basis == oracle_cpu.g1_ifft(powers)).all()
    w = py.fr_root_of_unity(n)
    for i in (0, 1, 12345, n - 1):
        wi = pow(w, i, py.R_MOD)
        li = (pow(tau, n, py.R_MOD) - 1) * wi * pow(n * (tau - wi), -1, py.R_MOD) % py.R_MOD
        assert basis[i].tobytes() == py.affine_bytes(py.g1_mul(py.G1_GENERATOR, li)), i
    ones = torch.from_numpy(np.tile(py.to_limbs(1, 4), (n, 1)).astype(np.uint64).view(np.int64)).cuda()
    total = device.msm(torch.from_numpy(basis).cuda(), ones)
    assert total.tobytes() == py.projective_bytes_normalised(py.G1_GENERATOR)


def test_kzg_commit_hiding_and_batch(oracle_cpu):
    from snarkvm_b200.algorithms import KZG10
    from snarkvm_b200 import device
    n = 1 << 12
    powers = device.generate_bases(n, seed=41)
    gamma = device.generate_bases(8, seed=42)
    hp, hg = powers.cpu().numpy(), gamma.cpu().numpy()
    coeffs = random_fr_mont(n, seed=1)
    coeffs[:37] = 0                                            # leading zeros (skip_leading_zeros_and_convert_to_bigints, mod.rs:455-467)
    blind = random_fr_mont(3, seed=2)                          # hiding_bound = Some(1) ⇒ degree-2 blinding polynomial
    got = KZG10.commit(powers, _dev(coeffs), gamma, _dev(blind))
    plain = oracle_cpu.msm(hp, oracle_cpu.fr_from_mont(coeffs), 0)
    rnd = oracle_cpu.msm(hg, oracle_cpu.fr_from_mont(blind), 0)
    assert (got == oracle_cpu.g1_add(plain, rnd)).all()
    with pytest.raises(ValueError):
        KZG10.commit(powers, _dev(coeffs), gamma, _dev(random_fr_mont(9, seed=3)))
    polys = [random_fr_mont(m, seed=10 + i) for i, m in enumerate((n, 1000, 1, n - 1))]
    batch = KZG10.batch_commit(powers, [_dev(p) for p in polys])
    for row, p in zip(batch, polys):
        assert (row == oracle_cpu.msm(hp, oracle_cpu.fr_from_mont(p), 0)).all()
    assert KZG10.batch_commit(powers, []).shape == (0, 18)


@pytest.mark.parametrize("n", [1, 7, 8, 9, 1000, 100003])
def test_batch_inversion_and_mul(oracle_cpu, n):
    from snarkvm_b200.algorithms import batch_inversion_and_mul
    v = random_fr_mont(n, seed=n)
    v[::5] = 0
    coeff = random_fr_mont(1, seed=99)[0]
    got = _host_u64(batch_inversion_and_mul(_dev(v), coeff))
    assert (got == oracle_cpu.fr_batch_inversion_and_mul(v, coeff)).all()
    one = fr_ints_to_mont_array([1])[0]
    back = _host_u64(batch_inversion_and_mul(_dev(got), one))   # (c/v)^{-1} = v/c
    cinv = oracle_cpu.fr_batch_inversion_and_mul(coeff.reshape(1, 4), one)[0]
    want = np.array([oracle_cpu.fr_mul(x, cinv) for x in v[:16]])
    assert (back[:16] == want).all()


@pytest.mark.parametrize("m,n", [(5, 8), (8, 8), (9, 8), (40, 8), (4096, 1024), (3 * 4096 - 5, 4096), (100, 4), (1, 1),
                                 (70000, 4), (65 * 8, 8), (65 * 8 + 3, 8), (100001, 1), (50000, 64)])   # many rows per column: the blocked suffix scan
def test_divide_by_vanishing_poly_and_evaluate(oracle_cpu, m, n):
    from snarkvm_b200.algorithms import DensePolynomial, EvaluationDomain
    p = random_fr_mont(m, seed=m + n)
    if m == 40:
        p[-3:] = 0
    poly = DensePolynomial(_dev(p))
    q, r = poly.divide_by_vanishing_poly(EvaluationDomain.new(n))
    wq, wr = oracle_cpu.poly_divide_by_vanishing(p, n)
    assert (_host_u64(q.coeffs).reshape(-1, 4) == wq).all() and (_host_u64(r.coeffs).reshape(-1, 4) == wr).all()
    for seed in (1, 2):
        z = random_fr_mont(1, seed=seed)[0]
        assert (poly.evaluate(z) == oracle_cpu.poly_evaluate(p, z)).all()
    zero = np.zeros(4, dtype=np.uint64)
    assert (poly.evaluate(zero) == p[0]).all()                 # dense.rs:101-102


@pytest.mark.parametrize("n", [8, 1024])
def test_evaluations_type(oracle_cpu, n):
    """Evaluations (fft/evaluations.rs): interpolate ∘ evaluate_over_domain = id, evaluate(point) equals the interpolated polynomial at
    the point (through evaluate_all_lagrange_coefficients, also for a point INSIDE the domain), elementwise * + − / against big ints,
    unequal domains and zero divisors are rejected"""
    from snarkvm_b200.algorithms import DensePolynomial, EvaluationDomain, Evaluations
    dom = EvaluationDomain.new(n)
    a, b = random_fr_mont(n, seed=n + 1), random_fr_mont(n, seed=n + 2)
    ea, eb = Evaluations.from_vec_and_domain(_dev(a), dom), Evaluations.from_vec_and_domain(_dev(b), dom)
    ai, bi = mont_array_to_fr_ints(a), mont_array_to_fr_ints(b)
    for got, op in ((ea * eb, lambda x, y: x * y), (ea + eb, lambda x, y: x + y), (ea - eb, lambda x, y: x - y),
                    (ea / eb, lambda x, y: x * pow(y, -1, py.R_MOD))):
        assert mont_array_to_fr_ints(_host_u64(got.evaluations)) == [op(x, y) % py.R_MOD for x, y in zip(ai, bi)]
    poly = ea.interpolate_by_ref()
    assert (_host_u64(poly.coeffs) == oracle_cpu.ntt(a, oracle_cpu.INVERSE)).all()
    assert (_host_u64(poly.evaluate_over_domain(dom)) == a).all()
    z = random_fr_mont(1, seed=99)[0]
    assert (ea.evaluate(z) == oracle_cpu.poly_evaluate(_host_u64(poly.coeffs).reshape(-1, 4), z)).all()
    w5 = fr_ints_to_mont_array([pow(py.fr_root_of_unity(n), 5, py.R_MOD)])[0]            # a domain element: the indicator branch
    assert (ea.evaluate(w5) == a[5]).all()
    short = Evaluations.from_vec_and_domain(_dev(a[: n // 2 + 1]), dom)                    # resize: zero-padded
    assert (_host_u64(short.evaluations)[n // 2 + 1:] == 0).all() and short.evaluations.shape[0] == n
    with pytest.raises(ValueError):
        ea * Evaluations.from_vec_and_domain(_dev(a), EvaluationDomain.new(2 * n))
    zb = b.copy(); zb[3] = 0
    with pytest.raises(ZeroDivisionError):
        ea / Evaluations.from_vec_and_domain(_dev(zb), dom)


def test_evaluate_large_and_over_domain(oracle_cpu):
    from snarkvm_b200.algorithms import DensePolynomial, EvaluationDomain
    m = (1 << 18) + 12345
    p = random_fr_mont(m, seed=5)
    z = random_fr_mont(1, seed=6)[0]
    assert (DensePolynomial(_dev(p)).evaluate(z) == oracle_cpu.poly_evaluate(p, z)).all()
    small = random_fr_mont(300, seed=7)
    ev = DensePolynomial(_dev(small)).evaluate_over_domain(EvaluationDomain.new(512))
    padded = np.zeros((512, 4), dtype=np.uint64); padded[:300] = small
    assert (_host_u64(ev).reshape(-1, 4) == oracle_cpu.ntt(padded, oracle_cpu.FORWARD)).all()
    # degree ≥ domain size (polynomial/mod.rs:277-288): per-chunk FFTs added up, restated here with the oracle
    big = random_fr_mont(1300, seed=8)
    ev = DensePolynomial(_dev(big)).evaluate_over_domain(EvaluationDomain.new(512))
    acc = np.zeros((512, 4), dtype=np.uint64)
    for c0 in range(0, 1300, 512):
        chunk = np.zeros((512, 4), dtype=np.uint64); chunk[: min(512, 1300 - c0)] = big[c0:c0 + 512]
        e = oracle_cpu.ntt(chunk, oracle_cpu.FORWARD)
        acc = np.array([oracle_cpu.fr_add(a, b) for a, b in zip(acc, e)])
    assert (_host_u64(ev).reshape(-1, 4) == acc).all()


@pytest.mark.parametrize("m", [1, 2, 3, 64, 65, 66, 4097, 64 * 256 + 1, 64 * 256 * 3 + 17, (1 << 20) + 5])
def test_divide_by_linear_vs_oracle(oracle_cpu, m):
    """compute_witness_polynomial (kzg10/mod.rs:220-241): chunk boundaries of the three-pass recurrence, zero / one / random points"""
    from snarkvm_b200 import device
    p = random_fr_mont(m, seed=m)
    if m > 3:
        p[-2:] = 0                                             # true degree below the slot count
    dp = _dev(p)
    points = [np.zeros(4, dtype=np.uint64), fr_ints_to_mont_array([1])[0], random_fr_mont(1, seed=3)[0]]
    for z in points[: 3 if m < (1 << 20) else 1] + points[2:]:
        got = _host_u64(device.poly_divide_by_linear(dp, z)).reshape(-1, 4)
        assert (got == oracle_cpu.poly_divide_by_linear(p, z)).all()


def test_kzg_open(oracle_cpu):
    """KZG10::open (kzg10/mod.rs:220-321), hiding and not: w = commit(p / (x − z)) [+ commit_γ(blinding / (x − z))], random_v = blinding(z)"""
    from snarkvm_b200.algorithms import KZG10
    from snarkvm_b200 import device
    n = 1 << 11
    powers = device.generate_bases(n, seed=51)
    gamma = device.generate_bases(4, seed=52)
    hp, hg = powers.cpu().numpy(), gamma.cpu().numpy()
    poly = random_fr_mont(n, seed=4)
    blind = random_fr_mont(3, seed=5)
    z = random_fr_mont(1, seed=6)[0]
    wq = oracle_cpu.poly_divide_by_linear(poly, z)
    bq = oracle_cpu.poly_divide_by_linear(blind, z)
    w_plain = oracle_cpu.msm(hp, oracle_cpu.fr_from_mont(wq), 0)
    w, v = KZG10.open(powers, _dev(poly), z)
    assert v is None and (w == w_plain).all()
    w, v = KZG10.open(powers, _dev(poly), z, gamma, _dev(blind))
    assert (w == oracle_cpu.g1_add(w_plain, oracle_cpu.msm(hg, oracle_cpu.fr_from_mont(bq), 0))).all()
    assert (v == oracle_cpu.poly_evaluate(blind, z)).all()


def test_sparse_matvec_vs_oracle(oracle_cpu):
    """z_A = A·z as the Varuna prover computes it (round_functions/mod.rs:130-189), CSR on the device"""
    import torch
    from snarkvm_b200 import CudaError, device
    rng = np.random.default_rng(3)
    nrows, npub, nprv = 5000, 17, 4000
    counts = rng.integers(0, 9, size=nrows)
    counts[7] = 0
    # hot rows (a variable every constraint uses, transposed): they leave the thread-per-row kernel and are cut into segments
    counts[100], counts[101], counts[2000], counts[2001], counts[4999] = 256, 257, 2048, 2049, 30000
    row_ptr = np.concatenate([[0], np.cumsum(counts)]).astype(np.uint32)
    nnz = int(row_ptr[-1])
    cols = rng.integers(0, npub + nprv, size=nnz).astype(np.uint32)
    vals = random_fr_mont(nnz, seed=1)
    vals[::3] = fr_ints_to_mont_array([1])[0]
    pub, prv = random_fr_mont(npub, seed=2), random_fr_mont(nprv, seed=3)
    x = np.concatenate([pub, prv])
    got = device.sparse_matvec(torch.from_numpy(row_ptr.view(np.int32)).cuda(), torch.from_numpy(cols.view(np.int32)).cuda(), _dev(vals), _dev(x))
    assert (_host_u64(got).reshape(-1, 4) == oracle_cpu.sparse_matvec(row_ptr, cols, vals, pub, prv)).all()
    for where in (5, int(row_ptr[4999]) + 12345):                   # an out-of-range column in a short row / inside a long row's segment
        bad = cols.copy(); bad[where] = npub + nprv
        with pytest.raises(CudaError):
            device.sparse_matvec(torch.from_numpy(row_ptr.view(np.int32)).cuda(), torch.from_numpy(bad.view(np.int32)).cuda(), _dev(vals), _dev(x))


def test_fr_vec_ops_and_domain_elements(oracle_cpu):
    from snarkvm_b200 import device
    n = 1000
    a, b = random_fr_mont(n, seed=1), random_fr_mont(n, seed=2)
    s = random_fr_mont(1, seed=3)[0]
    for op, f in ((device.FR_ADD, oracle_cpu.fr_add), (device.FR_SUB, oracle_cpu.fr_sub), (device.FR_MUL, oracle_cpu.fr_mul)):
        got = _host_u64(device.fr_vec_op(_dev(a), _dev(b), op)).reshape(-1, 4)
        assert (got == np.array([f(x, y) for x, y in zip(a, b)])).all(), op
        got = _host_u64(device.fr_vec_op(_dev(a), s, op)).reshape(-1, 4)
        assert (got == np.array([f(x, s) for x in a])).all(), op
    da = _dev(a)
    device.fr_vec_op(da, da, device.FR_MUL, out=da)           # aliasing: a ← a·a
    assert (_host_u64(da).reshape(-1, 4) == np.array([oracle_cpu.fr_mul(x, x) for x in a])).all()
    for lg in (0, 1, 3, 10):
        # elements = FFT of the polynomial X (the reference's domain KAT, circuit_0/domain/*.txt, is the lg = 3 case)
        m = 1 << lg
        x = np.zeros((m, 4), dtype=np.uint64)
        if m > 1:
            x[1] = fr_ints_to_mont_array([1])[0]
            want = oracle_cpu.ntt(x, oracle_cpu.FORWARD)
        else:
            want = fr_ints_to_mont_array([1])
        assert (_host_u64(device.domain_elements(lg)).reshape(-1, 4) == want).all(), lg


def test_kzg_open_lagrange(oracle_cpu):
    """KZG10::open_lagrange (kzg10/mod.rs:272-301) against the oracle pieces, and against open() on the coefficient form:
    both prove the same evaluation, so the witness commitments are the same group element."""
    from snarkvm_b200.algorithms import KZG10, EvaluationDomain, UniversalParams
    from snarkvm_b200 import device
    n = 128
    powers = device.generate_bases(n, seed=61)
    domain = EvaluationDomain.new(n)
    basis = UniversalParams(powers).lagrange_basis(domain)
    coeffs = random_fr_mont(n, seed=1)
    evals = oracle_cpu.ntt(coeffs, oracle_cpu.FORWARD)
    z = random_fr_mont(1, seed=2)[0]
    y = oracle_cpu.poly_evaluate(coeffs, z)
    w, v = KZG10.open_lagrange(basis, domain, _dev(evals), z, y)
    assert v is None
    # oracle: (eval_i − y)·(ω^i − z)^{-1} committed against the oracle's own Lagrange basis
    x = np.zeros((n, 4), dtype=np.uint64); x[1] = fr_ints_to_mont_array([1])[0]
    elems = oracle_cpu.ntt(x, oracle_cpu.FORWARD)
    div = np.array([oracle_cpu.fr_sub(e, z) for e in elems])
    div = oracle_cpu.fr_batch_inversion_and_mul(div, fr_ints_to_mont_array([1])[0])
    wit = np.array([oracle_cpu.fr_mul(d, oracle_cpu.fr_sub(e, y)) for d, e in zip(div, evals)])
    hbasis = oracle_cpu.g1_ifft(powers.cpu().numpy())
    assert (w == oracle_cpu.msm(hbasis, oracle_cpu.fr_from_mont(wit), 0)).all()
    w2, _ = KZG10.open(powers, _dev(coeffs), z)
    assert (w == w2).all()
    with pytest.raises(ValueError):
        KZG10.open_lagrange(basis, domain, _dev(evals), elems[5], y)      # a point of the domain
    with pytest.raises(ValueError):
        KZG10.open_lagrange(basis, domain, _dev(evals[:100]), z, y)
