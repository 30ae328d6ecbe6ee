"""GPU: Varuna circuit setup on the device (snarkvm_b200/varuna.py batch_circuit_setup, prove_vk, evaluate_index_polynomials and the
fused index arithmetization kernel behind them) against the CPU oracle (tests/setup_oracle.py, pinned in
tests/test_varuna_setup_oracle.py), and the link between the existing device prover and the new key: the prover's a_M / b_M commit
to the homomorphic combinations of the verifying key's commitments that the verifier forms (ahp/ahp.rs:430-444)."""
import random
from dataclasses import astuple

import numpy as np
import pytest

from oracle import bls12_377 as py
from oracle import sonic as osonic
from oracle import varuna as ov

import setup_oracle as so

pytestmark = pytest.mark.gpu
R = py.R_MOD
BETA, GAMMA = 0x1234567890ABCDEF1234567890ABCDEF % R, 0xFEDCBA0987654321FEDCBA % R
G = np.frombuffer(py.affine_bytes(py.G1_GENERATOR), dtype=np.uint8)


def _device_circuit(circuit: ov.Circuit):
    from snarkvm_b200 import varuna as dv
    mats = []
    for m in (circuit.a, circuit.b, circuit.c):
        row_ptr = np.concatenate([[0], np.cumsum([len(r) for r in m])]).astype(np.int64)
        cols = np.array([c for r in m for _, c in r], dtype=np.int64)
        vals = np.array([dv._mont(v) for r in m for v, _ in r], dtype=np.uint64).reshape(-1, 4)
        mats.append(dv.Matrix(row_ptr, cols, vals, "cuda"))
    return dv.Circuit(mats[0], mats[1], mats[2], circuit.num_public, circuit.num_variables)


def _ints(t):
    from snarkvm_b200 import device
    h = device.fr_from_mont(t.contiguous()).cpu().numpy().view(np.uint64).reshape(-1, 4)
    return [sum(int(v) << (64 * i) for i, v in enumerate(row)) for row in h]


def _one_entry_cs():
    """one constraint, one entry per matrix: every K has one element (nnz = 1, |X| = 1)"""
    cs = ov.ConstraintSystem()
    x = cs.alloc(5)
    cs.enforce([(3, x)], [(1, ("pub", 0))], [(3, x)])
    return cs


CASES = {
    "circuit_0": (lambda: ov.test_circuit(2, 4, 3, 7, 7), False),
    "test_circuit": (lambda: ov.test_circuit(3, 5, 2, 300, 200), False),
    "test_circuit_no_padding": (lambda: ov.test_circuit(3, 5, 2, 256, 100), False),      # nnz = |K| = 256 for A, B and C
    "random_r1cs": (lambda: so.random_r1cs(7, n_pub=4, n_prv=90, n_con=150), False),
    "nnz_1": (_one_entry_cs, False),
    "circuit_0_hiding": (lambda: ov.test_circuit(2, 4, 3, 7, 7), True),
    "random_r1cs_hiding": (lambda: so.random_r1cs(8, n_pub=8, n_prv=40, n_con=60), True),
}


def _pair(name):
    make, hiding = CASES[name]
    o = so.index(make(), hiding)
    return o, _device_circuit(o), hiding


@pytest.mark.parametrize("name", sorted(CASES))
def test_materialise_mode_equals_the_oracle(name):
    o, d, _ = _pair(name)
    if name == "test_circuit_no_padding":
        assert [m.nnz for m in (d.a, d.b, d.c)] == [K.size for K in d.non_zero_domains] == [256] * 3
    if name == "nnz_1":
        assert [K.size for K in d.non_zero_domains] == [1, 1, 1]
    for arith, want in zip(d.ariths, so.evaluations(o)):
        for got, w in zip(arith.vectors(), want):
            assert _ints(got) == w, name


@pytest.mark.parametrize("name", ["circuit_0", "test_circuit", "random_r1cs", "random_r1cs_hiding"])
def test_evaluate_mode_equals_the_oracle(name):
    from snarkvm_b200 import varuna as dv
    o, d, _ = _pair(name)
    rng = random.Random(len(name))
    points = [rng.randrange(R), rng.randrange(R), o.max_non_zero_domain.elements()[3 % o.max_non_zero_domain.size]]   # the last on K
    for z in points:
        combiners = [1] + [rng.randrange(R) for _ in range(11)]
        assert dv.evaluate_index_polynomials(d, z, combiners) == so.evaluate_index_polynomials(o, z, combiners), (name, z)


@pytest.fixture(scope="module")
def srs():
    from snarkvm_b200 import sonic_pc
    D = 1023
    powers, gamma = sonic_pc.synthetic_srs(D, BETA, GAMMA)
    return powers, gamma, powers.cpu().numpy(), gamma.cpu().numpy()


def _check_setup(vk, o, hiding, hp, hg):
    _, _, (info, comms, cid) = so.circuit_setup(hp, hg, o, hiding)
    assert astuple(vk.circuit_info) == info and vk.id == cid
    assert vk.circuit_commitments.shape == (12, 18) and (vk.circuit_commitments == comms).all()


@pytest.mark.parametrize("name", ["circuit_0", "test_circuit", "random_r1cs", "circuit_0_hiding", "random_r1cs_hiding"])
def test_circuit_setup_equals_the_oracle(oracle_cpu, srs, name):
    from snarkvm_b200 import varuna as dv
    powers, gamma, hp, hg = srs
    o, d, hiding = _pair(name)
    pk, vk = dv.circuit_setup(powers, gamma, d, hiding)
    _check_setup(vk, o, hiding, hp, hg)
    assert pk.circuit_verifying_key is vk and pk.circuit is d
    assert pk.committer_key.enforced_degree_bounds == sorted(set(vk.circuit_info.degree_bounds()))


def test_batch_of_three_circuits_in_one_pass_equals_three_setups(oracle_cpu, srs):
    from snarkvm_b200 import varuna as dv
    powers, gamma, hp, hg = srs
    pairs = [_pair(n) for n in ("circuit_0", "test_circuit", "random_r1cs")]
    batch = dv.batch_circuit_setup(powers, gamma, [d for _, d, _ in pairs])
    assert len(batch) == 3
    for (o, d, _), (pk, vk) in zip(pairs, batch):
        _, single = dv.circuit_setup(powers, gamma, d)
        assert (single.circuit_commitments == vk.circuit_commitments).all() and single.id == vk.id
        _check_setup(vk, o, False, hp, hg)


def test_closed_form_at_2_16_non_zeros(oracle_cpu):
    """TestCircuit with 2^16 constraints (2^16 entries in each matrix): C = p(β)·G for one index commitment"""
    from snarkvm_b200 import device, varuna as dv
    from snarkvm_b200.sonic_pc import synthetic_srs
    d, _ = dv.test_circuit_csr(3, 5, 2, 1 << 16, 1 << 10, "cuda")
    assert [m.nnz for m in (d.a, d.b, d.c)] == [1 << 16] * 3
    powers, gamma = synthetic_srs(d.info().max_degree(False), BETA, GAMMA)
    pk, vk = dv.circuit_setup(powers, gamma, d)
    polys = {p.label: p.polynomial for p in d.interpolate_matrix_evals()}
    labels = sorted(polys)
    for i in (labels.index(dv.index_polynomial_labels(vk.id)[3]), labels.index(dv.index_polynomial_labels(vk.id)[9])):
        pv = py.fr_from_mont(py.from_limbs(device.poly_evaluate(polys[labels[i]], dv._mont(BETA))))
        assert (vk.circuit_commitments[i] == oracle_cpu.g1_mul(G, osonic._scalars([pv])[0])).all(), labels[i]


def _affine(proj):
    return np.frombuffer(py.affine_bytes(py.projective_from_bytes(np.asarray(proj, dtype=np.uint64).tobytes())), dtype=np.uint8)


def _lin(cpu, points, scalars):
    return cpu.msm(np.stack([_affine(p) for p in points]), osonic._scalars([s % R for s in scalars]), cpu.BATCHED)


@pytest.mark.parametrize("name", ["test_circuit", "random_r1cs_hiding"])
def test_prove_vk_equals_the_oracle_and_holds_in_the_exponent(oracle_cpu, srs, name):
    from snarkvm_b200 import varuna as dv
    powers, gamma, hp, hg = srs
    o, d, hiding = _pair(name)
    pk, vk = dv.circuit_setup(powers, gamma, d, hiding)
    rng = random.Random(3)
    challenges = [rng.randrange(R) for _ in range(12)]
    opening = [rng.randrange(1 << 128), rng.randrange(1 << 128)]
    (w, rv), = dv.prove_vk(pk, vk, challenges, opening)
    ck, polys, _ = so.circuit_setup(hp, hg, o, hiding)
    (ww, wrv), = so.prove_vk(ck, polys, challenges, opening)
    assert rv is None and wrv is None and (w == ww).all()
    # the verifier's half: re-index, evaluate through the Lagrange coefficients, check in the exponent
    lc, z, v = dv.verify_vk_evaluation(d, vk, challenges)
    assert z == challenges[-1] and [c for c, _ in lc[1]] == [1] + challenges[:11]
    xi = opening[0]
    lhs = _lin(oracle_cpu, list(vk.circuit_commitments) + [oracle_cpu.g1_mul(G, osonic._scalars([1])[0])],
               [xi * c for c, _ in lc[1]] + [-xi * v])
    assert (lhs == _lin(oracle_cpu, [w], [BETA - z])).all()


@pytest.mark.parametrize("name", ["test_circuit", "random_r1cs"])
def test_prover_a_and_b_commit_to_the_verifiers_combinations(oracle_cpu, srs, name):
    """SonicKZG10.commit of the device prover's a_poly_M / b_poly_M equals v_rc·C_row_col_val and
    rc·(αβ·G − α·C_col − β·C_row + C_row_col) formed from the verifying key"""
    import torch
    from snarkvm_b200 import varuna as dv
    from snarkvm_b200.sonic_pc import LabeledPolynomial, SonicKZG10
    powers, gamma, _, _ = srs
    make, _ = CASES[name]
    o, d, _ = _pair(name)
    pk, vk = dv.circuit_setup(powers, gamma, d)
    cs = make()
    ov.pad_input_for_indexer_and_prover(cs)
    z = torch.from_numpy(np.array([dv._mont(v) for v in cs.public + cs.private], dtype=np.uint64).reshape(-1, 4).view(np.int64)).cuda()
    rng = random.Random(9)
    alpha, beta = rng.randrange(R), rng.randrange(R)
    p = dv.Prover(d, [z])
    p.fourth_round(alpha, beta)
    Rd, V = d.constraint_domain, d.variable_domain
    v_rc = (pow(alpha, Rd.size, R) - 1) * (pow(beta, V.size, R) - 1) % R
    rc = Rd.size * V.size % R
    comm = dict(zip(sorted(dv.index_polynomial_labels(vk.id)), vk.circuit_commitments))
    got, _ = SonicKZG10.commit(pk.committer_key, [LabeledPolynomial(f"{k}_{m}", poly) for m, a, b in zip("abc", p.a_polys, p.b_polys)
                                                  for k, poly in (("a", a), ("b", b))])
    g = oracle_cpu.g1_mul(G, osonic._scalars([1])[0])
    for i, m in enumerate("abc"):
        c = lambda k: comm[f"circuit_{vk.id.hex()}_{k}_{m}"]                                    # noqa: E731
        assert (got[2 * i] == _lin(oracle_cpu, [c("row_col_val")], [v_rc])).all(), m
        want_b = _lin(oracle_cpu, [g, c("col"), c("row"), c("row_col")], [rc * alpha * beta, -rc * alpha, -rc * beta, rc])
        assert (got[2 * i + 1] == want_b).all(), m


def test_undersized_srs_and_mismatched_circuit_raise(srs):
    from snarkvm_b200 import varuna as dv
    from snarkvm_b200.sonic_pc import synthetic_srs
    _, d, _ = _pair("test_circuit")
    small = synthetic_srs(d.info().max_degree(False) - 1, BETA, GAMMA)
    with pytest.raises(ValueError):
        dv.circuit_setup(*small, d)
    powers, gamma, _, _ = srs
    _, vk = dv.circuit_setup(powers, gamma, d)
    rng = random.Random(4)
    challenges = [rng.randrange(R) for _ in range(12)]
    dv.verify_vk_evaluation(d, vk, challenges)
    cs = ov.test_circuit(3, 5, 2, 300, 200)
    cs.c[7] = [(2, cs.c[7][0][1])]                                                                  # one entry changed: same info, other id
    other = _device_circuit(so.index(cs))
    assert other.info() == d.info() and other.id() != d.id()
    with pytest.raises(ValueError):
        dv.verify_vk_evaluation(other, vk, challenges)
    with pytest.raises(ValueError):
        dv.verify_vk_evaluation(_device_circuit(so.index(ov.test_circuit(3, 5, 2, 301, 200))), vk, challenges)


def test_malformed_matrices_are_rejected():
    """the wrapper rejects shapes, the kernel reports a column ≥ num_variables and a bad row_ptr as an error code"""
    import torch
    from snarkvm_b200 import CudaError, device
    _, d, _ = _pair("circuit_0")
    mats = d._csr()
    ks = [K.size for K in d.non_zero_domains]
    with pytest.raises(ValueError):
        device.index_arithmetize(mats, [ks[0] // 2, ks[1], ks[2]], d.num_variables, d.num_public)         # nnz > |K_A|
    with pytest.raises(ValueError):
        device.index_arithmetize(mats, ks, d.num_variables, d.variable_domain.size)                       # |X| = |C|
    bad_cols = mats[1][1].clone()
    bad_cols[2] = d.num_variables
    with pytest.raises(CudaError):
        device.index_arithmetize([mats[0], (mats[1][0], bad_cols, mats[1][2]), mats[2]], ks, d.num_variables, d.num_public)
    bad_ptr = mats[2][0].clone()
    bad_ptr[-1] += 1
    with pytest.raises(CudaError):
        device.index_arithmetize([mats[0], mats[1], (bad_ptr, mats[2][1], mats[2][2])], ks, d.num_variables, d.num_public)
    torch.cuda.synchronize()
    want = so.evaluations(so.index(ov.test_circuit(2, 4, 3, 7, 7)))
    assert _ints(device.index_arithmetize(mats, ks, d.num_variables, d.num_public)[0][3]) == want[0][3]          # still usable afterwards
