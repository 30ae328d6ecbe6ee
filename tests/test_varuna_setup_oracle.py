"""CPU: the setup and certificate oracle (tests/setup_oracle.py) pinned BY DEFINITION — the reference holds no vector for index
polynomials, their commitments, certificates or circuit ids — on a universal setup whose trapdoor β the test knows
(powers_of_beta_g[i] = β^i·G), so every group element has a closed form in the scalar field:
    index commitment      C = (Σ_κ e(κ)·L_κ(β))·G, from the evaluations and the Lagrange coefficients at β, not through the iFFT
    verifier's a, b       a_M = v_rc·row_col_val_M,  b_M = rc·(αβ − α·col_M − β·row_M + row_col_M)   (ahp/ahp.rs:430-444)
    certificate           ξ·(Σ c_i·C_i − v·G) = (β − z)·W, v from the verifier's evaluate_index_polynomials"""
import copy
import random

import numpy as np
import pytest

from oracle import bls12_377 as py
from oracle import sonic
from oracle import varuna as ov

import setup_oracle as so

R = py.R_MOD
BETA, GAMMA = 0x1234567890ABCDEF1234567890ABCDEF % R, 0xFEDCBA0987654321FEDCBA % R
D = 70                                                    # max_degree of the universal parameters
G = np.frombuffer(py.affine_bytes(py.G1_GENERATOR), dtype=np.uint8)


@pytest.fixture(scope="module")
def srs(oracle_cpu):
    def pts(scalars):
        out = np.zeros((len(scalars), 104), dtype=np.uint8)
        for i, s in enumerate(scalars):
            out[i] = _affine(oracle_cpu.g1_mul(G, sonic._scalars([s])[0]))
        return out
    return pts([pow(BETA, i, R) for i in range(D + 1)]), pts([GAMMA * pow(BETA, i, R) % R for i in range(D + 2)])


def _affine(proj):
    return np.frombuffer(py.affine_bytes(py.projective_from_bytes(np.asarray(proj, dtype=np.uint64).tobytes())), dtype=np.uint8)


def _g(cpu, k):
    return cpu.g1_mul(G, sonic._scalars([k % R])[0])


def _lin(cpu, points, scalars):
    """Σ s_i·P_i of projective images"""
    return cpu.msm(np.stack([_affine(p) for p in points]), sonic._scalars([s % R for s in scalars]), cpu.BATCHED)


CASES = [("circuit_0", lambda: ov.test_circuit(2, 4, 3, 7, 7), False),                 # the reference's circuit_0
         ("test_circuit", lambda: ov.test_circuit(3, 5, 2, 20, 13), False),             # R, C and K domains all differ
         ("random_r1cs", lambda: so.random_r1cs(1), False),
         ("circuit_0_hiding", lambda: ov.test_circuit(2, 4, 3, 7, 7), True),
         ("random_r1cs_hiding", lambda: so.random_r1cs(2, n_prv=24), True)]


def _circuits():
    """(name, oracle circuit, hiding) for every case"""
    return [(name, so.index(make(), hiding), hiding) for name, make, hiding in CASES]


@pytest.mark.parametrize("case", range(5))
def test_index_commitments_are_the_lagrange_forms(oracle_cpu, srs, case):
    name, circuit, hiding = _circuits()[case]
    ck, polys, (info, comms, cid) = so.circuit_setup(*srs, circuit, hiding)
    evals = dict(zip(so.labels(cid), [v for vecs in so.evaluations(circuit) for v in vecs]))
    doms = dict(zip(so.labels(cid), [a.domain for a in circuit.ariths for _ in range(4)]))
    assert sorted(polys) == sorted(evals) and len(comms) == 12
    for i, label in enumerate(sorted(evals)):
        lag = doms[label].evaluate_all_lagrange_coefficients(BETA)
        assert (comms[i] == _g(oracle_cpu, sum(e * l for e, l in zip(evals[label], lag)))).all(), (name, label)
        assert doms[label].fft(polys[label]) == evals[label], (name, label)                   # the polynomials interpolate K
        assert len(polys[label]) <= doms[label].size


def test_circuit_0_k_domain_is_the_reference_one(golden):
    circuit = _circuits()[0][1]
    assert circuit.max_non_zero_domain.elements() == [int(x) for x in golden["varuna_circuit_0_domain"]["K"]]


@pytest.mark.parametrize("case", [0, 2, 4])
def test_verifier_rebuilds_a_and_b_from_the_index_polynomials(case):
    """the prover's a_poly_M / b_poly_M (fourth round) equal the verifier's combinations of index polynomials, coefficient by
    coefficient (cmp_non_zero_domains, ahp.rs:430-444)"""
    name, make, hiding = CASES[case]
    circuit, cs = so.index(make(), hiding), make()
    if hiding:                                                  # the prover's instance carries the randomizing variables too
        so.add_randomizing_variables(cs)
    rng = random.Random(case)
    alpha, beta = rng.randrange(R), rng.randrange(R)
    prover = ov.Prover(circuit, [cs])
    prover.fourth_round(alpha, beta)
    polys = so.index_polynomials(circuit)
    cid = so.circuit_id(circuit).hex()
    Rd, V = circuit.constraint_domain, circuit.variable_domain
    v_rc = Rd.evaluate_vanishing_polynomial(alpha) * V.evaluate_vanishing_polynomial(beta) % R
    rc = Rd.size * V.size % R
    for m, a_poly, b_poly in zip("abc", prover.a_polys, prover.b_polys):
        p = lambda k: polys[f"circuit_{cid}_{k}_{m}"]                                                # noqa: E731
        assert a_poly == ov.poly_scale(p("row_col_val"), v_rc), (name, m)
        b = ov.poly_add([alpha * beta % R], ov.poly_add(ov.poly_scale(p("col"), -alpha % R), ov.poly_scale(p("row"), -beta % R)))
        assert b_poly == ov.poly_scale(ov.poly_add(b, p("row_col")), rc), (name, m)


@pytest.mark.parametrize("case", [1, 3])
def test_certificate_holds_in_the_exponent(oracle_cpu, srs, case):
    name, circuit, hiding = _circuits()[case]
    ck, polys, (info, comms, cid) = so.circuit_setup(*srs, circuit, hiding)
    rng = random.Random(10 + case)
    challenges = [rng.randrange(R) for _ in range(12)]
    xi = rng.randrange(1 << 128)
    (w, rv), = so.prove_vk(ck, polys, challenges, [xi, rng.randrange(1 << 128)])
    assert rv is None
    z, combiners = so.certificate_challenges(challenges)
    lc, v = so.evaluate_index_polynomials(circuit, z, combiners)
    assert lc[0] == "circuit_check" and [l for _, l in lc[1]] == sorted(polys) and [c for c, _ in lc[1]] == combiners
    assert v == sum(c * sonic.poly_eval(polys[l], z) for c, l in lc[1]) % R                     # Lagrange route = interpolated route

    def holds(comms, v):
        lhs = _lin(oracle_cpu, list(comms) + [_g(oracle_cpu, 1)], [xi * c for c in combiners] + [-xi * v])
        return (lhs == _lin(oracle_cpu, [w], [BETA - z])).all()
    assert holds(comms, v)
    assert not holds(comms, v + 1)
    bad = comms.copy()
    bad[5] = _g(oracle_cpu, 7)
    assert not holds(bad, v)


def test_circuit_id_and_info():
    a = so.index(ov.test_circuit(2, 4, 3, 7, 7))
    assert so.circuit_id(a) == so.circuit_id(so.index(ov.test_circuit(9, 9, 3, 7, 7)))          # the witness is not part of the index
    assert so.info(a) == (4, 7, 7, 7, 7, 7)
    cs = ov.test_circuit(2, 4, 3, 7, 7)
    cs.b[3] = [(2, cs.b[3][0][1])]                                                              # one coefficient 1 → 2
    assert so.info(so.index(cs)) == so.info(a) and so.circuit_id(so.index(cs)) != so.circuit_id(a)
    h = so.index(ov.test_circuit(2, 4, 3, 7, 7), hiding=True)
    assert so.info(h) == (4, 7 + 3, 7 + 1, 8, 8, 8)                                               # three randomizing variables, one constraint
    assert so.circuit_id(h) != so.circuit_id(a)
    assert so.labels(so.circuit_id(a))[3] == f"circuit_{so.circuit_id(a).hex()}_row_col_val_a"


def test_undersized_srs_raises(srs):
    circuit = so.index(ov.test_circuit(2, 4, 3, 7, 7))
    d = so.max_degree(circuit, False)
    with pytest.raises(ValueError):
        so.circuit_setup(srs[0][:d], srs[1], circuit)


def test_device_side_host_helpers_match_the_oracle():
    """CircuitInfo's serialisation, max_degree, degree bounds and labels of snarkvm_b200.varuna (host code) against the oracle"""
    from snarkvm_b200 import varuna as dv
    for name, circuit, hiding in _circuits():
        info = dv.CircuitInfo(*so.info(circuit))
        assert info.to_bytes() == b"".join(int(v).to_bytes(8, "little") for v in so.info(circuit))
        assert info.max_degree(hiding) == so.max_degree(circuit, hiding), name
        assert info.degree_bounds() == so.degree_bounds(circuit), name
        cid = so.circuit_id(circuit)
        assert dv.index_polynomial_labels(cid) == so.labels(cid)
    with pytest.raises(ValueError):
        dv.CircuitInfo(1, 2, 1, 1, 2, 2).degree_bounds()                                       # |K_A| = 1 has no degree bound
