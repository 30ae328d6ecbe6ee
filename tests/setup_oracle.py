"""TEST INFRASTRUCTURE ONLY — CPU restatement (Python big integers) of Varuna's circuit setup and key certificate, on top of the
prover oracle (oracle/varuna.py) and the SonicKZG10 oracle (oracle/sonic.py):

    ahp/matrices.rs:64-82             add_randomizing_variables           → index(cs, hiding=True)
    ahp/matrices.rs:102-190           MatrixEvals.row_col                 → row_col()
    ahp/indexer/indexer.rs:169-176    CircuitInfo                         → info()
    ahp/indexer/circuit.rs:109-121    Circuit::hash                       → circuit_id()
    ahp/indexer/indexer.rs:104-122    index_polynomial_labels             → labels()
    ahp/indexer/circuit.rs:142-148    interpolate_matrix_evals            → index_polynomials()
    ahp/ahp.rs:85-121                 max_degree / get_degree_bounds      → max_degree() / degree_bounds()
    varuna.rs:72-134                  batch_circuit_setup                 → circuit_setup()
    varuna.rs:236-276                 prove_vk                            → prove_vk()
    ahp/indexer/indexer.rs:232-260    evaluate_index_polynomials          → evaluate_index_polynomials() (Lagrange route)

The reference holds no vector for any of these, so tests/test_varuna_setup_oracle.py pins them by definition on a universal setup
with a known trapdoor."""
from __future__ import annotations

import copy
import hashlib
import struct

import numpy as np

from oracle import sonic
from oracle import varuna as ov

R = ov.R


def add_randomizing_variables(cs: ov.ConstraintSystem) -> None:
    """ahp/matrices.rs:64-82: three private variables (assigned one) and the constraint zk_0 · zk_1 = zk_2, in place"""
    zk = [cs.alloc(1) for _ in range(3)]
    cs.enforce([(1, zk[0])], [(1, zk[1])], [(1, zk[2])])


def index(cs: ov.ConstraintSystem, hiding: bool = False) -> ov.Circuit:
    """index_helper on a copy of `cs`: in the hiding mode the randomizing variables and their constraint come first, before the
    public variables are padded (indexer.rs:137-141); the default is the non-hiding index of oracle/varuna.py's Circuit"""
    cs = copy.deepcopy(cs)
    if hiding:
        add_randomizing_variables(cs)
    return ov.Circuit(cs)


def row_col(arith: ov.MatrixEvals) -> list:
    """row·col on K; the padding is 1·1 = 1 (matrices.rs:170-181)"""
    return [r * c % R for r, c in zip(arith.row, arith.col)]


def evaluations(circuit: ov.Circuit) -> list:
    """[(row, col, row_col, row_col_val)] for A, B, C"""
    return [(a.row, a.col, row_col(a), a.row_col_val) for a in circuit.ariths]


def info(circuit: ov.Circuit) -> tuple:
    nnz = [sum(len(r) for r in m) for m in (circuit.a, circuit.b, circuit.c)]
    return (circuit.num_public, circuit.num_variables, circuit.num_constraints, *nnz)


def circuit_id(circuit: ov.Circuit) -> bytes:
    h = hashlib.blake2s(digest_size=32)
    h.update(b"".join(struct.pack("<Q", v) for v in info(circuit)))
    for m in (circuit.a, circuit.b, circuit.c):
        h.update(struct.pack("<Q", len(m)))
        for row in m:
            h.update(struct.pack("<Q", len(row)))
            for val, col in row:
                h.update(val.to_bytes(32, "little") + struct.pack("<Q", col))
    return h.digest()


def labels(cid: bytes) -> list:
    return [f"circuit_{cid.hex()}_{p}_{m}" for m in "abc" for p in ("row", "col", "row_col", "row_col_val")]


def index_polynomials(circuit: ov.Circuit) -> dict:
    """label → coefficients (trimmed) of the twelve index polynomials"""
    polys = []
    for arith, vecs in zip(circuit.ariths, evaluations(circuit)):
        polys += [arith.domain.ifft(v) for v in vecs]
    return dict(zip(labels(circuit_id(circuit)), polys))


def max_degree(circuit: ov.Circuit, hiding: bool) -> int:
    zk = 1 if hiding else 0
    r, v = circuit.constraint_domain.size, circuit.variable_domain.size
    k = circuit.max_non_zero_domain.size
    return max(2 * r + 2 * zk - 2, 2 * v + 2 * zk - 2, v + 3 if hiding else 0, v, r, k - 1)


def degree_bounds(circuit: ov.Circuit) -> list:
    return [circuit.variable_domain.size - 2] + [d.size - 2 for d in circuit.non_zero_domains]


def circuit_setup(pp_powers, pp_gamma_powers, circuit: ov.Circuit, hiding: bool = False):
    """→ (committer key, label → coefficients, (info, commitments uint64 [12, 18] sorted by label, id))"""
    d = max_degree(circuit, hiding)
    if d > pp_powers.shape[0] - 1:
        raise ValueError("the universal SRS is too small for the circuit")
    ck = sonic.CommitterKey(pp_powers, pp_gamma_powers, d, (), 1, degree_bounds(circuit))
    polys = index_polynomials(circuit)
    names = sorted(polys)
    comms, _ = sonic.commit(ck, [(k, polys[k], None, None, False) for k in names])
    return ck, polys, (info(circuit), np.stack(comms), circuit_id(circuit))


def certificate_challenges(challenges):
    challenges = [c % R for c in challenges]
    return challenges[-1], [1] + challenges[:-1]


def prove_vk(ck, polys: dict, challenges, opening_challenges):
    point, combiners = certificate_challenges(challenges)
    lc = [("circuit_check", list(zip(combiners, sorted(polys))))]
    return sonic.open_combinations(ck, lc, {k: (p, None, None) for k, p in polys.items()}, [("circuit_check", ("challenge", point))],
                                   iter(opening_challenges))


def evaluate_index_polynomials(circuit: ov.Circuit, point: int, combiners):
    """the verifier's route: Σ_κ L_κ(point)·e(κ) per vector, no interpolation → (("circuit_check", terms), Σ combiner·evaluation)"""
    evals = []
    for arith, vecs in zip(circuit.ariths, evaluations(circuit)):
        lag = arith.domain.evaluate_all_lagrange_coefficients(point % R)
        evals += [sum(l * e for l, e in zip(lag, v)) % R for v in vecs]
    by_label = dict(zip(labels(circuit_id(circuit)), evals))
    combiners = [c % R for c in combiners]
    assert len(combiners) == len(by_label)
    terms = list(zip(combiners, sorted(by_label)))
    return ("circuit_check", terms), sum(c * by_label[k] for c, k in terms) % R


def random_r1cs(seed: int, n_pub: int = 4, n_prv: int = 27, n_con: int = 24) -> ov.ConstraintSystem:
    """A satisfied R1CS with general coefficients: rows of 1–4 entries, every tenth A row empty (and its C row with it), rows over
    public variables only, and repeated columns that the indexer merges (into_matrix_helper)."""
    import random
    rng = random.Random(seed)
    cs = ov.ConstraintSystem()
    for _ in range(n_pub - 1):
        cs.alloc_input(rng.randrange(R))
    for _ in range(n_prv):
        cs.alloc(rng.randrange(1, R))
    var = lambda: ("pub", rng.randrange(n_pub)) if rng.random() < 0.2 else ("priv", rng.randrange(n_prv))     # noqa: E731
    val = lambda v: cs.public[v[1]] if v[0] == "pub" else cs.private[v[1]]                                      # noqa: E731
    for i in range(n_con):
        if i % 10 == 0:
            la = []
        elif i % 10 == 1:
            la = [(rng.randrange(1, R), ("pub", rng.randrange(n_pub))) for _ in range(2)]
        else:
            la = [(rng.randrange(1, R), var()) for _ in range(rng.randrange(1, 5))]
        if i % 10 == 2:
            la.append((rng.randrange(1, R), la[0][1]))
        lb = [(rng.randrange(1, R), var()) for _ in range(rng.randrange(1, 4))]
        ab = sum(c * val(v) for c, v in la) % R * (sum(c * val(v) for c, v in lb) % R) % R
        j = ("priv", rng.randrange(n_prv))
        cs.enforce(la, lb, [(ab * pow(val(j), -1, R) % R, j)] if ab else [])
    return cs
