"""Phases of Varuna circuit setup (snarkvm_b200/varuna.py batch_circuit_setup + prove_vk) on the TestCircuit at 2^16, 2^18 and
2^20 constraints, each phase timed on its own with a device synchronise after it (median of --reps runs, one warm-up run first):

    arith      the fused index arithmetization kernel (device.index_arithmetize, materialise mode) for A, B, C
    arith_old  the host-expansion path it replaced: np.repeat of the row indices and reindex_by_subdomain on the host, upload of the
               per-entry index arrays, torch gathers from the |R| and |C| element tables, two fr_vec_op launches per matrix
    evaluate   the verifier's evaluate_index_polynomials (Lagrange coefficients of A, B, C's domains + the evaluate mode)
    id         Circuit.id: the copy of the matrix values to the host and the Blake2s hash over the serialised matrices
    interp     interpolate_matrix_evals: twelve iFFTs over K
    commit1    the twelve index polynomials committed in ONE sonic_commit_batch pass
    commit12   the same twelve as twelve separate kzg_commit calls
    setup      batch_circuit_setup end to end (trim, circuit id, interpolation, one commitment pass); the id is recomputed every run
    cert       prove_vk (interpolation + open_combinations)

`arith` is the arithmetization alone: building a Circuit also constructs the transposes, which still expand the CSR arrays on the
host.  The arithmetization outputs of the two paths are compared byte for byte at every size, and one commitment per size is
checked in closed form, C = p(β)·G with p(β) from poly_evaluate, on a generated SRS with a known trapdoor.  Prints the card name and power
limit (nvidia-smi query flags).  Usage: python tools/time_circuit_setup.py [--reps 5] [--lgs 16,18,20]"""
import argparse
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from snarkvm_b200 import device, varuna as dv  # noqa: E402
from snarkvm_b200.sonic_pc import synthetic_srs  # noqa: E402

R = dv.R_MOD
BETA, GAMMA = 0x1234567890ABCDEF1234567890ABCDEF % R, 0xFEDCBA0987654321FEDCBA % R


def arith_host_expansion(c: dv.Circuit) -> list:
    """the arithmetization as Circuit.__init__ computed it before the fused kernel (kept here as the baseline)"""
    dev = c.a.vals.device
    r_el = device.domain_elements(c.constraint_domain.log_size_of_group, dev)
    c_el = device.domain_elements(c.variable_domain.log_size_of_group, dev)
    one = torch.from_numpy(dv._mont(1).view(np.int64)).to(dev)
    out = []
    for m, K in zip((c.a, c.b, c.c), c.non_zero_domains):
        entry_rows = np.repeat(np.arange(m.nrows, dtype=np.int64), np.diff(m.row_ptr_h))
        entry_cols = dv.reindex_by_subdomain(c.variable_domain.size, c.input_domain.size, m.cols_h)
        row, col, rc = one.repeat(K.size, 1), one.repeat(K.size, 1), one.repeat(K.size, 1)
        rcv = torch.zeros((K.size, 4), dtype=torch.int64, device=dev)
        row[: m.nnz] = r_el[torch.from_numpy(entry_rows).to(dev)]
        col[: m.nnz] = c_el[torch.from_numpy(entry_cols).to(dev)]
        rc[: m.nnz] = device.fr_vec_op(row[: m.nnz].contiguous(), col[: m.nnz].contiguous(), device.FR_MUL)
        rcv[: m.nnz] = device.fr_vec_op(m.vals, rc[: m.nnz].contiguous(), device.FR_MUL)
        out.append((row, col, rc, rcv))
    return out


def timed(fn, reps):
    fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        torch.cuda.synchronize()
        ts.append((time.perf_counter() - t0) * 1e3)
    return statistics.median(ts), min(ts), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--lgs", default="16,18,20")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_circuit_setup needs a CUDA device")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    print(f"# device: {torch.cuda.get_device_name(0)} | nvidia-smi name, power.limit, clocks.max.sm: {smi[0] if smi else 'n/a'}")
    print(f"# median (min) of {args.reps} runs after one warm-up, ms; each phase ends in a device synchronise")
    lgs = [int(x) for x in args.lgs.split(",")]
    n_max = 1 << max(lgs)
    powers, gamma = synthetic_srs(2 * n_max - 2, BETA, GAMMA)
    for lg in lgs:
        n = 1 << lg
        circuit, _ = dv.test_circuit_csr(3, 5, 2, n, n - 10, "cuda")             # |R| = |C| = |K| = n
        info = circuit.info()
        ks = [K.size for K in circuit.non_zero_domains]
        rows = {}
        rows["arith"] = timed(lambda: device.index_arithmetize(circuit._csr(), ks, circuit.num_variables, circuit.num_public), args.reps)
        rows["arith_old"] = timed(lambda: arith_host_expansion(circuit), args.reps)
        same = all(torch.equal(x, y) for a, b in zip(rows["arith"][2], rows["arith_old"][2]) for x, y in zip(a, b))
        rows["evaluate"] = timed(lambda: dv.evaluate_index_polynomials(circuit, 12345, list(range(1, 13))), args.reps)
        rows["id"] = timed(lambda: (setattr(circuit, "_id", None), circuit.id()), args.reps)
        rows["interp"] = timed(circuit.interpolate_matrix_evals, args.reps)
        polys = [p.polynomial for p in rows["interp"][2]]
        base = powers[: info.max_degree(False) + 1]
        rows["commit1"] = timed(lambda: device.sonic_commit_batch([base] * 12, polys), args.reps)
        rows["commit12"] = timed(lambda: np.stack([device.kzg_commit(base, p) for p in polys]), args.reps)
        same_commit = bool((rows["commit1"][2] == rows["commit12"][2]).all())
        rows["setup"] = timed(lambda: (setattr(circuit, "_id", None), dv.batch_circuit_setup(powers, gamma, [circuit]))[1], args.reps)
        pk, vk = rows["setup"][2][0]
        challenges = list(range(2, 14))
        rows["cert"] = timed(lambda: dv.prove_vk(pk, vk, challenges, [7, 11]), args.reps)
        # closed form of the row_col_val_a commitment
        label = dv.index_polynomial_labels(vk.id)[3]
        poly = dict((p.label, p.polynomial) for p in rows["interp"][2])[label]
        pv = torch.from_numpy(device.poly_evaluate(poly, dv._mont(BETA)).view(np.int64).reshape(1, 4)).cuda()
        closed = bool((vk.circuit_commitments[sorted(dv.index_polynomial_labels(vk.id)).index(label)]
                       == device.msm(powers[:1], device.fr_from_mont(pv))).all())           # powers[0] = G
        print(f"2^{lg} constraints, nnz A/B/C = {info.num_non_zero_a}/{info.num_non_zero_b}/{info.num_non_zero_c}, "
              f"max_degree {info.max_degree(False)}: " + "  ".join(f"{k} {v[0]:.2f} ({v[1]:.2f})" for k, v in rows.items()))
        print(f"    arith speed-up x{rows['arith_old'][0] / rows['arith'][0]:.1f}, one pass vs twelve commits "
              f"x{rows['commit12'][0] / rows['commit1'][0]:.2f}; arith outputs identical: {same}; commitments identical: {same_commit}; "
              f"closed form C = p(beta)*G: {closed}", flush=True)
        if not (same and same_commit and closed):
            raise SystemExit("mismatch")


if __name__ == "__main__":
    main()
