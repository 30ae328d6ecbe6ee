"""Regenerates tests/golden/*.json|*.bin from the reference tree (run in the build container only;
/root/reference does not exist on the GPU box).  Only DATA is extracted — constants, known-answer
vectors and SRS points — never source code.

    python tests/golden/make_golden.py [/root/reference]
"""
import json
import os
import re
import sys

REF = sys.argv[1] if len(sys.argv) > 1 else "/root/reference"
OUT = os.path.dirname(os.path.abspath(__file__))


def read(p):
    with open(os.path.join(REF, p)) as f:
        return f.read()


def bigints(src, name):
    """All `BigInteger([...])` / `BigInteger::new([...])` limb lists following `const NAME`."""
    m = re.search(r"const\s+" + name + r"\b[^=]*=\s*(.*?);\s*\n", src, re.S)
    assert m, name
    body = m.group(1)
    out = []
    for lm in re.finditer(r"\[([^\[\]]*?)\]", body, re.S):
        toks = [t.strip() for t in lm.group(1).replace("\n", " ").split(",") if t.strip()]
        if not toks or not all(re.fullmatch(r"(0x[0-9a-fA-F_]+|[0-9_]+)(u64)?", t) for t in toks):
            continue
        out.append([int(t.replace("u64", "").replace("_", ""), 0) for t in toks])
    return out


def scalar_const(src, name):
    m = re.search(r"const\s+" + name + r"\s*:\s*u\d+\s*=\s*([0-9a-fx_]+)", src)
    return int(m.group(1).replace("_", ""), 0)


golden = {}
fr = read("curves/src/bls12_377/fr.rs")
golden["fr"] = {
    "source": "curves/src/bls12_377/fr.rs:60-192",
    "MODULUS": bigints(fr, "MODULUS")[0], "R": bigints(fr, "R")[0], "R2": bigints(fr, "R2")[0],
    "INV": scalar_const(fr, "INV"), "GENERATOR": bigints(fr, "GENERATOR")[0],
    "TWO_ADICITY": scalar_const(fr, "TWO_ADICITY"),
    "TWO_ADIC_ROOT_OF_UNITY": bigints(fr, "TWO_ADIC_ROOT_OF_UNITY")[0],
    "POWERS_OF_ROOTS_OF_UNITY": bigints(fr, "POWERS_OF_ROOTS_OF_UNITY"),
    "T": bigints(fr, "T")[0],
}
fq = read("curves/src/bls12_377/fq.rs")
golden["fq"] = {
    "source": "curves/src/bls12_377/fq.rs:30-176 ; KAT curves/src/bls12_377/tests.rs:460-476 (GENERATOR^T == TWO_ADIC_ROOT)",
    "MODULUS": bigints(fq, "MODULUS")[0], "R": bigints(fq, "R")[0], "R2": bigints(fq, "R2")[0],
    "INV": scalar_const(fq, "INV"), "GENERATOR": bigints(fq, "GENERATOR")[0],
    "TWO_ADICITY": scalar_const(fq, "TWO_ADICITY"),
    "TWO_ADIC_ROOT_OF_UNITY": bigints(fq, "TWO_ADIC_ROOT_OF_UNITY")[0],
    "POWERS_OF_ROOTS_OF_UNITY": bigints(fq, "POWERS_OF_ROOTS_OF_UNITY"),
    "T": bigints(fq, "T")[0],
}
g1 = read("curves/src/bls12_377/g1.rs")
gx = re.search(r"pub const G1_GENERATOR_X.*?new\(\[(.*?)\]\)", g1, re.S).group(1)
gy = re.search(r"pub const G1_GENERATOR_Y.*?new\(\[(.*?)\]\)", g1, re.S).group(1)
golden["g1"] = {
    "source": "curves/src/bls12_377/g1.rs:219-253 (Montgomery limbs) and the decimal comments above them",
    "GENERATOR_X_MONT": [int(t) for t in gx.replace("\n", " ").split(",") if t.strip()],
    "GENERATOR_Y_MONT": [int(t) for t in gy.replace("\n", " ").split(",") if t.strip()],
    "GENERATOR_X_DEC": re.search(r"G1_GENERATOR_X =\s*\n///\s*(\d+)", g1).group(1),
    "GENERATOR_Y_DEC": re.search(r"G1_GENERATOR_Y =\s*\n///\s*(\d+)", g1).group(1),
}
g2src = read("curves/src/bls12_377/g2.rs")
fq2src = read("curves/src/bls12_377/fq2.rs")
def _new_limbs(src, name):
    body = re.search(r"pub const " + name + r"\b.*?new\(\[(.*?)\]\)", src, re.S).group(1)
    return [int(t) for t in body.replace("\n", " ").split(",") if t.strip()]
golden["g2"] = {
    "source": "curves/src/bls12_377/g2.rs:38-107,228-282 (WEIERSTRASS_B, COFACTOR, generator; Montgomery limbs) and "
              "curves/src/bls12_377/fq2.rs:29-65 (NONRESIDUE); KAT curves/src/bls12_377/tests.rs:673-678 (generator on curve, order r)",
    "GENERATOR_X_C0_MONT": _new_limbs(g2src, "G2_GENERATOR_X_C0"), "GENERATOR_X_C1_MONT": _new_limbs(g2src, "G2_GENERATOR_X_C1"),
    "GENERATOR_Y_C0_MONT": _new_limbs(g2src, "G2_GENERATOR_Y_C0"), "GENERATOR_Y_C1_MONT": _new_limbs(g2src, "G2_GENERATOR_Y_C1"),
    "WEIERSTRASS_B_MONT": bigints(g2src, "WEIERSTRASS_B"),
    "COFACTOR": bigints(g2src, "COFACTOR")[0],
    "NONRESIDUE_MONT": bigints(fq2src, "NONRESIDUE")[0],
}
dom = {}
for name in ("R", "C", "K"):
    txt = read(f"algorithms/src/snark/varuna/resources/circuit_0/domain/{name}.txt")
    dom[name] = [s.strip() for s in txt.strip().strip("[]").split(",")]
golden["varuna_circuit_0_domain"] = {
    "source": "algorithms/src/snark/varuna/resources/circuit_0/domain/{R,C,K}.txt (test_varuna_with_prover_test_vectors, "
              "algorithms/src/snark/varuna/tests.rs:533-809): elements ω^i of the size-8/4/… domains, decimal",
    **dom,
}
# Varuna prover known-answer vectors (the only reference-held vectors that pin iFFT / FFT / polymul / division OUTPUTS)
base = "algorithms/src/snark/varuna/resources/circuit_0"
kat = {"source": base + "/{polynomials/*.txt, *.input} — test_varuna_with_prover_test_vectors (algorithms/src/snark/varuna/tests.rs:623-803): "
                 "7×7 TestCircuit (mul_depth 3), VarunaNonHidingMode, fixed challenges; polynomial coefficients in decimal, low degree first"}
for name in ("w_lde", "z_lde", "h_0", "g_1", "h_1", "g_a", "g_b", "g_c", "h_2"):
    txt = read(f"{base}/polynomials/{name}.txt")
    kat[name] = [s.strip() for s in txt.strip().strip("[]").split(",")]
kat["challenges"] = read(f"{base}/challenges.input").split()
wit = read(f"{base}/witness.input").strip().splitlines()
kat["witness_a_b"] = json.loads(wit[0])
kat["full_assignment"] = json.loads(wit[1])
inst = read(f"{base}/instance.input").split("\n")
mats, cur = {}, None
for line in inst:
    line = line.strip()
    if line in ("A", "B", "C"):
        cur = line; mats[cur] = []
    elif line:
        mats[cur].append([int(t) for t in line.rstrip(",").split(",")])
kat["instance"] = mats
golden["varuna_circuit_0_prover"] = kat
with open(os.path.join(OUT, "reference_constants.json"), "w") as f:
    json.dump(golden, f, indent=1)

# first 512 real SRS points (uncompressed: x LE 48 B, y LE 48 B with flags in the top 2 bits)
with open(os.path.join(REF, "parameters/src/mainnet/resources/powers-of-beta-15.usrs"), "rb") as f:
    blob = f.read(8 + 512 * 96)
with open(os.path.join(OUT, "powers_of_beta_15_first512.usrs"), "wb") as f:
    f.write((512).to_bytes(8, "little") + blob[8:])
print("wrote", os.listdir(OUT))
