#!/usr/bin/env python
"""Writes tests/golden/reference_pins.json: what the original plonkathon modules compute for the inputs of
tests/test_oracle_vs_reference.py, tests/test_synthetic_vs_reference.py and the section-table test of
tests/test_setup_host.py, so that those comparisons run without the original project.

    python tests/golden/make_reference_pins.py <path to a plonkathon checkout>

The original modules run unmodified over oracle/shims (the py_ecc / merlin layer they import)."""
import hashlib
import json
import os
import random
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.path.abspath(sys.argv[1])
sys.path.insert(0, os.path.join(ROOT, "oracle", "shims"))
sys.path.insert(0, REF)
sys.path.insert(0, ROOT)

import curve  # noqa: E402  original
import poly  # noqa: E402  original
import py_ecc.bn128 as b  # noqa: E402  (shim)
from compiler.program import Program  # noqa: E402  original

from oracle import plonk_oracle as O  # noqa: E402
from plonkathon_b200 import synthetic as syn  # noqa: E402

S = curve.Scalar
s = str


def values(p):
    return [s(x.n) for x in p.values]


# ---------------------------------------------------------------- poly.py / curve.py
rng = random.Random(7)
transforms = []
for logn in (0, 1, 2, 5, 9):
    v = [rng.randrange(O.R_MOD) for _ in range(1 << logn)]
    transforms.append({"log_n": logn, "input": [s(a) for a in v],
                       "fft": values(poly.Polynomial([S(a) for a in v], poly.Basis.MONOMIAL).fft()),
                       "ifft": values(poly.Polynomial([S(a) for a in v], poly.Basis.LAGRANGE).ifft())})
pts = [b.multiply(b.G1, rng.randrange(1, 1000)) for _ in range(20)]
sc = [rng.randrange(O.R_MOD) for _ in range(20)]
lc = curve.ec_lincomb(list(zip(pts, sc)))
nums = [rng.randrange(10 ** 20) for _ in range(40)]
fac = [rng.randrange(2 ** 256) for _ in range(40)]
modules = {
    "transforms": transforms,
    "roots_of_unity_16": [s(x.n) for x in S.roots_of_unity(16)],
    "ec_lincomb": {"points": [[s(p[0].n), s(p[1].n)] for p in pts], "scalars": [s(x) for x in sc],
                   "result": [s(lc[0].n), s(lc[1].n)]},
    "lincomb": {"nums": [s(x) for x in nums], "factors": [s(x) for x in fac], "result": s(curve.lincomb(nums, fac))},
}

# ---------------------------------------------------------------- compiler/program.py on synthetic.py's circuits
compiler = []
for log_n, fill in ((3, 1.0), (5, 1.0), (6, 0.8)):
    c = syn.build_circuit(log_n, seed=log_n, n_public=2, fill=fill, with_text=True)
    prog = Program(c.text, 1 << log_n)
    pk = prog.common_preprocessed_input()
    compiler.append({
        "log_n": log_n, "seed": log_n, "n_public": 2, "fill": fill,
        "text_sha256": hashlib.sha256("\n".join(c.text).encode()).hexdigest(),
        **{k: values(getattr(pk, k)) for k in ("QL", "QR", "QM", "QO", "QC", "S1", "S2", "S3")},
        "wires": [[w.L, w.R, w.O] for w in prog.wires()],
        "public": list(prog.get_public_assignments()),
    })

# ---------------------------------------------------------------- the shipped ceremony file's section table
ptau = open(os.path.join(REF, "test", "powersOfTau28_hez_final_11.ptau"), "rb").read()
sections, pos = [], 12
for _ in range(int.from_bytes(ptau[8:12], "little")):
    sections.append([int.from_bytes(ptau[pos:pos + 4], "little"), pos, int.from_bytes(ptau[pos + 4:pos + 12], "little")])
    pos += 12 + sections[-1][2]
assert pos == len(ptau)
lag = next(x for x in sections if x[0] == 12)
ceremony = {"length": len(ptau), "head": ptau[:12].hex(), "sections": sections,
            "lagrange_p0_p4_sha256": hashlib.sha256(ptau[lag[1] + 12:lag[1] + 12 + 64 * 31]).hexdigest()}

with open(os.path.join(HERE, "reference_pins.json"), "w") as f:
    json.dump({"kind": "reference", "modules": modules, "compiler": compiler, "ptau": ceremony}, f)
print("wrote", os.path.join(HERE, "reference_pins.json"))
