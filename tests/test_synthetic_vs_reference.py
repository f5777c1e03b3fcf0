"""CPU: the array-level circuit builder (plonkathon_b200/synthetic.py) against what the original project's own
compiler made of the same wiring (tests/golden/reference_pins.json, written by make_reference_pins.py) -- selectors,
permutation polynomials, wire values and public inputs must agree element for element."""
import hashlib

from plonkathon_b200 import synthetic as syn
from tests.golden_io import ints, load_json


def test_builder_matches_reference_compiler():
    for ref in load_json("reference_pins.json")["compiler"]:
        log_n = ref["log_n"]
        c = syn.build_circuit(log_n, seed=ref["seed"], n_public=ref["n_public"], fill=ref["fill"], with_text=True)
        # the pins are the compiler's output for exactly this program text
        assert hashlib.sha256("\n".join(c.text).encode()).hexdigest() == ref["text_sha256"], log_n
        S1, S2, S3 = syn.permutation_polys(c.wire_L, c.wire_R, c.wire_O, c.group_order, c.n_constraints)
        assert (ints(ref["QL"]) == c.QL and ints(ref["QR"]) == c.QR and ints(ref["QM"]) == c.QM
                and ints(ref["QO"]) == c.QO and ints(ref["QC"]) == c.QC), log_n
        assert ints(ref["S1"]) == S1 and ints(ref["S2"]) == S2 and ints(ref["S3"]) == S3, log_n
        names = {("v%d" % i): v for i, v in enumerate(c.values)}
        names[None] = 0
        A, B, C = c.wires_values()
        m = c.n_constraints
        assert [names[w[0]] for w in ref["wires"]] == A[:m]
        assert [names[w[1]] for w in ref["wires"]] == B[:m]
        assert [names[w[2]] for w in ref["wires"]] == C[:m]
        assert [names[v] for v in ref["public"]] == c.public_values()
