"""CPU: the oracle restatement vs what the original project's own unmodified modules (poly.py, curve.py, run over
oracle/shims) computed for the same inputs, stored in tests/golden/reference_pins.json by make_reference_pins.py."""
from oracle import plonk_oracle as O
from tests.golden_io import ints, load_json


def test_restatement_matches_reference_modules():
    ref = load_json("reference_pins.json")["modules"]
    for t in ref["transforms"]:
        v = ints(t["input"])
        assert len(v) == 1 << t["log_n"]
        assert O.fft(v) == ints(t["fft"]), t["log_n"]
        assert O.ifft(v) == ints(t["ifft"]), t["log_n"]
    assert O.roots_of_unity(16) == ints(ref["roots_of_unity_16"])
    lc = ref["ec_lincomb"]
    assert O.ec_lincomb([(tuple(ints(p)), s) for p, s in zip(lc["points"], ints(lc["scalars"]))]) == tuple(ints(lc["result"]))
    # the mock-adder self-test of curve.py:115-142 against the restated lincomb
    nums, fac = ints(ref["lincomb"]["nums"]), ints(ref["lincomb"]["factors"])
    assert O.lincomb(nums, fac, lambda x, y: x + y, 0) == int(ref["lincomb"]["result"]) == sum(a * f for a, f in zip(nums, fac))
