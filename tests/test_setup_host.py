"""CPU: host logic of plonkathon_b200/setup.py for the Lagrange-basis SRS (SURVEY 8(f) N4) -- the snarkjs section
walker and the decoding of section 12 -- checked against the section table of the reference's ceremony file, and
through properties of the committed fixture (tests/golden/ptau_lagrange_p0_p4.bin, the first 31 points
of that section): for every domain size the Lagrange points sum to the generator, and the size-8 block reproduces
the reference's commitment KAT (test.py:23-28) with no inverse transform."""
import hashlib
import os

from oracle import plonk_oracle as O
from plonkathon_b200.setup import PTAU_SECTION_LAGRANGE_G1, decode_ptau_coordinates, ptau_sections
from tests.golden_io import GOLDEN, PTAU_HEAD, load_json, pt

FIXTURE = os.path.join(GOLDEN, "ptau_lagrange_p0_p4.bin")
FACTOR = pow(2, 256, O.Q_MOD)


def blocks():
    raw = decode_ptau_coordinates(open(FIXTURE, "rb").read(), FACTOR)
    pts = [(int.from_bytes(raw[i:i + 32], "little"), int.from_bytes(raw[i + 32:i + 64], "little"))
           for i in range(0, len(raw), 64)]
    return {1 << p: pts[(1 << p) - 1:(2 << p) - 1] for p in range(5)}


def test_section_walker_on_a_synthesised_file():
    head = open(PTAU_HEAD, "rb").read()
    lag = open(FIXTURE, "rb").read()

    def section(sid, data):
        return sid.to_bytes(4, "little") + len(data).to_bytes(8, "little") + data

    body = section(1, head[24:68]) + section(2, head[80:80 + 64 * 16]) + section(3, head[-256:]) + section(12, lag)
    f = b"ptau" + (1).to_bytes(4, "little") + (4).to_bytes(4, "little") + body
    secs = ptau_sections(f)
    assert sorted(secs) == [1, 2, 3, 12] and secs[1] == (24, 44) and secs[2] == (80, 1024)
    off, size = secs[PTAU_SECTION_LAGRANGE_G1]
    assert f[off:off + size] == lag
    assert 12 not in ptau_sections(f[:-1]) and ptau_sections(b"nope") == {} and ptau_sections(b"") == {}
    # the committed head of the real file: header and the monomial G1 section are complete, the rest is cut off
    assert ptau_sections(head) == {1: (24, 44), 2: (80, 262080)}


def test_section_walker_on_the_reference_file():
    """the reference's ceremony file rebuilt at full length from its recorded section table (reference_pins.json),
    the committed head and the committed section-12 points; every other byte is zero"""
    real = load_json("reference_pins.json")["ptau"]
    contents = bytearray(real["length"])
    head = open(PTAU_HEAD, "rb").read()
    contents[:len(head)] = head
    assert bytes(contents[:12]) == bytes.fromhex(real["head"])
    for sid, pos, size in real["sections"]:
        contents[pos:pos + 12] = sid.to_bytes(4, "little") + size.to_bytes(8, "little")
    lag = open(FIXTURE, "rb").read()
    contents[869812:869812 + len(lag)] = lag
    secs = ptau_sections(bytes(contents))
    assert secs == {sid: (pos + 12, size) for sid, pos, size in real["sections"]}
    assert secs[2] == (80, 262080) and secs[3][0] == 262172 and secs[12] == (869812, 64 * (2 ** 13 - 1))
    assert hashlib.sha256(lag).hexdigest() == real["lagrange_p0_p4_sha256"]


def test_lagrange_blocks_are_lagrange_bases():
    for n, pts in blocks().items():
        assert len(pts) == n and all(O.g1_is_on_curve(p) for p in pts)
        total = None
        for p in pts:
            total = O.g1_add(total, p)
        assert total == O.G1, n  # sum_i L_i(X) == 1
    # sum_i w^i L_i(tau) = [tau]_1: ties the blocks to the monomial section of the same ceremony
    osetup = O.Setup.from_file(PTAU_HEAD)
    for n in (2, 8, 16):
        w = O.root_of_unity(n)
        assert O.ec_lincomb_naive([(p, pow(w, i, O.R_MOD)) for i, p in enumerate(blocks()[n])]) == osetup.powers_of_x[1]


def test_commitment_kat_from_the_lagrange_block():
    kat = load_json("circuits.json")["commit_kat"]
    got = O.ec_lincomb_naive([(p, int(v)) for p, v in zip(blocks()[8], kat["lagrange"])])
    assert got == pt(kat["point"])
