"""CPU: the wide-product building blocks of csrc/field.cuh (fp_mul_wide, fp_mad_wide, fp_sqr_wide, fp_redc,
fp_mul_sum2) and the group law built on them, compiled for the host with the PTX carry primitives emulated, checked
against Python ints and the oracle's affine group law."""
import ctypes
import os
import random
import subprocess

import pytest

from oracle import plonk_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, "plonkathon_b200", "csrc")
R256 = 1 << 256
FIELDS = [(0, O.R_MOD), (1, O.Q_MOD)]


@pytest.fixture(scope="module")
def lib():
    out = os.path.join(ROOT, "build", "host_selftest_wide.so")
    os.makedirs(os.path.dirname(out), exist_ok=True)
    src = os.path.join(CSRC, "host_selftest.cpp")
    deps = [src] + [os.path.join(CSRC, h) for h in ("field.cuh", "curve.cuh", "msm_digits.cuh", "msm_bucket.cuh",
                                                    "modinv.cuh", "ntt_shard.cuh")]
    if not os.path.exists(out) or any(os.path.getmtime(d) > os.path.getmtime(out) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-shared", "-fPIC", "-x", "c++", src,
                               "-I", CSRC, "-o", out])
    return ctypes.CDLL(out)


def limbs(x, n=8):
    return (ctypes.c_uint32 * n)(*[(x >> (32 * i)) & 0xFFFFFFFF for i in range(n)])


def unlimbs(buf, n):
    return sum(int(buf[i]) << (32 * i) for i in range(n))


def wide(lib, field, op, a=0, b=0, c=0, d=0, t=0):
    """returns (value, return code): 16 output limbs for ops 0, 1, 4 and 8 for ops 2, 3"""
    out = (ctypes.c_uint32 * 16)()
    rc = lib.hs_wide_op(field, op, limbs(a), limbs(b), limbs(c), limbs(d), limbs(t, 16), out)
    assert rc >= 0
    return unlimbs(out, 16 if op in (0, 1, 4) else 8), rc


@pytest.mark.parametrize("field,p", FIELDS)
def test_wide_products(lib, field, p):
    rng = random.Random(100 + field)
    top = R256 - 1
    vals = [0, 1, 2, 0xFFFFFFFF, 1 << 32, p - 1, p - 2, R256 % p, top, top - 1, (1 << 255) + 1] + \
        [rng.randrange(R256) for _ in range(300)] + [rng.randrange(p) for _ in range(300)]
    for i, a in enumerate(vals):
        b = vals[(i * 13 + 5) % len(vals)]
        assert wide(lib, field, 0, a, b)[0] == a * b
        assert wide(lib, field, 1, a)[0] == a * a
        # the accumulating form returns the 17th limb of t + a b
        for t in (0, rng.randrange(1 << 512), (1 << 512) - 1):
            got, carry = wide(lib, field, 4, a, b, t=t)
            assert got + (carry << 512) == t + a * b


@pytest.mark.parametrize("field,p", FIELDS)
def test_redc(lib, field, p):
    rng = random.Random(200 + field)
    rinv = pow(R256, -1, p)
    hi = p * R256 - 1
    ts = [0, 1, hi, hi - 1, p, p * p - 1, (p - 1) * (p - 1), R256 - 1, R256, (p - 1) * R256, (p - 1) * R256 + R256 - 1] + \
        [rng.randrange(p * R256) for _ in range(2000)] + [hi - rng.randrange(1 << 64) for _ in range(50)]
    for t in ts:
        assert wide(lib, field, 2, t=t)[0] == t * rinv % p, hex(t)


@pytest.mark.parametrize("field,p", FIELDS)
def test_mul_sum2(lib, field, p):
    rng = random.Random(300 + field)
    rinv = pow(R256, -1, p)
    one = R256 % p
    special = [0, 1, p - 1, one, p - one, (p - 1) // 2]
    tuples = [(p - 1,) * 4, (0,) * 4, (one,) * 4, (p - 1, p - 1, 0, 0), (0, 0, p - 1, p - 1), (one, p - 1, one, 1)]
    tuples += [tuple(rng.choice(special) for _ in range(4)) for _ in range(200)]
    tuples += [tuple(rng.randrange(p) for _ in range(4)) for _ in range(2000)]
    for a, b, c, d in tuples:
        assert wide(lib, field, 3, a, b, c, d)[0] == (a * b + c * d) * rinv % p
    # and the squaring built on fp_sqr_wide + fp_redc (field op 8) over the same extremes
    for a in special + [rng.randrange(p) for _ in range(500)]:
        out = (ctypes.c_uint32 * 8)()
        assert lib.hs_field_op(field, 8, limbs(a), limbs(0), out) == 0
        assert unlimbs(out, 8) == a * a * rinv % p


# ---- group law: long random chains against the oracle ----------------------------------------------------------------
def mont(x):
    return x * R256 % O.Q_MOD


def unmont(x):
    return x * pow(R256, -1, O.Q_MOD) % O.Q_MOD


def aff_buf(pt):
    return limbs(mont(pt[0]) | (mont(pt[1]) << 256), 16)


def xyzz_of(pt):
    if pt is None:
        return limbs(0, 32)
    return limbs(mont(pt[0]) | (mont(pt[1]) << 256) | (mont(1) << 512) | (mont(1) << 768), 32)


def to_affine(lib, acc):
    out = (ctypes.c_uint32 * 32)()
    inf = lib.hs_curve_op(3, acc, limbs(0, 32), 0, out)
    return None if inf else (unmont(unlimbs(out, 8)), unmont(unlimbs(out[8:16], 8)))


def neg_xyzz(acc):
    """-P in XYZZ: Y -> q - Y (Montgomery form commutes with negation)"""
    v = unlimbs(acc, 32)
    y = (v >> 256) & (R256 - 1)
    v ^= y << 256
    v |= ((O.Q_MOD - y) % O.Q_MOD) << 256
    return limbs(v, 32)


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_group_law_chains(lib, seed):
    """64 steps mixing P + Q, P + P, P + (-P) and identity operands through g1_add_mixed_uniform (op 4),
    g1_add_uniform (op 5) and g1_double (op 2); the accumulator keeps a non-trivial ZZ along the way"""
    rng = random.Random(seed)
    pool = [O.g1_multiply(O.G1, rng.randrange(1, O.R_MOD)) for _ in range(6)]
    acc, exp = xyzz_of(None), None
    history = []  # (XYZZ buffer, point) of earlier accumulators
    kinds = set()
    for step in range(64):
        out = (ctypes.c_uint32 * 32)()
        k = rng.randrange(9)
        if exp is None and k in (1, 2, 5, 6):
            k = 0
        if k == 0:    # mixed add of a fresh point (from the identity too)
            q = rng.choice(pool)
            assert lib.hs_curve_op(4, acc, aff_buf(q), 0, out) == 0
            nxt = O.g1_add(exp, q)
        elif k == 1:  # mixed P + P
            assert lib.hs_curve_op(4, acc, aff_buf(exp), 0, out) == 0
            nxt = O.g1_double(exp)
        elif k == 2:  # mixed P + (-P)
            assert lib.hs_curve_op(4, acc, aff_buf(O.g1_neg(exp)), 0, out) == 0
            nxt = None
        elif k == 3:  # XYZZ add of an earlier accumulator (or the identity)
            buf, pt = rng.choice(history) if history else (xyzz_of(None), None)
            assert lib.hs_curve_op(5, acc, buf, 0, out) == 0
            nxt = O.g1_add(exp, pt)
        elif k == 4:  # XYZZ add of the identity
            assert lib.hs_curve_op(5, acc, xyzz_of(None), 0, out) == 0
            nxt = exp
        elif k == 5:  # XYZZ P + P with both sides in non-trivial coordinates
            same = (ctypes.c_uint32 * 32)(*acc)
            assert lib.hs_curve_op(5, acc, same, 0, out) == 0
            nxt = O.g1_double(exp)
        elif k == 6:  # XYZZ P + (-P)
            assert lib.hs_curve_op(5, acc, neg_xyzz(acc), 0, out) == 0
            nxt = None
        elif k == 7:  # doubling
            assert lib.hs_curve_op(2, acc, limbs(0, 32), 0, out) == 0
            nxt = O.g1_double(exp) if exp is not None else None
        else:         # XYZZ add of a fresh point with ZZ = 1
            q = rng.choice(pool)
            assert lib.hs_curve_op(5, acc, xyzz_of(q), 0, out) == 0
            nxt = O.g1_add(exp, q)
        kinds.add(k)
        acc, exp = out, nxt
        assert to_affine(lib, acc) == exp, f"step {step}, kind {k}"
        history.append((acc, exp))
    assert len(kinds) >= 7
