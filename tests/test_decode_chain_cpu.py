"""CPU checks of the two pieces of point decompression that run as fixed schedules (csrc/fields.cuh fp_sqrt with
the generated addition chain of csrc/fp_sqrt_chain.cuh, csrc/g1.cuh g1_in_subgroup_endo), compiled for the host
through tests/hostcheck/hostcheck.cpp:
  * the chain computes exactly a^((p+1)/4), read off the generated code and checked on values;
  * the subgroup test's final projective comparison of t = [z^2] phi(P) with -P, on inputs where t is the point at
    infinity and where t is +P instead of -P."""
import ctypes
import os
import random
import re
import subprocess
import sys

import pytest

from oracle import bls12381 as b
from util import RP, RP_INV, aff_enc

P, R = b.P, b.R
Z = 0xD201000000010000  # |z|
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CHAIN = os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "fp_sqrt_chain.cuh")


@pytest.fixture(scope="module")
def hc(tmp_path_factory):
    out = str(tmp_path_factory.mktemp("hc") / "libhostcheck.so")
    src = os.path.join(HERE, "hostcheck", "hostcheck.cpp")
    extra = os.environ.get("CDL_HOSTCHECK_FLAGS", "").split()
    subprocess.run(["g++", "-O2", "-std=c++17", *extra, "-x", "c++", "-shared", "-fPIC", "-o", out, src], check=True)
    return ctypes.CDLL(out)


def chain_exponent(text):
    """the exponent the generated fp_pow_sqrt_exp raises a to, and its squaring and product counts"""
    e, nsqr, nmul = {"a": 1}, 0, 0
    body = text[text.index("fp_pow_sqrt_exp"):]
    for line in body.splitlines()[1:]:
        line = line.strip()
        if m := re.fullmatch(r"FpM::sqr\((\w+), (\w+)\);", line):
            e[m[1]] = 2 * e[m[2]]
            nsqr += 1
        elif m := re.fullmatch(r"FpM::mul\((\w+), (\w+), (\w+)\);", line):
            e[m[1]] = e[m[2]] + e[m[3]]
            nmul += 1
        elif m := re.fullmatch(r"fp_sqr_n\(r, (\d+)\);", line):
            e["r"] <<= int(m[1])
            nsqr += int(m[1])
        elif m := re.fullmatch(r"r = (\w+);", line):
            e["r"] = e[m[1]]
        else:
            assert line in ("}", "") or line.startswith("Fp "), line
    return e["r"], nsqr, nmul


def test_sqrt_chain_is_the_exponent():
    with open(CHAIN) as f:
        text = f.read()
    exp, nsqr, nmul = chain_exponent(text)
    assert exp == (P + 1) // 4
    assert f"{nsqr} squarings and {nmul} products" in text
    assert nsqr + nmul < 384 + 110  # shorter than the 4-bit fixed window with its 16-entry table
    # the header is what tools/sqrt_chain.py writes
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "sqrt_chain.py"), "--check"],
                         capture_output=True, text=True, timeout=300)
    assert res.returncode == 0, res.stdout + res.stderr


def test_sqrt_chain_values(hc):
    random.seed(31)
    vals = [0, 1, 2, 4, P - 1, P - 4, (P - 1) // 2] + [random.randrange(P) for _ in range(400)]
    vals += [v * v % P for v in vals[:100]]
    n = len(vals)
    out = ctypes.create_string_buffer(48 * n)
    ok = (ctypes.c_int * n)()
    hc.hc_fp_sqrt(b"".join((v * RP % P).to_bytes(48, "little") for v in vals), out, ok, n)
    got = [int.from_bytes(out.raw[48 * i:48 * i + 48], "little") * RP_INV % P for i in range(n)]
    e = (P + 1) // 4
    assert got == [pow(v, e, P) for v in vals]  # non-squares too: the candidate is a^((p+1)/4) whatever a is
    assert list(ok) == [int(pow(v, 2 * e, P) == v) for v in vals]
    assert sum(ok) > 100 and sum(ok) < n


# affine group law on y^2 = x^3 + b' for any b' (a = 0): the subgroup test's formulas never use the curve
# constant, so an input off y^2 = x^3 + 4 runs on the curve through it
def _add(p1, p2):
    if p1 is None:
        return p2
    if p2 is None:
        return p1
    (x1, y1), (x2, y2) = p1, p2
    if x1 == x2:
        if (y1 + y2) % P == 0:
            return None
        lam = 3 * x1 * x1 * pow(2 * y1, -1, P) % P
    else:
        lam = (y2 - y1) * pow(x2 - x1, -1, P) % P
    x3 = (lam * lam - x1 - x2) % P
    return x3, (lam * (x1 - x3) - y1) % P


def _mul(pt, k):
    acc = None
    for bit in bin(k)[2:]:
        acc = _add(acc, acc)
        if bit == "1":
            acc = _add(acc, pt)
    return acc


def _beta():
    """the cube root of unity with phi(x, y) = (beta x, y) = (z^2 - 1) (x, y) on G1"""
    g = 2
    while pow(g, (P - 1) // 3, P) == 1:
        g += 1
    w = pow(g, (P - 1) // 3, P)
    lam_g = b.g1_mul(b.G1_GEN, (Z * Z - 1) % R)
    beta = next(c for c in (w, w * w % P) if (c * b.G1_GEN[0] % P, b.G1_GEN[1]) == lam_g)
    assert (beta * RP % P).to_bytes(48, "little") == _csrc_beta()
    return beta


def _csrc_beta():
    with open(os.path.join(ROOT, "go-curdleproofs_b200", "csrc", "fields.cuh")) as f:
        words = re.search(r"#define CDL_FP_BETA\s+\{([^}]*)\}", f.read())[1]
    return b"".join(int(w.strip().rstrip("u"), 16).to_bytes(4, "little") for w in words.split(","))


def _t(pt, beta):
    """t = [z^2] phi(P), the value the test compares with -P"""
    return _mul((beta * pt[0] % P, pt[1]), Z * Z)


def _in_subgroup(hc, pts):
    out = (ctypes.c_int * len(pts))()
    hc.hc_g1_in_subgroup(b"".join(aff_enc(p) for p in pts), out, len(pts))
    return list(out)


def test_subgroup_check_t_at_infinity(hc):
    """Points (x0, 0) are of order 2 on y^2 = x^3 - x0^3; z is even, so [z^2] phi(P) is the point at infinity,
    which is never -P for a finite P.  The doubling runs reach infinity after the first doubling and the mixed
    additions restart from phi(P) each time.  The Jacobian infinities these formulas produce have X != 0, so the
    x comparison alone already rejects them: this checks the result on that path, not the explicit infinity
    guard before the comparison."""
    random.seed(41)
    beta = _beta()
    pts = [(x, 0) for x in [1, 2, P - 1] + [random.randrange(1, P) for _ in range(5)]]
    for pt in pts:
        assert _t(pt, beta) is None
    assert _in_subgroup(hc, pts) == [0] * len(pts)


def test_subgroup_check_t_equals_plus_p(hc):
    """(0, +-2) are the points of order 3 on the curve itself and phi fixes them; z^2 = 1 mod 3, so
    t = [z^2] phi(P) = +P: the x coordinates agree and the y coordinates differ in sign.  The same holds for
    (0, y) on any curve y^2 = x^3 + y^2.  Beside them, points with t = -P (G1 points and the same construction
    shifted into G1) pass."""
    random.seed(43)
    beta = _beta()
    bad = [(0, 2), (0, P - 2)] + [(0, random.randrange(1, P)) for _ in range(4)]
    for pt in bad:
        assert _t(pt, beta) == pt
    assert [int(b.g1_in_subgroup(p)) for p in bad[:2]] == [0, 0]
    good = [b.g1_mul(b.G1_GEN, random.randrange(1, R)) for _ in range(3)]
    for pt in good:
        assert _t(pt, beta) == b.g1_neg(pt)
    assert _in_subgroup(hc, bad + good) == [0] * len(bad) + [1] * len(good)
