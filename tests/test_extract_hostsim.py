"""CPU check of the extraction walk (csrc/extract.cuh, the code k_extract runs) against the big-integer oracle: the key's
endomorphism digits and c.1 - key * c.0 on G1 and G2, for edge-case keys and bases.  Not a product path: tests only."""
import ctypes
import os
import random
import subprocess

import pytest

from conv import fr_b, g1_b, g1_i, g2_b, g2_i
from oracle.bls12_381 import G1, G2, G1_GEN, G2_GEN_FP2, R, X_ABS, g1_mul, g2_mul

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "hostsim", "libhostsim_extract.so")


@pytest.fixture(scope="module")
def L():
    """g++ build of tests/hostsim/extract_hostsim.cpp (extract.cuh and the headers under it, for the host): rebuilt only
    when a source is newer than the cached library."""
    src = os.path.join(HERE, "hostsim", "extract_hostsim.cpp")
    csrc = os.path.join(HERE, "..", "groth-sahai-rs_b200", "csrc")
    deps = [src] + [os.path.join(csrc, f) for f in os.listdir(csrc) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(SO) or os.path.getmtime(SO) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-frounding-math", "-shared", "-fPIC", "-I", csrc, "-o", SO, src])
    return ctypes.CDLL(SO)


def call(fn, n, *args):
    out = ctypes.create_string_buffer(n)
    fn(out, *args)
    return out.raw

rng = random.Random(29)
X2 = X_ABS * X_ABS
# 0, 1, 2, r - 1, x^2 (GLV halves 0 and 1); all-ones GLV halves; GLV halves x^2 - 1, x^2 - 2 whose top windows carry;
# GLS digits 2^63 - 1 (all ones) and |x| - 1 (top windows carry)
EDGE = [0, 1, 2, R - 1, X2, (2 ** 127 - 1) + (2 ** 126 - 1) * X2, (X2 - 1) + (X2 - 2) * X2,
        sum((2 ** 63 - 1) * X_ABS ** j for j in range(3)) + (2 ** 62 - 1) * X_ABS ** 3,
        sum((X_ABS - 1) * X_ABS ** j for j in range(3)) + (X_ABS - 2) * X_ABS ** 3]


def digits(L, k, g2):
    raw = call(L.hs_extract_digits, 133, fr_b(k), 1 if g2 else 0)
    d = [[int.from_bytes(raw[33 * j + i:33 * j + i + 1], "little", signed=True) for i in range(33)] for j in range(4)]
    return d, raw[132]


def test_key_digits(L):
    """The digits recombine to the key (part weights 1, x^2 on G1; |x|^j on G2), lie in [-8, 8), and npos ends at the
    top non-zero digit; the edge keys really hit the all-ones and carry cases."""
    for k in EDGE + [rng.randrange(R) for _ in range(200)]:
        for g2 in (False, True):
            d, npos = digits(L, k, g2)
            parts, nwin = (4, 16) if g2 else (2, 32)
            weight = (lambda j: X_ABS ** j) if g2 else (lambda j: X2 ** j)
            assert sum(d[j][i] * 16 ** i * weight(j) for j in range(parts) for i in range(nwin + 1)) % R == k
            assert all(-8 <= v < 8 for row in d for v in row)
            assert all(d[j][i] == 0 for j in range(4) for i in range(33) if j >= parts or i > nwin or i >= npos)
            assert npos == 0 if k == 0 else any(d[j][npos - 1] for j in range(parts))
    assert [r[32] for r in digits(L, EDGE[6], False)[0][:2]] == [1, 1]          # both GLV halves carry out
    assert digits(L, EDGE[5], False)[0][:2] == [[-1] + [0] * 30 + [-8, 1], [-1] + [0] * 30 + [4, 0]]   # 2^127 - 1, 2^126 - 1
    assert all(r[16] == 1 for r in digits(L, EDGE[8], True)[0])                 # every GLS digit carries out
    assert digits(L, EDGE[4], False)[0][1][0] == 1 and digits(L, EDGE[4], False)[1] == 1


def _check(L, k, c0, c1, g2):
    mul, grp, enc, dec = (g2_mul, G2, g2_b, g2_i) if g2 else (g1_mul, G1, g1_b, g1_i)
    fn, size = (L.hs_extract_g2, 192) if g2 else (L.hs_extract_g1, 96)
    got = dec(call(fn, size, enc(c0) + enc(c1), fr_b(k)))
    want = grp.add(c1, grp.neg(mul(c0, k)))
    assert got == want, (k, g2)


def test_extract_walk_g1(L):
    bases = [None, G1_GEN] + [g1_mul(G1_GEN, rng.randrange(R)) for _ in range(3)]
    keys = EDGE + [rng.randrange(R) for _ in range(12)]
    for i, k in enumerate(keys):
        c0 = bases[i % len(bases)]
        x = g1_mul(G1_GEN, rng.randrange(R))
        for c1 in (None, x, G1.add(x, g1_mul(c0, k)), g1_mul(c0, k)):   # -k c0, x - k c0, x, and the identity
            _check(L, k, c0, c1, False)
    for k in EDGE:
        _check(L, k, G1_GEN, None, False)


def test_extract_walk_g2(L):
    bases = [None, G2_GEN_FP2] + [g2_mul(G2_GEN_FP2, rng.randrange(R)) for _ in range(2)]
    keys = EDGE + [rng.randrange(R) for _ in range(6)]
    for i, k in enumerate(keys):
        c0 = bases[i % len(bases)]
        y = g2_mul(G2_GEN_FP2, rng.randrange(R))
        for c1 in (None, G2.add(y, g2_mul(c0, k)), g2_mul(c0, k)):
            _check(L, k, c0, c1, True)
    for k in EDGE:
        _check(L, k, G2_GEN_FP2, None, True)
