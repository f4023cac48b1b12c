"""CPU check of the Fp2 dot products with one Montgomery reduction per output component (coop12.cuh cq_fp2_dot_w) and
of the cooperative ops built on them (line step, squaring, general product, Miller loop, final exponentiation), against
the big-int oracle and byte for byte against the three-reduction forms they replace."""
import ctypes, os, random, subprocess
import pytest
from conv import fp_i, fp12_b, fp12_i, g1_b, g2_b
from oracle.bls12_381 import (P, R, G1_GEN, G2_GEN_FP2, g1_mul, g2_mul, Fp2, Fp6, Fp12, FP12_ONE, multi_miller_loop,
                              final_exponentiation)

HERE = os.path.dirname(os.path.abspath(__file__))
SRC = os.path.join(HERE, "hostsim", "coop_hostsim.cpp")
CSRC = os.path.join(HERE, "..", "groth-sahai-rs_b200", "csrc")
RINV = pow(2 ** 384, -1, P)


def _build(name, defines):
    so = os.path.join(HERE, "hostsim", name)
    deps = [SRC] + [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h"))]
    if not os.path.exists(so) or os.path.getmtime(so) < max(os.path.getmtime(d) for d in deps):
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-frounding-math", "-shared", "-fPIC", "-I", CSRC] + defines +
                              ["-o", so, SRC])
    return ctypes.CDLL(so)


@pytest.fixture(scope="module")
def libs():
    """(default forms, three-reduction forms): two host builds of the same header"""
    new = _build("libcoop_hostsim.so", [])
    old = _build("libcoop_hostsim_k3.so", ["-DGS_LINE_KARATSUBA=1", "-DGS_MUL_KARATSUBA=1"])
    assert new.hs_forms() == 22 and old.hs_forms() == 11
    return new, old


def call(fn, n, *args):
    out = ctypes.create_string_buffer(n)
    fn(out, *args)
    return out.raw


rng = random.Random(23)
# raw Montgomery limbs (any canonical value < p): the edges of the representation, not of the represented value
EDGE = [0, 1, P - 1, P - 2, (P - 1) // 2, (P + 1) // 2, 2 ** 380, 2 ** 352 - 1]


def raw(x): return x.to_bytes(48, "little")
def val(x): return x * RINV % P          # the element a raw limb pattern stands for
def fp12_raw(cs): return b"".join(raw(c) for c in cs)   # 12 raw Fp in tower order
def rfp12(): return Fp12(*(Fp6(*(Fp2(rng.randrange(P), rng.randrange(P)) for _ in range(3))) for _ in range(2)))


def dot_expected(ys, xs):
    """raw result of sum Y_t X_t with Montgomery operands: (sum y x) / R in each component"""
    c0 = sum(y0 * x0 - y1 * x1 for (y0, y1), (x0, x1) in zip(ys, xs)) * RINV % P
    c1 = sum(y0 * x1 + y1 * x0 for (y0, y1), (x0, x1) in zip(ys, xs)) * RINV % P
    return raw(c0) + raw(c1)


def test_dot_w_edges(libs):
    new, _ = libs
    cases = []
    for nt in (1, 2, 3, 4):
        # all zero, all p - 1 (component sums 2p - 2 on both sides), P0 - P1 at its most negative and most positive
        cases.append(([(0, 0)] * nt, [(0, 0)] * nt))
        cases.append(([(P - 1, P - 1)] * nt, [(P - 1, P - 1)] * nt))
        cases.append(([(0, P - 1)] * nt, [(0, P - 1)] * nt))
        cases.append(([(P - 1, 0)] * nt, [(P - 1, 0)] * nt))
        cases.append(([(P - 1, P - 1)] * nt, [(0, P - 1)] * nt))
        for _ in range(60):
            cases.append(([(rng.choice(EDGE), rng.choice(EDGE)) for _ in range(nt)],
                          [(rng.choice(EDGE), rng.choice(EDGE)) for _ in range(nt)]))
        for _ in range(60):
            cases.append(([(rng.randrange(P), rng.randrange(P)) for _ in range(nt)],
                          [(rng.randrange(P), rng.randrange(P)) for _ in range(nt)]))
    for i, (ys, xs) in enumerate(cases):
        yb = b"".join(raw(a) + raw(b) for a, b in ys)
        xb = b"".join(raw(a) + raw(b) for a, b in xs)
        assert call(new.hs_dot_w, 96, len(ys), yb, xb, [0, 13, 31][i % 3]) == dot_expected(ys, xs), (ys, xs)


def _fp12_cases():
    cs = [[0] * 12, [P - 1] * 12, [1] * 12, [P - 1, 0] * 6, [0, P - 1] * 6, [P - 1] * 6 + [0] * 6, [0] * 6 + [P - 1] * 6]
    cs += [[rng.choice(EDGE) for _ in range(12)] for _ in range(12)]
    return [fp12_raw(c) for c in cs] + [fp12_b(rfp12()) for _ in range(8)]


def test_line_sqr_mul_vs_oracle_and_k3(libs):
    """line step, squaring (every coefficient: the xi wrap-around and the doubled terms) and general product on edge
    and random values: equal to the oracle and, byte for byte, to the three-reduction forms"""
    new, old = libs
    vals = _fp12_cases()
    for i, a in enumerate(vals):
        lane = [0, 9, 31][i % 3]
        A = fp12_i(a)
        tile = [rng.choice(EDGE) if i % 2 else rng.randrange(P) for _ in range(4)]
        tb = b"".join(raw(t) for t in tile)
        al, be = Fp2(val(tile[0]), val(tile[1])), Fp2(val(tile[2]), val(tile[3]))
        # alpha + beta w^2 + w^3 in the tower: w^2 = v, w^3 = v w
        line = Fp12(Fp6(al, be, Fp2(0, 0)), Fp6(Fp2(0, 0), Fp2(1, 0), Fp2(0, 0)))
        got = call(new.hs_line_mul_u, 576, a, tb, lane)
        assert got == call(old.hs_line_mul_u, 576, a, tb, lane)
        assert fp12_i(got) == A * line
        got = call(new.hs_sqr, 576, a, lane)
        assert got == call(old.hs_sqr, 576, a, lane)
        assert fp12_i(got) == A * A
        b = vals[(i * 7 + 3) % len(vals)]
        got = call(new.hs_mul, 576, a, b, lane)
        assert got == call(old.hs_mul, 576, a, b, lane)
        assert fp12_i(got) == A * fp12_i(b)


def test_miller_and_final_exp(libs):
    """the Miller loop of k_miller4 (affine lines, unit-gamma line steps, squarings) and the final-exponentiation
    program, against the oracle's pairing product, and equal to the three-reduction forms"""
    new, old = libs
    ps = [g1_mul(G1_GEN, rng.randrange(R)) for _ in range(4)]
    qs = [g2_mul(G2_GEN_FP2, rng.randrange(R)) for _ in range(4)]
    ps[1] = None
    g1s = b"".join(g1_b(p) for p in ps)
    g2s = b"".join(g2_b(q) for q in qs)
    ml = call(new.hs_miller, 576, 4, g1s, g2s, 5)
    assert ml == call(old.hs_miller, 576, 4, g1s, g2s, 5)
    fe = call(new.hs_final_exp, 576, ml, 20)
    assert fe == call(old.hs_final_exp, 576, ml, 20)
    assert fp12_i(fe) == final_exponentiation(multi_miller_loop(list(zip(ps, qs))))
    f = rfp12()
    assert fp12_i(call(new.hs_final_exp, 576, fp12_b(f), 0)) == final_exponentiation(f)
    assert fp12_i(call(new.hs_final_exp, 576, fp12_b(FP12_ONE), 31)) == FP12_ONE
