"""Zero-knowledge simulation on the big-integer oracle (no CUDA): the formulas of gs_simulate_batch checked two ways (the
direct formula and the reference-order prove of the augmented equation must agree), and simulated proofs of random,
almost surely false statements verified under the hiding key and rejected under the binding key of the same draws."""
import pytest

from gsutil import SeededRng, draw_rands, make_crs
from oracle import gs as ogs
from oracle.bls12_381 import FP12_ONE, R, g1_mul, g2_mul
from simulate_ref import augmented, hiding_crs, simulate


@pytest.fixture(scope="module")
def keys():
    crs, (p1, p2, a1, a2, t1, t2) = make_crs(5)
    return crs, hiding_crs(crs), t1, t2


def random_statement(ty, m, n, crs, rng):
    """constants, Gamma and a random target: for MSMEG1 / MSMEG2 / Quad a statement nobody knows a witness for"""
    g1, g2 = crs.g1_gen, crs.g2_gen
    a = [g1_mul(g1, rng.fr()) if ty in (0, 1) else rng.fr() for _ in range(n)]
    b = [g2_mul(g2, rng.fr()) if ty in (0, 2) else rng.fr() for _ in range(m)]
    gam = [[rng.fr() for _ in range(n)] for _ in range(m)]
    target = {0: FP12_ONE, 1: g1_mul(g1, rng.fr()), 2: g2_mul(g2, rng.fr()), 3: rng.fr()}[ty]
    return ogs.Equation(ty, a, b, gam, target)


def _same(a: ogs.CProof, b: ogs.CProof):
    return (a.xcoms.coms == b.xcoms.coms and a.ycoms.coms == b.ycoms.coms and
            a.equ_proofs[0].pi == b.equ_proofs[0].pi and a.equ_proofs[0].theta == b.equ_proofs[0].theta)


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
@pytest.mark.parametrize("m,n", [(1, 1), (2, 2)])
def test_direct_formula_equals_prove_of_the_augmented_equation(keys, ty, m, n):
    _, hid, t1, t2 = keys
    rng = SeededRng(900 + 10 * ty + m)
    equ = random_statement(ty, m, n, hid, rng)
    xr, yr, T = draw_rands(ty, m, n, rng)
    sim = simulate(equ, hid, t1, t2, xr, yr, T)
    aug, xv, yv, xr2, yr2 = augmented(equ, t1, t2, xr, yr)
    ref = ogs.commit_and_prove(aug, xv, yv, hid, xr2, yr2, T)
    # the extra variable's commitment is W2 (W1): the commitment of 0 with randomness t2 (t1)
    if ty in (1, 3):
        assert ref.ycoms.coms[n] == ogs.w2(hid)
        ref.ycoms.coms = ref.ycoms.coms[:n]
    if ty == 2:
        assert ref.xcoms.coms[m] == ogs.w1(hid)
        ref.xcoms.coms = ref.xcoms.coms[:m]
    assert _same(sim, ref)


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
@pytest.mark.parametrize("m,n", [(1, 1), (2, 2)])
def test_simulated_proofs_of_random_targets_verify_under_the_hiding_key_only(keys, ty, m, n):
    crs, hid, t1, t2 = keys
    rng = SeededRng(950 + 10 * ty + m)
    equ = random_statement(ty, m, n, hid, rng)
    xr, yr, T = draw_rands(ty, m, n, rng)
    sim = simulate(equ, hid, t1, t2, xr, yr, T)
    assert ogs.verify(equ, sim, hid)
    assert not ogs.verify(equ, sim, crs)
    if ty == 0:
        return   # nothing is absorbed through the trapdoor
    # a wrong trapdoor: t2 (t1 for MSMEG2) off by one
    wrong = simulate(equ, hid, (t1 + 1) % R if ty == 2 else t1, t2 if ty == 2 else (t2 + 1) % R, xr, yr, T)
    assert not ogs.verify(equ, wrong, hid)
