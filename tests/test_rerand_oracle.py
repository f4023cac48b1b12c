"""Proof rerandomisation on the big-integer oracle (no CUDA): the formulas of gs_rerandomize_batch checked against a
fresh commit_and_prove, for all four equation types."""
import pytest

from gsutil import SeededRng, draw_rands, make_crs, random_instance
from oracle import gs as ogs
from rerand_ref import combined_rands, rerandomize


@pytest.fixture(scope="module")
def crs():
    return make_crs(1)[0]


def _case(ty, m, n, crs, seed):
    rng = SeededRng(seed)
    equ, xv, yv = random_instance(ty, m, n, crs, rng)
    xr, yr, T = draw_rands(ty, m, n, rng)
    proof = ogs.commit_and_prove(equ, xv, yv, crs, xr, yr, T)
    return rng, equ, xv, yv, (xr, yr, T), proof


def _same(a: ogs.CProof, b: ogs.CProof):
    return (a.xcoms.coms == b.xcoms.coms and a.ycoms.coms == b.ycoms.coms and
            a.equ_proofs[0].pi == b.equ_proofs[0].pi and a.equ_proofs[0].theta == b.equ_proofs[0].theta)


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_rerandomised_equals_fresh_proof(ty, crs):
    m, n = 2, 3
    rng, equ, xv, yv, rands, proof = _case(ty, m, n, crs, 700 + ty)
    new = draw_rands(ty, m, n, rng)
    out = rerandomize(equ, proof, crs, *new)
    xr2, yr2, T2 = combined_rands(equ.gamma, *rands, *new)
    fresh = ogs.commit_and_prove(equ, xv, yv, crs, xr2, yr2, T2)
    assert _same(out, fresh)
    assert out.xcoms.coms != proof.xcoms.coms and out.equ_proofs[0].pi != proof.equ_proofs[0].pi
    assert ogs.verify(equ, out, crs)


@pytest.mark.parametrize("ty", [0, 3])
def test_zero_randomness_returns_the_input(ty, crs):
    m, n = 2, 2
    _, equ, _, _, _, proof = _case(ty, m, n, crs, 720 + ty)
    cx, cy = (2 if ty in (0, 1) else 1), (2 if ty in (0, 2) else 1)
    out = rerandomize(equ, proof, crs, [[0] * cx] * m, [[0] * cy] * n, [[0] * cx] * cy)
    assert _same(out, proof)


@pytest.mark.parametrize("ty", [1, 2])
def test_false_statement_still_fails(ty, crs):
    m, n = 1, 2
    rng, equ, _, _, _, proof = _case(ty, m, n, crs, 740 + ty)
    equ.target = ogs.G1.add(equ.target, crs.g1_gen) if ty == 1 else ogs.G2.add(equ.target, crs.g2_gen)
    assert not ogs.verify(equ, proof, crs)
    out = rerandomize(equ, proof, crs, *draw_rands(ty, m, n, rng))
    assert not ogs.verify(equ, out, crs)
