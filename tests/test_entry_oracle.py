"""The one-entry tamper of entry_ref.py, confirmed by the big-integer oracle's own per-entry comparison (no GPU): for every
equation type and both keys a proof can be made wrong in exactly one chosen ComT entry, by gt_gen^lambda exactly, and
the C oracle rejects it; errors that cancel in an unweighted product of the entries, and an error that cancels under one
particular set of randomised-verifier weights, are built the same way.  These are the inputs test_gpu_entry.py hands
to every GPU verifier."""
import random

import pytest

from entry_ref import *  # noqa: F401,F403
from test_randfold_each_oracle import each_check

M = N = 2


@pytest.fixture(scope="module")
def draws():
    return make_crs(1)[1]


def oracle_ratios(key, ty, arrays):
    return ratios(*oracle_form(ty, M, N, arrays), key.crs)


@pytest.mark.parametrize("hiding", [False, True], ids=["binding", "hiding"])
@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_each_entry_alone(draws, ty, hiding):
    key = Key(draws, hiding)
    case = Case(ty, M, N, key.crs, seed=5000 + 10 * ty + hiding)
    c, d = com_logs(key, case)
    assert case.xc == b"".join(g1_b(g1_mul(key.crs.g1_gen, k)) for x in c for k in x), "x-commitment logs"
    assert case.yc == b"".join(g2_b(g2_mul(key.crs.g2_gen, k)) for y in d for k in y), "y-commitment logs"
    assert oracle_ratios(key, ty, case.verify_arrays()) == [FP12_ONE] * 4
    for t, E in enumerate(errors(key, ty, lam=7)):
        bad = tamper(key, case, E, i=t % M, j=(t // 2) % N)
        assert oracle_ratios(key, ty, bad) == gt_of(key.crs, E), f"error {E}"
        assert not cb.verify(ty, M, N, bad, key.crsb, NT), f"error {E} accepted"
    if not reachable(key, ty):
        with pytest.raises(ValueError):
            tamper(key, case, unit(3))


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_cancelling_errors(draws, ty):
    """E00 - E11 and E01 - E10: the unweighted product of the four entries is unchanged, the weighted fold is not"""
    key = Key(draws)
    case = Case(ty, M, N, key.crs, seed=5100 + ty)
    for k, E in enumerate(([[1, 0], [0, R - 1]], [[0, 1], [R - 1, 0]])):
        bad = tamper(key, case, E)
        r = oracle_ratios(key, ty, bad)
        assert r == gt_of(key.crs, E)
        assert r[0] * r[1] * r[2] * r[3] == FP12_ONE
        equ, proof = oracle_form(ty, M, N, bad)
        rho = random.Random(5110 + 2 * ty + k).randbytes(24)
        assert not each_check(equ, proof, key.crs, *weights_of(rho, 0, 1)), f"cancelling error {E} accepted"


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_weight_cancelling_error(draws, ty):
    """sigma beta E00 + sigma E01 + tau beta E10 + tau E11 = 0 for the weights one rho gives: the per-proof fold accepts
    the proof with exactly those weights and rejects it once one used bit of sigma, tau or beta changes; bit 63 of sigma
    and tau is not used"""
    key = Key(draws)
    case = Case(ty, 1, 1, key.crs, seed=5200 + ty)
    count, p = 3, 1
    rho = random.Random(5210 + ty).randbytes(8 * (2 * count + 1))
    E = weight_cancelling(*weights_of(rho, p, count))
    bad = tamper(key, case, E)
    equ, proof = oracle_form(ty, 1, 1, bad)
    assert ratios(equ, proof, key.crs) == gt_of(key.crs, E)
    assert not cb.verify(ty, 1, 1, bad, key.crsb, NT)
    assert each_check(equ, proof, key.crs, *weights_of(rho, p, count))
    for word, bit in ((2 * p, 0), (2 * p, 62), (2 * p + 1, 17), (2 * count, 5), (2 * count, 63)):
        assert not each_check(equ, proof, key.crs, *weights_of(flip_bit(rho, word, bit), p, count)), (word, bit)
    for word in (2 * p, 2 * p + 1):
        assert weights_of(flip_bit(rho, word, 63), p, count) == weights_of(rho, p, count)
