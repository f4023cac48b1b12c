"""Extraction with the binding key on the big-integer oracle (no CUDA): the formulas of gs_extract checked on commitments
the oracle makes under generate_crs, for all four commitment kinds."""
import pytest

from extract_ref import extract_g1, extract_g2, key_matches
from gsutil import SeededRng, draw_rands, make_crs, random_instance
from oracle import gs as ogs
from oracle.bls12_381 import G1, G2, R, g1_mul, g2_mul
from rerand_ref import rerandomize


@pytest.fixture(scope="module")
def crs_draws():
    return make_crs(3)


def test_all_four_kinds_extract_to_the_witnesses(crs_draws):
    crs, (p1, p2, a1, a2, _, _) = crs_draws
    rng = SeededRng(31)
    X = [rng.g1() for _ in range(3)] + [None]
    Y = [rng.g2() for _ in range(3)] + [None]
    xs = [rng.fr() for _ in range(3)] + [0, 1, R - 1]
    ys = [rng.fr() for _ in range(3)] + [0, 1, R - 1]
    r2 = lambda k: [[rng.fr(), rng.fr()] for _ in range(k)]
    r1 = lambda k: [[rng.fr()] for _ in range(k)]
    c = ogs.batch_commit_g1(X, crs, r2(len(X))).coms
    assert [extract_g1(x, a1) for x in c] == X
    d = ogs.batch_commit_g2(Y, crs, r2(len(Y))).coms
    assert [extract_g2(y, a2) for y in d] == Y
    cs = ogs.batch_commit_scalar_to_b1(xs, crs, r1(len(xs))).coms
    assert [extract_g1(x, a1) for x in cs] == [g1_mul(p1, x) or None for x in xs]
    ds = ogs.batch_commit_scalar_to_b2(ys, crs, r1(len(ys))).coms
    assert [extract_g2(y, a2) for y in ds] == [g2_mul(p2, y) or None for y in ys]


def test_zero_randomness_and_identity_witnesses(crs_draws):
    """c.0 = O (the randomness sums to zero) extracts to c.1; X = O gives c.1 = a1 c.0 and extracts to O."""
    crs, (p1, p2, a1, a2, _, _) = crs_draws
    rng = SeededRng(32)
    x, y = rng.g1(), rng.g2()
    c = ogs.batch_commit_g1([x, None, None], crs, [[0, 0], [0, 0], [rng.fr(), rng.fr()]]).coms
    assert c[0] == (None, x) and c[1] == (None, None) and c[2][0] is not None
    assert [extract_g1(e, a1) for e in c] == [x, None, None]
    d = ogs.batch_commit_g2([y, None, None], crs, [[0, 0], [0, 0], [rng.fr(), rng.fr()]]).coms
    assert [extract_g2(e, a2) for e in d] == [y, None, None]
    # r0 + t1 r1 = 0: both coordinates collapse onto iota_1(X) although the randomness is not zero
    t1 = crs_draws[1][4]
    r1 = rng.fr()
    c = ogs.batch_commit_g1([x], crs, [[(-t1 * r1) % R, r1]]).coms[0]
    assert c == (None, x) and extract_g1(c, a1) == x


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_rerandomised_commitments_extract_to_the_original_values(ty, crs_draws):
    crs, (p1, p2, a1, a2, _, _) = crs_draws
    rng = SeededRng(40 + ty)
    m, n = 2, 3
    equ, xv, yv = random_instance(ty, m, n, crs, rng)
    proof = ogs.commit_and_prove(equ, xv, yv, crs, *draw_rands(ty, m, n, rng))
    out = rerandomize(equ, proof, crs, *draw_rands(ty, m, n, rng))
    assert out.xcoms.coms != proof.xcoms.coms
    want_x = xv if ty in (0, 1) else [g1_mul(p1, x) for x in xv]
    want_y = yv if ty in (0, 2) else [g2_mul(p2, y) for y in yv]
    for coms in (proof.xcoms.coms, out.xcoms.coms):
        assert [extract_g1(c, a1) for c in coms] == want_x
    for coms in (proof.ycoms.coms, out.ycoms.coms):
        assert [extract_g2(d, a2) for d in coms] == want_y


def test_key_check(crs_draws):
    crs, (p1, p2, a1, a2, t1, t2) = crs_draws
    assert key_matches(crs, a1, a2) == (True, True)
    assert key_matches(crs, a2, a1) == (False, False)
    assert key_matches(crs, (a1 + 1) % R, 0) == (False, False)
    assert key_matches(crs, t1, t2) == (False, False)
    # the hiding key u[1] - iota_1(g1), v[1] - iota_2(g2): u[1] extracts to -g1, so the right a1 is rejected too
    hid = ogs.CRS(u=[crs.u[0], ogs.com1_add(crs.u[1], ogs.com1_neg(ogs.com1_linear_map(crs.g1_gen)))],
                  v=[crs.v[0], ogs.com2_add(crs.v[1], ogs.com2_neg(ogs.com2_linear_map(crs.g2_gen)))],
                  g1_gen=crs.g1_gen, g2_gen=crs.g2_gen, gt_gen=crs.gt_gen)
    assert extract_g1(hid.u[1], a1) == G1.neg(crs.g1_gen)
    assert extract_g2(hid.v[1], a2) == G2.neg(crs.g2_gen)
    assert key_matches(hid, a1, a2) == (False, False)
    # another CRS's key does not match this one
    other, (_, _, b1, b2, _, _) = make_crs(4)
    assert key_matches(other, b1, b2) == (True, True) and key_matches(crs, b1, b2) == (False, False)
