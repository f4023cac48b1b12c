"""The per-proof check of gs_verify_each_rand, restated with the big-integer oracle and checked on the CPU, independently of
any CUDA code.  Proof p is accepted iff ONE folded pairing product over the slots of verifier.rs:23-157's equation
        F(iota(A), d) + F(c, iota(B)) + F(c, Gamma d) = iota_T(t) + F(u, pi) + F(theta, v)
matches its folded right-hand side, with that proof's weights (sigma_p, tau_p) and the call's beta:
        fold1(x) = sigma x.0 + tau x.1   (x in Com1),      fold2(y) = beta y.0 + y.1   (y in Com2),
ComT entry (a, b) raised to w_a * beta_b, (w_0, w_1) = (sigma, tau), (beta_0, beta_1) = (beta, 1); nothing is multiplied
across proofs.  Honest proofs of all four types pass for random weights; every single-element tampering fails; a proof
whose error sits in ONE ComT entry fails, for each of the four entries; two proofs with exchanged targets both fail."""
import random

import pytest

from gsutil import SeededRng, make_crs, random_instance, draw_rands
from oracle import gs as ogs
from oracle.bls12_381 import G1, G2, R, FP12_ONE, g1_mul, g2_mul, pairing

XA = 0xD201000000010000


def fold1(x, sg, tu):
    return G1.add(g1_mul(x[0], sg), g1_mul(x[1], tu))


def fold2(y, beta):
    return G2.add(g2_mul(y[0], beta), y[1])


def weights(seed):
    """(sigma, tau, beta) as the GPU uses them: 63-bit sigma, tau; beta = b0 + b1 |x| from one 64-bit word"""
    w = random.Random(seed)
    sg, tu, word = w.getrandbits(63), w.getrandbits(63), w.getrandbits(64)
    return sg, tu, ((word & 0xFFFFFFFF) + (word >> 32) * XA) % R


def each_check(equ, proof, crs, sg, tu, beta, err=None):
    """True iff the folded per-proof equation holds.  err = (entry e, g): the right-hand ComT's entry e multiplied by the
    GT element g (a proof whose error sits in that one entry)."""
    ty = equ.equ_type
    ep = proof.equ_proofs[0]
    pairs_l = list(zip(ogs._map_x(ty, equ.a_consts, crs), proof.ycoms.coms))
    pairs_l += list(zip(proof.xcoms.coms, ogs._map_y(ty, equ.b_consts, crs)))
    gd = ogs.col_vec_to_vec(ogs.com_left_mul(ogs.vec_to_col_vec(proof.ycoms.coms), equ.gamma, 2))
    pairs_l += list(zip(proof.xcoms.coms, gd))
    pairs_r = list(zip(crs.u, ep.pi)) if ty in (ogs.PPE, ogs.MSMEG1) else [(crs.u[0], ep.pi[0])]
    pairs_r += list(zip(ep.theta, crs.v)) if ty in (ogs.PPE, ogs.MSMEG2) else [(ep.theta[0], crs.v[0])]
    lin_t = list({ogs.PPE: lambda: ogs.comt_linear_map_ppe(equ.target),
                  ogs.MSMEG1: lambda: ogs.comt_linear_map_msmeg1(equ.target, crs),
                  ogs.MSMEG2: lambda: ogs.comt_linear_map_msmeg2(equ.target, crs),
                  ogs.QUAD: lambda: ogs.comt_linear_map_quad(equ.target, crs)}[ty]())
    if err is not None:
        lin_t[err[0]] = lin_t[err[0]] * err[1]
    ex = [sg * beta % R, sg, tu * beta % R, tu]
    t = FP12_ONE
    for e in range(4):
        t = t * lin_t[e].pow(ex[e])

    def prod(pairs):
        acc = FP12_ONE
        for x, y in pairs:
            acc = acc * pairing(fold1(x, sg, tu), fold2(y, beta))
        return acc

    return prod(pairs_l) == t * prod(pairs_r)


def instance(ty, m, n, seed, crs):
    rng = SeededRng(seed)
    equ, xv, yv = random_instance(ty, m, n, crs, rng)
    xr, yr, T = draw_rands(ty, m, n, rng)
    return equ, ogs.commit_and_prove(equ, xv, yv, crs, xr, yr, T)


@pytest.fixture(scope="module")
def crs():
    return make_crs(1)[0]


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_honest_proofs_pass_for_random_weights(crs, ty):
    m, n = (2, 1) if ty != 3 else (1, 2)
    equ, proof = instance(ty, m, n, 400 + ty, crs)
    assert ogs.verify(equ, proof, crs)
    for seed in (1, 2):
        assert each_check(equ, proof, crs, *weights(10 * ty + seed))


def _tamperings(equ, proof):
    """every element of a 1 x 1 PPE instance and its proof changed once (a point: its double; a scalar: plus one; the
    target: squared), each as an (equation, proof) pair"""
    ep = proof.equ_proofs[0]
    E = lambda **kw: ogs.Equation(kw.get("ty", equ.equ_type), kw.get("a", equ.a_consts), kw.get("b", equ.b_consts),
                                  kw.get("g", equ.gamma), kw.get("t", equ.target))
    P = lambda **kw: ogs.CProof(kw.get("xc", proof.xcoms), kw.get("yc", proof.ycoms),
                                [ogs.EquProof(kw.get("pi", ep.pi), kw.get("th", ep.theta), ep.equ_type, ep.rand)])
    dbl1, dbl2 = (lambda p: G1.add(p, p)), (lambda q: G2.add(q, q))
    out = [("A", E(a=[dbl1(equ.a_consts[0])]), proof), ("B", E(b=[dbl2(equ.b_consts[0])]), proof),
           ("Gamma", E(g=[[(equ.gamma[0][0] + 1) % R]]), proof), ("t", E(t=equ.target * equ.target), proof)]
    for a in range(2):
        c = [tuple(dbl1(x) if i == a else x for i, x in enumerate(proof.xcoms.coms[0]))]
        out.append((f"c.{a}", equ, P(xc=ogs.Commit(c, proof.xcoms.rand))))
        d = [tuple(dbl2(y) if i == a else y for i, y in enumerate(proof.ycoms.coms[0]))]
        out.append((f"d.{a}", equ, P(yc=ogs.Commit(d, proof.ycoms.rand))))
        for k in range(2):
            pi = [tuple(dbl2(y) if (j, i) == (k, a) else y for i, y in enumerate(row)) for j, row in enumerate(ep.pi)]
            out.append((f"pi{k}.{a}", equ, P(pi=pi)))
            th = [tuple(dbl1(x) if (j, i) == (k, a) else x for i, x in enumerate(row)) for j, row in enumerate(ep.theta)]
            out.append((f"theta{k}.{a}", equ, P(th=th)))
    return out


def test_every_single_element_tampering_fails(crs):
    equ, proof = instance(0, 1, 1, 420, crs)
    w = weights(42)
    assert each_check(equ, proof, crs, *w)
    for name, e, p in _tamperings(equ, proof):
        assert not ogs.verify(e, p, crs), name
        assert not each_check(e, p, crs, *w), f"{name} accepted"


def test_error_in_one_comt_entry_fails(crs):
    """Each of the four entries carries a weight of its own (sigma beta, sigma, tau beta, tau): an error confined to any
    one of them is caught."""
    equ, proof = instance(0, 1, 1, 430, crs)
    w = weights(43)
    g = crs.gt_gen
    for e in range(4):
        assert not each_check(equ, proof, crs, *w, err=(e, g)), f"error in entry {e} accepted"


def test_exchanged_targets_both_fail(crs):
    (e0, p0), (e1, p1) = instance(0, 2, 1, 440, crs), instance(0, 2, 1, 441, crs)
    x0 = ogs.Equation(e0.equ_type, e0.a_consts, e0.b_consts, e0.gamma, e1.target)
    x1 = ogs.Equation(e1.equ_type, e1.a_consts, e1.b_consts, e1.gamma, e0.target)
    assert not ogs.verify(x0, p0, crs) and not ogs.verify(x1, p1, crs)
    assert not each_check(x0, p0, crs, *weights(44))
    assert not each_check(x1, p1, crs, *weights(45))
