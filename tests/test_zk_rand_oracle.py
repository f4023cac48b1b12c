"""The per-statement check of gs_zk_ppe_verify_each_rand, restated with the big-integer oracle and zk_ref.py and checked on
the CPU, independently of any CUDA code.  Statement i is PPE' (target 1) and its K equations L_k : Z_k - delta P_k = O
(target O, whose ComT image is 1).  Every equation e gets weights of its own (sigma_e, tau_e), the call one beta; the
statement is accepted iff ONE folded pairing product over the slots of all 1 + K equations is 1:
        prod_e prod_slots e( sigma_e x.0 + tau_e x.1 ,  beta y.0 + y.1 )  over  lhs slots and the negated rhs slots.
Real proofs pass under the binding key, simulated proofs of false targets under the hiding key; every single-element
tampering fails; a Z other than P that still satisfies PPE' fails; and errors +D on PPE''s theta_0 and -D on L_1's theta
(both paired with v_1) fail with independent weights but cancel when PPE' and L_1 share theirs."""
import random

import pytest

from gsutil import SeededRng, make_crs
from oracle import gs as ogs
from oracle.bls12_381 import G1, G2, FP12_ONE, R, g1_mul, g2_mul, multi_pairing
from simulate_ref import hiding_crs
from test_randfold_each_oracle import fold1, fold2
from test_zk_oracle import draws, satisfied
import zk_ref

XA = 0xD201000000010000


def weights(seed, K):
    """[(sigma_e, tau_e) for e = PPE', L_1..L_K] and beta, as the GPU draws them: the low 63 bits of 2 (1 + K) words,
    beta = b0 + b1 |x| from one 64-bit word"""
    w = random.Random(seed)
    st = [(w.getrandbits(63), w.getrandbits(63)) for _ in range(1 + K)]
    word = w.getrandbits(64)
    return st, ((word & 0xFFFFFFFF) + (word >> 32) * XA) % R


def slot_pairs(equ, xcoms, ycoms, ep, crs):
    """the (Com1, Com2) slots of one equation of target 1: lhs, then rhs with its G1 side negated"""
    ty = equ.equ_type
    pairs = list(zip(ogs._map_x(ty, equ.a_consts, crs), ycoms.coms))
    pairs += list(zip(xcoms.coms, ogs._map_y(ty, equ.b_consts, crs)))
    gd = ogs.col_vec_to_vec(ogs.com_left_mul(ogs.vec_to_col_vec(ycoms.coms), equ.gamma, 2))
    pairs += list(zip(xcoms.coms, gd))
    rhs = list(zip(crs.u, ep.pi)) + (list(zip(ep.theta, crs.v)) if ty == ogs.PPE else [(ep.theta[0], crs.v[0])])
    return pairs + [(ogs.com1_neg(x), y) for x, y in rhs]


def statement_check(a, b, gamma, pairs, proof, crs, w):
    """True iff the folded per-statement product is 1 (one final exponentiation)"""
    (st, beta), (xcoms, ycoms, pf, lin) = w, proof
    m = len(b)
    ppe, lins = zk_ref.augmented(a, b, gamma, pairs)
    eqs = [(ppe, xcoms, ycoms, pf)] + [(L, *zk_ref.lin_coms(xcoms, m, k, crs), lin[k]) for k, L in enumerate(lins)]
    folded = []
    for (sg, tu), (equ, xc, yc, ep) in zip(st, eqs):
        folded += [(fold1(x, sg, tu), fold2(y, beta)) for x, y in slot_pairs(equ, xc, yc, ep, crs)]
    return multi_pairing(folded) == FP12_ONE


@pytest.fixture(scope="module")
def keys():
    crs, (p1, p2, a1, a2, t1, t2) = make_crs(6)
    return crs, hiding_crs(crs), t1, t2


SHAPES = [(1, 1, 1), (2, 2, 1), (1, 1, 2)]


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_real_proofs_pass_under_the_binding_key(keys, m, n, K):
    crs = keys[0]
    rng = SeededRng(5000 + 100 * m + 10 * n + K)
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(m, n, K, rng))
    assert zk_ref.verify(a, b, gam, pairs, proof, crs)
    for seed in (1, 2):
        assert statement_check(a, b, gam, pairs, proof, crs, weights(seed, K))


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_simulated_proofs_of_false_targets_pass_under_the_hiding_key(keys, m, n, K):
    crs, hid, t1, t2 = keys
    rng = SeededRng(5100 + 100 * m + 10 * n + K)
    a, b, gam, _, _, _, _ = satisfied(m, n, K, hid, rng)
    pairs = [(g1_mul(hid.g1_gen, rng.fr()), g2_mul(hid.g2_gen, rng.fr())) for _ in range(K)]   # no known witness
    sim = zk_ref.simulate(a, b, gam, pairs, hid, t1, t2, *draws(m, n, K, rng))
    w = weights(3, K)
    assert statement_check(a, b, gam, pairs, sim, hid, w)
    assert not statement_check(a, b, gam, pairs, sim, crs, w)


def _tamperings(a, b, gam, pairs, proof):
    """every element of a (1, 1, 1) statement and its proof changed once (a point: its double; a scalar: plus one), each as
    (name, a, b, gamma, pairs, proof)"""
    xcoms, ycoms, pf, lin = proof
    dbl1, dbl2 = (lambda p: G1.add(p, p)), (lambda q: G2.add(q, q))
    com1 = lambda c, i: tuple(dbl1(x) if j == i else x for j, x in enumerate(c))
    com2 = lambda c, i: tuple(dbl2(y) if j == i else y for j, y in enumerate(c))
    P, Q = pairs[0]
    out = [("A", [dbl1(a[0])], b, gam, pairs, proof), ("B", a, [dbl2(b[0])], gam, pairs, proof),
           ("Gamma", a, b, [[(gam[0][0] + 1) % R]], pairs, proof), ("P", a, b, gam, [(dbl1(P), Q)], proof),
           ("Q", a, b, gam, [(P, dbl2(Q))], proof)]
    for i in range(2):
        for j in range(2):   # X_1 and Z_1
            xc = ogs.Commit([com1(c, i) if k == j else c for k, c in enumerate(xcoms.coms)], xcoms.rand)
            out.append((f"c{j}.{i}", a, b, gam, pairs, (xc, ycoms, pf, lin)))
        yc = ogs.Commit([com2(ycoms.coms[0], i)], ycoms.rand)
        out.append((f"d.{i}", a, b, gam, pairs, (xcoms, yc, pf, lin)))
        for k in range(2):
            e = ogs.EquProof([com2(y, i) if r == k else y for r, y in enumerate(pf.pi)], pf.theta, pf.equ_type, pf.rand)
            out.append((f"pi{k}.{i}", a, b, gam, pairs, (xcoms, ycoms, e, lin)))
            e = ogs.EquProof(pf.pi, [com1(x, i) if r == k else x for r, x in enumerate(pf.theta)], pf.equ_type, pf.rand)
            out.append((f"theta{k}.{i}", a, b, gam, pairs, (xcoms, ycoms, e, lin)))
            e = ogs.EquProof([com2(y, i) if r == k else y for r, y in enumerate(lin[0].pi)], lin[0].theta, lin[0].equ_type,
                             lin[0].rand)
            out.append((f"lin_pi{k}.{i}", a, b, gam, pairs, (xcoms, ycoms, pf, [e])))
        e = ogs.EquProof(lin[0].pi, [com1(lin[0].theta[0], i)], lin[0].equ_type, lin[0].rand)
        out.append((f"lin_theta.{i}", a, b, gam, pairs, (xcoms, ycoms, pf, [e])))
    return out


def test_every_single_element_tampering_fails(keys):
    crs = keys[0]
    rng = SeededRng(5200)
    a, b, gam, pairs, X, Y, _ = satisfied(1, 1, 1, crs, rng)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(1, 1, 1, rng))
    w = weights(4, 1)
    assert statement_check(a, b, gam, pairs, proof, crs, w)
    for name, *t in _tamperings(a, b, gam, pairs, proof):
        assert not zk_ref.verify(*t, crs), name
        assert not statement_check(*t, crs, w), f"{name} accepted"


def test_z_that_satisfies_ppe_prime_but_not_p_fails(keys):
    """Z_k = P_k + s_k g1 with s_1 q_1 + s_2 q_2 = 0: PPE' holds, the L_k do not"""
    crs = keys[0]
    rng = SeededRng(5300)
    a, b, gam, pairs, X, Y, qs = satisfied(1, 1, 2, crs, rng)
    s = rng.fr()
    shift = [s, (-s * qs[0] * pow(qs[1], -1, R)) % R]
    Z = [G1.add(p, g1_mul(crs.g1_gen, d)) for (p, _), d in zip(pairs, shift)]
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(1, 1, 2, rng), Z=Z)
    ppe, _ = zk_ref.augmented(a, b, gam, pairs)
    assert ogs.verify(ppe, ogs.CProof(proof[0], proof[1], [proof[2]]), crs)
    assert not statement_check(a, b, gam, pairs, proof, crs, weights(5, 2))


def test_cross_equation_cancellation_needs_independent_weights(keys):
    """+D on both coordinates of PPE''s theta_0 and -D on L_1's theta: both are paired with v_1, so the errors cancel when
    PPE' and L_1 share their weights, and are caught when the weights are drawn per equation"""
    crs = keys[0]
    rng = SeededRng(5400)
    a, b, gam, pairs, X, Y, _ = satisfied(1, 1, 1, crs, rng)
    xcoms, ycoms, pf, lin = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(1, 1, 1, rng))
    D = (g1_mul(crs.g1_gen, rng.fr()), g1_mul(crs.g1_gen, rng.fr()))
    th0 = ogs.com1_add(pf.theta[0], D)
    pf2 = ogs.EquProof(pf.pi, [th0, pf.theta[1]], pf.equ_type, pf.rand)
    lin2 = [ogs.EquProof(lin[0].pi, [ogs.com1_add(lin[0].theta[0], ogs.com1_neg(D))], lin[0].equ_type, lin[0].rand)]
    bad = (xcoms, ycoms, pf2, lin2)
    assert not zk_ref.verify(a, b, gam, pairs, bad, crs)
    st, beta = weights(6, 1)
    assert not statement_check(a, b, gam, pairs, bad, crs, (st, beta))
    assert statement_check(a, b, gam, pairs, bad, crs, ([st[0], st[0]], beta))
