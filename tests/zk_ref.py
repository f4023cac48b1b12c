"""Big-integer restatement of zero-knowledge proofs of PPEs with targets given as pairs (gs_zk_ppe_*_batch), on the
oracle's types: the reference the zero-knowledge tests compare against.  TEST INFRASTRUCTURE ONLY, like oracle/.

A PPE  sum_j e(A_j, Y_j) + sum_i e(X_i, B_i) + sum_ij gamma_ij e(X_i, Y_j) = sum_k e(P_k, Q_k)  becomes
    PPE'  target 1 over the x-variables (X | Z), constants (B | -Q), Gamma with K zero rows
    L_k   the MSMEG1 equation Z_k - delta P_k = O  (a = [-P_k], b = [1], Gamma = [[0]])
where delta's commitment is fixed to W2 = 1 W2 + 0 v[0], taken from the CRS by the verifier.  The real prover proves
(X, Y, Z = P, delta = 1); the simulator proves (O, O, Z = O, delta = 0) with delta's randomness t2 (under the hiding key
W2 = t2 v[0]), i.e. PPE' through simulate_ref.simulate with target 1 and L_k as the prover with y_rand [t2]."""
from oracle import gs as ogs
from oracle.bls12_381 import FP12_ONE, G1, G2

import simulate_ref


def augmented(a, b, gamma, pairs):
    """(PPE', [L_1..L_K]) as oracle Equations"""
    n, K = len(a), len(pairs)
    ppe = ogs.Equation(0, list(a), list(b) + [G2.neg(q) for _, q in pairs], [list(r) for r in gamma] + [[0] * n for _ in range(K)],
                       FP12_ONE)
    return ppe, [ogs.Equation(1, [G1.neg(p)], [1], [[0]], None) for p, _ in pairs]


def lin_coms(xcoms: ogs.Commit, m, k, crs, delta_com=None):
    """(x-commitments, y-commitments) of L_k: [c_{m+k}] and [W2] (or another delta commitment)"""
    return (ogs.Commit([xcoms.coms[m + k]], [xcoms.rand[m + k]] if xcoms.rand else []),
            ogs.Commit([delta_com or ogs.w2(crs)], [[0]]))


def prove(a, b, gamma, pairs, X, Y, crs, R, S, T, Ts, Z=None):
    """(xcoms, ycoms, PPE' proof, [L_k proofs]) of the real prover; Z (default P) are the values committed as Z_k"""
    m = len(b)
    Z = [p for p, _ in pairs] if Z is None else Z
    ppe, lins = augmented(a, b, gamma, pairs)
    xcoms = ogs.batch_commit_g1(list(X) + list(Z), crs, R)
    ycoms = ogs.batch_commit_g2(list(Y), crs, S)
    pf = ogs.prove(ppe, list(X) + list(Z), list(Y), xcoms, ycoms, crs, T)
    lin = []
    for k, (L, z) in enumerate(zip(lins, Z)):
        xc, _ = lin_coms(xcoms, m, k, crs)
        lin.append(ogs.prove(L, [z], [1], xc, ogs.Commit([ogs.w2(crs)], [[0]]), crs, Ts[k]))
    return xcoms, ycoms, pf, lin


def simulate(a, b, gamma, pairs, hid, t1, t2, R, S, T, Ts):
    """the simulator's output under the hiding key `hid` with trapdoor (t1, t2): no witness"""
    m = len(b)
    ppe, lins = augmented(a, b, gamma, pairs)
    sim = simulate_ref.simulate(ppe, hid, t1, t2, R, S, T)
    lin = []
    for k, L in enumerate(lins):
        xc = ogs.Commit([sim.xcoms.coms[m + k]], [R[m + k]])
        lin.append(ogs.prove(L, [None], [0], xc, ogs.Commit([ogs.w2(hid)], [[t2]]), hid, Ts[k]))
    return sim.xcoms, sim.ycoms, sim.equ_proofs[0], lin


def verify(a, b, gamma, pairs, proof, crs, delta_com=None):
    """PPE' on (c, d, pi, theta) and every L_k on ([c_{m+k}], [W2]); `delta_com` replaces W2 (a forged delta)"""
    xcoms, ycoms, pf, lin = proof
    m = len(b)
    ppe, lins = augmented(a, b, gamma, pairs)
    if not ogs.verify(ppe, ogs.CProof(xcoms, ycoms, [pf]), crs):
        return False
    for k, (L, p) in enumerate(zip(lins, lin)):
        xc, yc = lin_coms(xcoms, m, k, crs, delta_com)
        if not ogs.verify(L, ogs.CProof(xc, yc, [p]), crs):
            return False
    return True
