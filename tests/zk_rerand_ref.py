"""Big-integer restatement of zero-knowledge PPE proof rerandomisation (gs_zk_ppe_rerandomize_batch), on the oracle's
types: the reference the zk rerandomisation tests compare against.  TEST INFRASTRUCTURE ONLY, like oracle/.

With fresh R' ((m + K) x 2), S' (n x 2), T' (2 x 2) and T'_k (1 x 2):
    PPE'  rerand_ref.rerandomize of the augmented statement (zk_ref.augmented) under R', S', T'
    L_k   delta's fresh randomness 0; Gamma = 0 and b = [1] leave fixed-base terms only:
            lin_pi'_c  = lin_pi_c + R'[m+k][c] W2 - T'_k[c] v[0]
            lin_theta' = lin_theta + T'_k[0] u[0] + T'_k[1] u[1]
The result equals zk_ref.prove (or zk_ref.simulate) under combined(...)."""
from oracle import gs as ogs
from oracle.bls12_381 import R

import rerand_ref
import zk_ref


def lin_rerandomize(p: ogs.EquProof, crs, r_row, t_k) -> ogs.EquProof:
    """L_k's proof under the row r_row of R' that moves its x-commitment and T'_k = t_k (1 x 2)"""
    w2 = ogs.w2(crs)
    pi = [ogs.com2_add(ogs.com2_add(p.pi[c], ogs.com2_scalar_mul(w2, r_row[c])), ogs.com2_scalar_mul(crs.v[0], -t_k[0][c] % R))
          for c in range(2)]
    theta = [ogs.com1_add(ogs.com1_add(p.theta[0], ogs.com1_scalar_mul(crs.u[0], t_k[0][0])), ogs.com1_scalar_mul(crs.u[1], t_k[0][1]))]
    return ogs.EquProof(pi, theta, ogs.MSMEG1, [])


def rerandomize(a, b, gamma, pairs, proof, crs, R2, S2, T2, Ts2, lin_rows=None):
    """(xcoms, ycoms, PPE' proof, [L_k proofs]) rerandomised; `lin_rows` replaces the R' rows the L_k use (default: rows
    m .. m + K - 1 of R2, the rows that move c_{m+k})"""
    xcoms, ycoms, pf, lin = proof
    m = len(b)
    ppe, _ = zk_ref.augmented(a, b, gamma, pairs)
    out = rerand_ref.rerandomize(ppe, ogs.CProof(xcoms, ycoms, [pf]), crs, R2, S2, T2)
    rows = R2[m:] if lin_rows is None else lin_rows
    return out.xcoms, out.ycoms, out.equ_proofs[0], [lin_rerandomize(p, crs, r, t) for p, r, t in zip(lin, rows, Ts2)]


def combined(a, b, gamma, pairs, rands, rands2):
    """(R + R', S + S', T + T' + S'^T Gamma'^T R, [T_k + T'_k]): the randomness of the fresh proof that equals the
    rerandomised one (Gamma' = Gamma with K zero rows)"""
    (R1, S1, T1, Ts1), (R2, S2, T2, Ts2) = rands, rands2
    ppe, _ = zk_ref.augmented(a, b, gamma, pairs)
    Rc, Sc, Tc = rerand_ref.combined_rands(ppe.gamma, R1, S1, T1, R2, S2, T2)
    return Rc, Sc, Tc, [[[(x + y) % R for x, y in zip(t1[0], t2[0])]] for t1, t2 in zip(Ts1, Ts2)]
