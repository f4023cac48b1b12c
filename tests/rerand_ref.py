"""Big-integer restatement of proof rerandomisation (gs_rerandomize_batch), on the oracle's types: the reference the
rerandomisation tests compare against.  TEST INFRASTRUCTURE ONLY, like oracle/.

With fresh R' (m x cx), S' (n x cy) and T' (cy x cx, the layout of pf_rand):
    c' = c + R' u_x                     d' = d + S' v_y
    pi'    = pi    + R'^T iota_y(B) + (R'^T Gamma) d + (R'^T Gamma S' - T'^T) v_y
    theta' = theta + S'^T iota_x(A) + (S'^T Gamma^T) c + T' u_x
pi' and theta' use the OLD c and d.  The result equals commit_and_prove of the same witnesses under
combined_rands(...)."""
from oracle import gs as ogs
from oracle.bls12_381 import R


def _col(v): return ogs.vec_to_col_vec(v)


def _add_vec(a, b, which):
    add = ogs.com1_add if which == 1 else ogs.com2_add
    return [add(x, y) for x, y in zip(a, b)]


def rerandomize(equ: ogs.Equation, proof: ogs.CProof, crs: ogs.CRS, x_rand2, y_rand2, pf_rand2) -> ogs.CProof:
    ty = equ.equ_type
    cx = 2 if ty in (ogs.PPE, ogs.MSMEG1) else 1
    cy = 2 if ty in (ogs.PPE, ogs.MSMEG2) else 1
    c, d = proof.xcoms.coms, proof.ycoms.coms
    ep = proof.equ_proofs[0]
    assert (len(x_rand2), len(x_rand2[0])) == (len(c), cx) and (len(y_rand2), len(y_rand2[0])) == (len(d), cy)
    assert (len(pf_rand2), len(pf_rand2[0])) == (cy, cx)
    ux, vy = crs.u[:cx], crs.v[:cy]
    xc = _add_vec(c, ogs.col_vec_to_vec(ogs.com_left_mul(_col(ux), x_rand2, 1)), 1)
    yc = _add_vec(d, ogs.col_vec_to_vec(ogs.com_left_mul(_col(vy), y_rand2, 2)), 2)

    rt = ogs.fr_transpose(x_rand2)
    rg = ogs.fr_right_mul(rt, equ.gamma)
    coef = ogs.fr_add(ogs.fr_right_mul(rg, y_rand2), ogs.fr_neg(ogs.fr_transpose(pf_rand2)))
    pi = ep.pi
    for term in (ogs.com_left_mul(_col(ogs._map_y(ty, equ.b_consts, crs)), rt, 2), ogs.com_left_mul(_col(d), rg, 2),
                 ogs.com_left_mul(_col(vy), coef, 2)):
        pi = _add_vec(pi, [row[0] for row in term], 2)

    st = ogs.fr_transpose(y_rand2)
    sg = ogs.fr_right_mul(st, ogs.fr_transpose(equ.gamma))
    theta = ep.theta
    for term in (ogs.com_left_mul(_col(ogs._map_x(ty, equ.a_consts, crs)), st, 1), ogs.com_left_mul(_col(c), sg, 1),
                 ogs.com_left_mul(_col(ux), pf_rand2, 1)):
        theta = _add_vec(theta, [row[0] for row in term], 1)
    return ogs.CProof(ogs.Commit(xc, []), ogs.Commit(yc, []), [ogs.EquProof(pi, theta, ty, [])])


def combined_rands(gamma, x_rand, y_rand, pf_rand, x_rand2, y_rand2, pf_rand2):
    """(R + R', S + S', T + T' + S'^T Gamma^T R): the randomness under which a fresh proof equals the rerandomised one."""
    add = lambda a, b: [[(x + y) % R for x, y in zip(ra, rb)] for ra, rb in zip(a, b)]
    sgr = ogs.fr_right_mul(ogs.fr_right_mul(ogs.fr_transpose(y_rand2), ogs.fr_transpose(gamma)), x_rand)
    return add(x_rand, x_rand2), add(y_rand, y_rand2), add(add(pf_rand, pf_rand2), sgr)
