"""Big-integer restatement of zero-knowledge simulation with the hiding key (gs_simulate_batch), on the oracle's types: the
reference the simulation tests compare against.  TEST INFRASTRUCTURE ONLY, like oracle/.

The hiding key of generate_crs's draws (p1, p2, a1, a2, t1, t2) differs from the binding one in u[1] and v[1] only:
u[1] = (t1 p1, t1 q1 - g1), so W1 = u[1] + iota_1(g1) = t1 u[0] and likewise W2 = t2 v[0].  With R (m x cx), S (n x cy) and
T (cy x cx), the simulator outputs
    c = R u_x                  d = S v_y
    pi    = R^T iota_y(B) + (R^T Gamma S - T^T) v_y   [- t1 iota_2(T2)   MSMEG2]
    theta = S^T iota_x(A) + T u_x                     [- t2 iota_1(T1)   MSMEG1;   - t t2 W1   Quad]
which is also the reference-order prove of an augmented equation with zero witnesses and one more public variable
(`augmented`): its commitment is W2 (W1), the commitment of 0 with randomness t2 (t1)."""
from oracle import gs as ogs
from oracle.bls12_381 import G1, G2, R as ORDER, g1_mul, g2_mul


def hiding_crs(crs: ogs.CRS) -> ogs.CRS:
    """generator.rs:62-77: the binding key with u[1] - iota_1(g1) and v[1] - iota_2(g2)."""
    return ogs.CRS(u=[crs.u[0], ogs.com1_add(crs.u[1], ogs.com1_neg(ogs.com1_linear_map(crs.g1_gen)))],
                   v=[crs.v[0], ogs.com2_add(crs.v[1], ogs.com2_neg(ogs.com2_linear_map(crs.g2_gen)))],
                   g1_gen=crs.g1_gen, g2_gen=crs.g2_gen, gt_gen=crs.gt_gen)


def _shape(ty):
    return (2 if ty in (0, 1) else 1), (2 if ty in (0, 2) else 1)


def _lincomb(terms, add, smul, zero):
    acc = zero
    for com, s in terms:
        acc = add(acc, smul(com, s % ORDER))
    return acc


def simulate(equ: ogs.Equation, crs: ogs.CRS, t1, t2, xr, yr, T) -> ogs.CProof:
    """The simulator's direct formula (`crs` is the hiding key whose trapdoor is t1, t2)."""
    ty = equ.equ_type
    cx, cy = _shape(ty)
    m, n = len(equ.gamma), len(equ.gamma[0])
    c1 = lambda terms: _lincomb(terms, ogs.com1_add, ogs.com1_scalar_mul, ogs.COM1_ZERO)
    c2 = lambda terms: _lincomb(terms, ogs.com2_add, ogs.com2_scalar_mul, ogs.COM2_ZERO)
    xcoms = [c1([(crs.u[k], xr[i][k]) for k in range(cx)]) for i in range(m)]
    ycoms = [c2([(crs.v[k], yr[j][k]) for k in range(cy)]) for j in range(n)]
    iota_b = ogs._map_y(ty, equ.b_consts, crs)
    iota_a = ogs._map_x(ty, equ.a_consts, crs)
    rg = [[sum(xr[k][i] * equ.gamma[k][j] for k in range(m)) % ORDER for j in range(n)] for i in range(cx)]
    coef = [[(sum(rg[i][j] * yr[j][l] for j in range(n)) - T[l][i]) % ORDER for l in range(cy)] for i in range(cx)]
    pi = [c2([(iota_b[k], xr[k][i]) for k in range(m)] + [(crs.v[l], coef[i][l]) for l in range(cy)]) for i in range(cx)]
    theta = [c1([(iota_a[j], yr[j][i]) for j in range(n)] + [(crs.u[l], T[i][l]) for l in range(cx)]) for i in range(cy)]
    if ty == 1:
        theta[0] = ogs.com1_add(theta[0], (None, g1_mul(equ.target, (-t2) % ORDER)))
    elif ty == 2:
        pi[0] = ogs.com2_add(pi[0], (None, g2_mul(equ.target, (-t1) % ORDER)))
    elif ty == 3:
        theta[0] = ogs.com1_add(theta[0], ogs.com1_scalar_mul(ogs.w1(crs), (-equ.target * t2) % ORDER))
    return ogs.CProof(ogs.Commit(xcoms, xr), ogs.Commit(ycoms, yr), [ogs.EquProof(pi, theta, ty, T)])


def augmented(equ: ogs.Equation, t1, t2, xr, yr):
    """(equation, xvars, yvars, x_rand, y_rand) of the augmented statement whose reference-order prove with zero
    witnesses is the simulated proof: one more y-variable with randomness [t2] and constant -T1 / -t (MSMEG1 / Quad), one
    more x-variable with randomness [t1] and constant -T2 (MSMEG2), Gamma padded with zeros; PPE is unchanged."""
    ty = equ.equ_type
    m, n = len(equ.gamma), len(equ.gamma[0])
    zero_x, zero_y = (None if ty in (0, 1) else 0), (None if ty in (0, 2) else 0)
    a, b, gam = list(equ.a_consts), list(equ.b_consts), [list(r) for r in equ.gamma]
    xr, yr = [list(r) for r in xr], [list(r) for r in yr]
    if ty == 1:
        a.append(G1.neg(equ.target))
    elif ty == 3:
        a.append((-equ.target) % ORDER)
    if ty in (1, 3):
        gam = [r + [0] for r in gam]
        yr.append([t2])
        n += 1
    if ty == 2:
        b.append(G2.neg(equ.target))
        gam.append([0] * n)
        xr.append([t1])
        m += 1
    return ogs.Equation(ty, a, b, gam, equ.target), [zero_x] * m, [zero_y] * n, xr, yr
