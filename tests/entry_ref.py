"""Proofs that are wrong in a chosen ComT entry, and the per-entry comparison that confirms it.  TEST INFRASTRUCTURE ONLY.

A verifier decides a proof from the 2 x 2 matrix of GT values D = LHS - RHS (written additively, in the exponent of
gt_gen = e(g1, g2)) of verifier.rs:23-157.  Every element of a case here is a known multiple of the CRS generators: the CRS
comes from make_crs's draws (p1, p2, a1, a2, t1, t2), witnesses and constants are seeded scalars (bigcase.py), commitments
have known randomness.  So D is linear in what a tamper changes:
    Gamma_ij += gamma        adds  gamma * (c_i (x) d_j)      (the discrete logs of the two commitments)
    theta_0.a += eps_a g1    adds  -eps (x) v_0               (v_0 = (1, a2) under both keys)
    pi_0.b    += eta_b g2    adds  -u_0 (x) eta               (u_0 = (1, a1))
The theta_0 / pi_0 changes span the 3-dimensional kernel of f(M) = M11 - a2 M10 - a1 M01 + a1 a2 M00 -- the binding
property -- so the Gamma step carries f(E) and then eps, eta give exactly D = E, for any 2 x 2 matrix E.  Under the hiding
key theta_1 / pi_1 (along v_1, u_1) reach outside the kernel too, except for Quad (see `reachable`).  Gamma, theta and pi
belong to one equation, so the same works for one equation of a statement over shared commitments."""
from bigcase import *  # noqa: F401,F403
from oracle import gs as ogs
from oracle.bls12_381 import FP12_ONE, G1, G2, final_exponentiation

import simulate_ref
from test_randfold_each_oracle import XA


class Key:
    """Discrete logs of the binding key of make_crs's draws, or of its hiding key (simulate_ref.hiding_crs)."""

    def __init__(self, draws, hiding=False):
        _, _, a1, a2, t1, t2 = draws
        crs = ogs.generate_crs(*draws)
        self.crs = simulate_ref.hiding_crs(crs) if hiding else crs
        self.crsb = crs_bytes(self.crs)
        self.a1, self.a2, self.hiding = a1, a2, hiding
        h = 1 if hiding else 0
        self.u = [(1, a1), (t1, (a1 * t1 - h) % R)]
        self.v = [(1, a2), (t2, (a2 * t2 - h) % R)]
        self.w1 = (t1, (a1 * t1 - h + 1) % R)              # u[1] + iota_1(g1)
        self.w2 = (t2, (a2 * t2 - h + 1) % R)

    def com_x(self, ty, x, r):
        """discrete logs of the x-commitment of x with randomness r (cx scalars)"""
        if ty in (0, 1):
            return ((r[0] + r[1] * self.u[1][0]) % R, (r[0] * self.a1 + r[1] * self.u[1][1] + x) % R)
        return ((x * self.w1[0] + r[0]) % R, (x * self.w1[1] + r[0] * self.a1) % R)

    def com_y(self, ty, y, s):
        if ty in (0, 2):
            return ((s[0] + s[1] * self.v[1][0]) % R, (s[0] * self.a2 + s[1] * self.v[1][1] + y) % R)
        return ((y * self.w2[0] + s[0]) % R, (y * self.w2[1] + s[0] * self.a2) % R)


def unit(e, lam=1):
    """lam E_e: the error lam in entry e = (e // 2, e % 2) only"""
    E = [[0, 0], [0, 0]]
    E[e // 2][e % 2] = lam % R
    return E


def reachable(key, ty):
    """False where no change of Gamma, theta or pi leaves the kernel of f: Quad under the hiding key, where W1 = t1 u_0 and
    W2 = t2 v_0 put every commitment, constant and target term of the equation into it (the zero-knowledge property)"""
    return not (ty == 3 and key.hiding)


def errors(key, ty, lam=1):
    """the error matrices the tests plant: lam in one entry, for each entry; where single entries are not reachable, the
    row errors e_a (x) v_0 and column errors u_0 (x) e_b (entries {0, 1}, {2, 3}, {0, 2}, {1, 3})"""
    if reachable(key, ty):
        return [unit(e, lam) for e in range(4)]
    u0, v0 = key.u[0], key.v[0]
    return [[[lam * v0[b] * (a == r) % R for b in range(2)] for a in range(2)] for r in range(2)] + \
           [[[lam * u0[a] * (b == t) % R for b in range(2)] for a in range(2)] for t in range(2)]


def solve(key, ty, c, d, E):
    """(gamma, theta deltas [row][coordinate], pi deltas [column][coordinate]) with
    gamma c (x) d - sum_k eps_k (x) v_k - sum_k u_k (x) eta_k = E,  k over the theta rows / pi columns of type ty.
    Gamma comes first, so it carries the part outside the kernel of f whenever it can (the binding key); under the hiding
    key the second theta row / pi column, along v_1 / u_1, can do that as well."""
    cx, cy = cb.cx_of(ty), cb.cy_of(ty)
    cols = [[c[a] * d[b] % R for a in range(2) for b in range(2)]]
    for k in range(cy):
        cols += [[-(a == t) * key.v[k][b] % R for a in range(2) for b in range(2)] for t in range(2)]
    for k in range(cx):
        cols += [[-key.u[k][a] * (b == t) % R for a in range(2) for b in range(2)] for t in range(2)]
    rows = [[col[r] for col in cols] + [E[r // 2][r % 2] % R] for r in range(4)]
    piv, r = [], 0
    for col in range(len(cols)):
        p = next((i for i in range(r, 4) if rows[i][col]), None)
        if p is None:
            continue
        rows[r], rows[p] = rows[p], rows[r]
        inv = pow(rows[r][col], -1, R)
        rows[r] = [x * inv % R for x in rows[r]]
        for i in range(4):
            if i != r and rows[i][col]:
                f = rows[i][col]
                rows[i] = [(x - f * y) % R for x, y in zip(rows[i], rows[r])]
        piv.append(col)
        r += 1
    if any(row[-1] for row in rows[r:]):
        raise ValueError("E is not reachable through Gamma, theta and pi")
    z = [0] * len(cols)
    for i, col in enumerate(piv):
        z[col] = rows[i][-1]
    return z[0], [z[1 + 2 * k:3 + 2 * k] for k in range(cy)], [z[1 + 2 * cy + 2 * k:3 + 2 * cy + 2 * k] for k in range(cx)]


def _add1(b, k, g):
    return g1_b(G1.add(g1_i(b), g1_mul(g, k))) if k else b


def _add2(b, k, g):
    return g2_b(G2.add(g2_i(b), g2_mul(g, k))) if k else b


def tamper_arrays(key, ty, m, n, gamma, pi, theta, c, d, E, eq=0, i=0, j=0):
    """(gamma, pi, theta) of a batch with equation `eq` changed so that its error matrix becomes E; c, d: the discrete logs
    of that equation's c_i and d_j"""
    g, eps, eta = solve(key, ty, c, d, E)
    cx, cy = cb.cx_of(ty), cb.cy_of(ty)
    gb = bytearray(gamma)
    o = 32 * ((eq * m + i) * n + j)
    gb[o:o + 32] = fr_b((fr_i(bytes(gb[o:o + 32])) + g) % R)
    pb = bytearray(pi)
    for k in range(cx):
        for b in range(2):
            o = (eq * cx + k) * 384 + 192 * b
            pb[o:o + 192] = _add2(bytes(pb[o:o + 192]), eta[k][b], key.crs.g2_gen)
    tb = bytearray(theta)
    for k in range(cy):
        for a in range(2):
            o = (eq * cy + k) * 192 + 96 * a
            tb[o:o + 96] = _add1(bytes(tb[o:o + 96]), eps[k][a], key.crs.g1_gen)
    return bytes(gb), bytes(pb), bytes(tb)


def _rand_rows(buf, k):
    s = [fr_i(buf[32 * t:32 * (t + 1)]) for t in range(len(buf) // 32)]
    return [s[r * k:(r + 1) * k] for r in range(len(s) // k)]


def com_logs(key, case):
    """discrete logs of a Case's / Statement's commitments (c, d)"""
    ty = case.ty
    xr, yr = _rand_rows(case.xr, cb.cx_of(ty)), _rand_rows(case.yr, cb.cy_of(ty))
    return ([key.com_x(ty, x, r) for x, r in zip(case.xs, xr)], [key.com_y(ty, y, s) for y, s in zip(case.ys, yr)])


def tamper(key, case, E, eq=0, i=0, j=0, arrays=None):
    """the verify arrays of a bigcase.Case (eq = 0) or Statement (equation eq) whose error matrix is E (`arrays`: the
    case's arrays with other equations changed already)"""
    arrays = list(arrays or case.verify_arrays())
    c, d = com_logs(key, case)
    arrays[2], arrays[6], arrays[7] = tamper_arrays(key, case.ty, case.m, case.n, arrays[2], arrays[6], arrays[7], c[i], d[j],
                                                    E, eq, i, j)
    return arrays


# ---------------------------------------------------------------- the oracle's view, entry by entry
def oracle_form(ty, m, n, arrays, p=0):
    """(Equation, CProof) of proof p of a batch in gs_verify_batch layout"""
    sz = [n * cb.x_size(ty), m * cb.y_size(ty), m * n * 32, cb.target_size(ty), m * 192, n * 384, cb.cx_of(ty) * 384,
          cb.cy_of(ty) * 192]
    A, B, G, T, xc, yc, pi, th = [a[p * s:(p + 1) * s] for a, s in zip(arrays, sz)]
    cut = lambda b, k: [b[t:t + k] for t in range(0, len(b), k)]
    a = [g1_i(x) for x in cut(A, 96)] if ty in (0, 1) else [fr_i(x) for x in cut(A, 32)]
    b = [g2_i(y) for y in cut(B, 192)] if ty in (0, 2) else [fr_i(y) for y in cut(B, 32)]
    gam = [[fr_i(G[32 * (r * n + k):32 * (r * n + k + 1)]) for k in range(n)] for r in range(m)]
    t = {0: fp12_i, 1: g1_i, 2: g2_i, 3: fr_i}[ty](T)
    proof = ogs.CProof(ogs.Commit([com1_i(x) for x in cut(xc, 192)], []), ogs.Commit([com2_i(y) for y in cut(yc, 384)], []),
                       [ogs.EquProof([com2_i(x) for x in cut(pi, 384)], [com1_i(x) for x in cut(th, 192)], ty, [])])
    return ogs.Equation(ty, a, b, gam, t), proof


def entries(equ, proof, crs):
    """[(LHS_e, RHS_e) for e = 0..3]: ogs.verify's two ComT values, entry by entry"""
    ty = equ.equ_type
    ep = proof.equ_proofs[0]
    lhs = ogs.comt_add(ogs.comt_add(ogs.comt_pairing_sum(ogs._map_x(ty, equ.a_consts, crs), proof.ycoms.coms),
                                    ogs.comt_pairing_sum(proof.xcoms.coms, ogs._map_y(ty, equ.b_consts, crs))),
                       ogs.comt_pairing_sum(proof.xcoms.coms, ogs.col_vec_to_vec(
                           ogs.com_left_mul(ogs.vec_to_col_vec(proof.ycoms.coms), equ.gamma, 2))))
    lin_t = [lambda: ogs.comt_linear_map_ppe(equ.target), lambda: ogs.comt_linear_map_msmeg1(equ.target, crs),
             lambda: ogs.comt_linear_map_msmeg2(equ.target, crs), lambda: ogs.comt_linear_map_quad(equ.target, crs)][ty]()
    com1_pf2 = ogs.comt_pairing_sum(crs.u, ep.pi) if ty in (0, 1) else ogs.comt_pairing(crs.u[0], ep.pi[0])
    pf1_com2 = ogs.comt_pairing_sum(ep.theta, crs.v) if ty in (0, 2) else ogs.comt_pairing(ep.theta[0], crs.v[0])
    rhs = ogs.comt_add(ogs.comt_add(lin_t, com1_pf2), pf1_com2)
    return list(zip(lhs, rhs))


def ratios(equ, proof, crs):
    """LHS_e / RHS_e for e = 0..3: gt_gen^E[e] for a proof whose error matrix is E"""
    return [l * r.inv() for l, r in entries(equ, proof, crs)]


def gt_of(crs, E):
    return [crs.gt_gen.pow(E[e // 2][e % 2]) for e in range(4)]


def finish(partials, p, count):
    """the four final-exponentiated entries of statement p from the ranks' gs_verify_partial outputs (rank-major,
    [p][e] within a rank): the product of the ranks' Miller partials, then the final exponentiation"""
    nparts = len(partials) // (count * 2304)
    out = []
    for e in range(4):
        f = FP12_ONE
        for r in range(nparts):
            o = (r * count + p) * 2304 + e * 576
            f = f * fp12_i(partials[o:o + 576])
        out.append(final_exponentiation(f))
    return out


# ---------------------------------------------------------------- the weights of the randomised verifiers
M63 = (1 << 63) - 1


def rho_words(rho):
    return [int.from_bytes(rho[8 * k:8 * (k + 1)], "little") for k in range(len(rho) // 8)]


def weights_of(rho, p, count):
    """(sigma_p, tau_p, beta) as the GPU takes them from rho: rho[2p], rho[2p + 1] masked to 63 bits, beta = lo32 + hi32 |x|
    of rho[2 count] (verify.cu rand_weights / rand_beta)"""
    w = rho_words(rho)
    word = w[2 * count]
    return w[2 * p] & M63, w[2 * p + 1] & M63, ((word & 0xFFFFFFFF) + (word >> 32) * XA) % R


def weight_cancelling(sg, tu, beta):
    """E = E00 - (sigma beta / tau) E11: sigma beta E00 + sigma E01 + tau beta E10 + tau E11 = 0, so the fold with exactly
    these weights cannot see it, while any other sigma, tau or beta can (each one appears in the cancelling term)"""
    assert tu % R
    return [[1, 0], [0, (-sg * beta * pow(tu, -1, R)) % R]]


def flip_bit(rho, word, bit):
    b = bytearray(rho)
    b[8 * word + bit // 8] ^= 1 << (bit % 8)
    return bytes(b)
