"""gs_zk_ppe_prove_batch / _simulate_batch / _verify_batch on the GPU, through the C ABI.  Each output is compared byte for
byte with the composition of existing entry points on the augmented statement (PPE' with target 1, the K equations
Z_k - delta P_k = O), and the first and last statement of a batch with the C oracle's prove of the augmented equations.
Witnesses, constants and target pairs are multiples of the generators with known discrete logs (bigcase.py)."""
import ctypes

import pytest

from bigcase import *  # noqa: F401,F403
from simulate_ref import hiding_crs

pytestmark = pytest.mark.gpu

OK, EDIM, EARG = 0, 1, 3
vp = ctypes.c_void_p
ONE, ZERO_FR = fr_b(1), fr_b(0)


@pytest.fixture(scope="module")
def keys():
    crs, (_, _, _, _, t1, t2) = make_crs(3)
    return crs, hiding_crs(crs), t1, t2


@pytest.fixture(scope="module")
def eng():
    import groth_sahai_rs_b200 as gsb
    e = gsb.Engine(0)
    yield e
    e.close()


def cut(b, size):
    return [b[i:i + size] for i in range(0, len(b), size)]


class ZkCase:
    """E statements of shape (m, n, K); `true_targets`: the pairs multiply to the value of the witnesses, else random"""

    def __init__(self, m, n, K, crs, seed, E=1, true_targets=True):
        rng = SeededRng(seed)
        self.m, self.n, self.K, self.E = m, n, K, E
        a, b, xs, ys = fr_list(rng, E * n), fr_list(rng, E * m), fr_list(rng, E * m), fr_list(rng, E * n)
        gam = [[fr_list(rng, n) for _ in range(m)] for _ in range(E)]
        ps, qs = fr_list(rng, E * K), fr_list(rng, E * K)
        if true_targets:
            for i in range(E):
                val = sum(a[i * n + j] * ys[i * n + j] for j in range(n)) + sum(xs[i * m + k] * b[i * m + k] for k in range(m)) + \
                    sum(gam[i][k][j] * xs[i * m + k] * ys[i * n + j] for k in range(m) for j in range(n))
                rest = (val - sum(ps[i * K + k] * qs[i * K + k] for k in range(K - 1))) % R
                qs[i * K + K - 1] = rest * pow(ps[i * K + K - 1], -1, R) % R
        g1s = g1_multiples(crs, a + xs + ps + [(-p) % R for p in ps])
        g2s = g2_multiples(crs, b + ys + qs + [(-q) % R for q in qs])
        self.A, self.X = b"".join(g1s[:E * n]), b"".join(g1s[E * n:E * (n + m)])
        self.P, self.negP = g1s[E * (n + m):E * (n + m + K)], g1s[E * (n + m + K):]
        self.B, self.Y = b"".join(g2s[:E * m]), b"".join(g2s[E * m:E * (m + n)])
        self.Q, self.negQ = g2s[E * (m + n):E * (m + n + K)], g2s[E * (m + n + K):]
        self.G = b"".join(frmat_b(g) for g in gam)
        self.gam, self.xs, self.ys = gam, xs, ys
        self.xr, self.yr = fr_list(rng, E * (m + K) * 2), fr_list(rng, E * n * 2)
        self.Tr, self.Lr = fr_list(rng, E * 4), fr_list(rng, E * K * 2)

    def stmt(self):
        return self.A, self.B, self.G, b"".join(self.P), b"".join(self.Q)

    def rand(self):
        return frs_b(self.xr), frs_b(self.yr), frs_b(self.Tr), frs_b(self.Lr)

    # ---- the augmented statement, built here without the code under test
    def x_and_p(self, i):
        m, K = self.m, self.K
        return self.X[i * m * 96:(i + 1) * m * 96] + b"".join(self.P[i * K:(i + 1) * K])

    def ppe_prime(self):
        """(a, b', Gamma') of every statement"""
        m, n, K, E = self.m, self.n, self.K, self.E
        b = b"".join(self.B[i * m * 192:(i + 1) * m * 192] + b"".join(self.negQ[i * K:(i + 1) * K]) for i in range(E))
        g = b"".join(frmat_b(self.gam[i] + [[0] * n] * K) for i in range(E))
        return self.A, b, g

    def lin(self):
        """(a, b, Gamma, Z-randomness) of the E K equations L_k"""
        m, K = self.m, self.K
        zr = b"".join(frs_b(self.xr[(i * (m + K) + m + k) * 2:(i * (m + K) + m + k) * 2 + 2]) for i in range(self.E) for k in range(K))
        return b"".join(self.negP), ONE * self.E * K, ZERO_FR * self.E * K, zr


def composition_prove(eng, c):
    m, n, K, E = c.m, c.n, c.K, c.E
    xp = b"".join(c.x_and_p(i) for i in range(E))
    xr, yr, Tr, Lr = c.rand()
    xc, yc = eng.batch_commit_g1(xp, xr), eng.batch_commit_g2(c.Y, yr)
    pi, th = eng.prove_batch(0, E, m + K, n, *c.ppe_prime(), xp, c.Y, xr, yr, Tr)
    la, lb, lg, zr = c.lin()
    lpi, lth = eng.prove_batch(1, E * K, 1, 1, la, lb, lg, b"".join(c.P), ONE * E * K, zr, ZERO_FR * E * K, Lr)
    return xc, yc, pi, th, lpi, lth


def oracle_prove(c, crsb, i):
    """the C oracle's commit + prove of statement i's augmented equations"""
    m, n, K = c.m, c.n, c.K
    _, b, g = c.ppe_prime()
    xr, yr = frs_b(c.xr[i * (m + K) * 2:(i + 1) * (m + K) * 2]), frs_b(c.yr[i * n * 2:(i + 1) * n * 2])
    Y = c.Y[i * n * 192:(i + 1) * n * 192]
    xc, yc = cb.commit_x(0, c.x_and_p(i), xr, crsb, NT), cb.commit_y(0, Y, yr, crsb, NT)
    pi, th = cb.prove(0, m + K, n, c.A[i * n * 96:(i + 1) * n * 96], b[i * (m + K) * 192:(i + 1) * (m + K) * 192],
                      g[i * (m + K) * n * 32:(i + 1) * (m + K) * n * 32], c.x_and_p(i), Y, xr, yr,
                      frs_b(c.Tr[i * 4:(i + 1) * 4]), crsb, NT)
    lpi, lth = b"", b""
    for k in range(K):
        j = i * K + k
        p, t = cb.prove(1, 1, 1, c.negP[j], ONE, ZERO_FR, c.P[j], ONE, frs_b(c.xr[(i * (m + K) + m + k) * 2:][:2]), ZERO_FR,
                        frs_b(c.Lr[j * 2:j * 2 + 2]), crsb, NT)
        lpi, lth = lpi + p, lth + t
    return xc, yc, pi, th, lpi, lth


def statement_of(out, c, i):
    m, n, K = c.m, c.n, c.K
    sizes = ((m + K) * 192, n * 384, 768, 384, K * 768, K * 192)
    return tuple(o[i * s:(i + 1) * s] for o, s in zip(out, sizes))


@pytest.mark.parametrize("m,n,K", [(1, 1, 1), (4, 4, 1), (4, 4, 2), (4, 4, 3), (1, 4, 1)])
def test_real_proofs_equal_the_composition_and_verify(eng, keys, m, n, K):
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    c = ZkCase(m, n, K, crs, seed=3000 + 100 * m + 10 * n + K, E=3)
    out = eng.zk_ppe_prove_batch(c.E, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())
    assert out == composition_prove(eng, c)
    for i in (0, c.E - 1):
        assert statement_of(out, c, i) == oracle_prove(c, crs_bytes(crs), i), f"statement {i}"
    assert eng.zk_ppe_verify_batch(c.E, m, n, K, *c.stmt(), *out) == b"\x01" * c.E
    # the other statements' pairs: the targets no longer hold
    shifted = (c.A, c.B, c.G, b"".join(c.P[K:] + c.P[:K]), b"".join(c.Q[K:] + c.Q[:K]))
    assert eng.zk_ppe_verify_batch(c.E, m, n, K, *shifted, *out) == b"\x00" * c.E


@pytest.mark.parametrize("K", [1, 2])
def test_simulated_proofs_equal_the_composition_and_verify_for_false_targets(eng, keys, K):
    crs, hid, t1, t2 = keys
    eng.crs_load(crs_bytes(hid))
    m = n = 4
    c = ZkCase(m, n, K, hid, seed=3100 + K, E=3, true_targets=False)
    tkey = fr_b(t1) + fr_b(t2)
    xr, yr, Tr, Lr = c.rand()
    out = eng.zk_ppe_simulate_batch(c.E, m, n, K, *c.stmt(), xr, yr, Tr, Lr, tkey)
    ppe = eng.simulate_batch(0, c.E, m + K, n, *c.ppe_prime(), fp12_b(FP12_ONE) * c.E, xr, yr, Tr, tkey)
    la, lb, lg, zr = c.lin()
    lin = eng.simulate_batch(1, c.E * K, 1, 1, la, lb, lg, bytes(96) * c.E * K, zr, fr_b(t2) * c.E * K, Lr, tkey)
    assert out == ppe + lin[2:]
    assert eng.zk_ppe_verify_batch(c.E, m, n, K, *c.stmt(), *out) == b"\x01" * c.E
    eng.crs_load(crs_bytes(crs))
    assert eng.zk_ppe_verify_batch(c.E, m, n, K, *c.stmt(), *out) == b"\x00" * c.E


def test_verdicts_are_the_and_of_the_pieces_under_tampering(eng, keys):
    """6,000 statements (two verify passes of PPE' and of the 12,000 L_k; then again in upload chunks of 480 statements),
    64 distinct ones tiled, one tamper per statement from a mask: every proof element, an X and a Z commitment, a y
    commitment, an L_k proved with y_rand 1 (delta's commitment then is not W2), the target pairs of another statement;
    verdicts equal the AND of gs_verify_batch on PPE' and on every L_k with the commitments [c_{m+k}], [W2]."""
    import random
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    m, n, K, E0, E = 2, 2, 2, 64, 6000
    base = ZkCase(m, n, K, crs, seed=3200, E=E0)
    c = ZkCase.__new__(ZkCase)
    c.m, c.n, c.K, c.E = m, n, K, E
    tile = lambda b, per: b"".join(b[(i % E0) * per:(i % E0 + 1) * per] for i in range(E))
    c.A, c.X, c.B, c.Y, c.G = tile(base.A, n * 96), tile(base.X, m * 96), tile(base.B, m * 192), tile(base.Y, n * 192), \
        tile(base.G, m * n * 32)
    c.gam = [base.gam[i % E0] for i in range(E)]
    c.P, c.negP = [base.P[(i % E0) * K + k] for i in range(E) for k in range(K)], [base.negP[(i % E0) * K + k] for i in range(E) for k in range(K)]
    c.Q, c.negQ = [base.Q[(i % E0) * K + k] for i in range(E) for k in range(K)], [base.negQ[(i % E0) * K + k] for i in range(E) for k in range(K)]
    rng = SeededRng(3201)
    c.xr, c.yr, c.Tr, c.Lr = fr_list(rng, E * (m + K) * 2), fr_list(rng, E * n * 2), fr_list(rng, E * 4), fr_list(rng, E * K * 2)
    out = [bytearray(o) for o in eng.zk_ppe_prove_batch(E, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())]
    la, lb, lg, zr = c.lin()
    # L_k proved with delta's randomness 1 instead of 0
    bad_pi, bad_th = eng.prove_batch(1, E * K, 1, 1, la, lb, lg, b"".join(c.P), ONE * E * K, zr, ONE * E * K, frs_b(c.Lr))
    P, Q = list(c.P), list(c.Q)
    sizes = ((m + K) * 192, n * 384, 768, 384, K * 768, K * 192)
    mask = random.Random(3202).choices(range(10), k=E)
    for i, t in enumerate(mask):
        j = (i + 1) % E     # a statement with other values (E0 does not divide 1)
        if t <= 5:          # 0: X commitment, 1: y commitment, 2: pi, 3: theta, 4: lin_pi, 5: lin_theta
            s = sizes[t]
            out[t][i * s:i * s + 192] = out[t][j * s:j * s + 192]
        elif t == 6:        # the commitment of Z_K
            s = sizes[0]
            at = i * s + (m + K - 1) * 192
            out[0][at:at + 192] = out[0][j * s + (m + K - 1) * 192:j * s + (m + K) * 192]
        elif t == 7:        # L_1 proved with y_rand 1
            out[4][i * K * 768:i * K * 768 + 768] = bad_pi[i * K * 768:i * K * 768 + 768]
            out[5][i * K * 192:i * K * 192 + 192] = bad_th[i * K * 192:i * K * 192 + 192]
        elif t == 8:        # target pairs exchanged with the next statement
            P[i * K:(i + 1) * K], Q[i * K:(i + 1) * K] = c.P[j * K:(j + 1) * K], c.Q[j * K:(j + 1) * K]
        # t == 9: untouched
    out = [bytes(o) for o in out]
    c.P, c.Q = P, Q
    got = eng.zk_ppe_verify_batch(E, m, n, K, *c.stmt(), *out)
    # the pieces: PPE' of the (possibly exchanged) pairs, and every L_k on [c_{m+k}], [W2]
    negP = {p: q for p, q in zip(base.P, base.negP)}
    negQ = {p: q for p, q in zip(base.Q, base.negQ)}
    c.negP, c.negQ = [negP[p] for p in P], [negQ[q] for q in Q]
    ok_ppe = eng.verify_batch(0, E, m + K, n, *c.ppe_prime(), fp12_b(FP12_ONE) * E, out[0], out[1], out[2], out[3])
    la, lb, lg, _ = c.lin()
    zc = b"".join(out[0][i * sizes[0] + (m + k) * 192:i * sizes[0] + (m + k + 1) * 192] for i in range(E) for k in range(K))
    ok_lin = eng.verify_batch(1, E * K, 1, 1, la, lb, lg, bytes(96) * E * K, zc, com2_b(ogs.w2(crs)) * E * K, out[4], out[5])
    want = bytes(ok_ppe[i] & min(ok_lin[i * K:(i + 1) * K]) for i in range(E))
    assert got == want
    assert all(got[i] == (1 if t == 9 else 0) for i, t in enumerate(mask))
    # the same call with passes of 240 problems: the statements are uploaded in chunks of 4 * 240 / K = 480 (12 full
    # chunks and a partial one), and the verdicts do not change
    import os
    import groth_sahai_rs_b200 as gsb
    old = os.environ.get("GS_VERIFY_BATCH_MAX")
    os.environ["GS_VERIFY_BATCH_MAX"] = "240"
    try:
        small = gsb.Engine(0)
    finally:
        os.environ.pop("GS_VERIFY_BATCH_MAX", None) if old is None else os.environ.__setitem__("GS_VERIFY_BATCH_MAX", old)
    small.crs_load(crs_bytes(crs))
    assert small.zk_ppe_verify_batch(E, m, n, K, *c.stmt(), *out) == got
    small.close()


def test_return_codes(eng, keys):
    import groth_sahai_rs_b200 as gsb
    crs, hid, t1, t2 = keys
    eng.crs_load(crs_bytes(hid))
    lib = eng.lib
    m, n, K = 2, 2, 1
    c = ZkCase(m, n, K, hid, seed=3300)
    xr, yr, Tr, Lr = c.rand()
    good = [ctypes.create_string_buffer(x, len(x)) for x in (*c.stmt(), c.X, c.Y, xr, yr, Tr, Lr)]
    key = ctypes.create_string_buffer(fr_b(t1) + fr_b(t2), 64)
    outs = [ctypes.create_string_buffer(b"\xa5" * (1 << 13), 1 << 13) for _ in range(6)]
    P = [ctypes.cast(b, vp) for b in good]
    O = [ctypes.cast(o, vp) for o in outs]
    fresh = gsb.Engine(0)
    E, F = eng.h, fresh.h

    def prove(h, count=1, mm=m, nn=n, kk=K, null=None):
        q = [None if i == null else x for i, x in enumerate(P + O)]
        return lib.gs_zk_ppe_prove_batch(h, count, mm, nn, kk, *q)

    def simulate(h, count=1, mm=m, nn=n, kk=K, null=None, tk=None):
        q = [None if i == null else x for i, x in enumerate(P[:5] + P[7:] + [ctypes.cast(tk or key, vp)] + O)]
        return lib.gs_zk_ppe_simulate_batch(h, count, mm, nn, kk, *q)

    def verify(h, count=1, mm=m, nn=n, kk=K, null=None):
        q = [None if i == null else x for i, x in enumerate(P[:5] + O + [O[0]])]
        return lib.gs_zk_ppe_verify_batch(h, count, mm, nn, kk, *q)

    wrong = ctypes.create_string_buffer(fr_b(t1) + fr_b((t2 + 1) % R), 64)
    cases = {}
    for name, f, nargs in (("prove", prove, 17), ("simulate", simulate, 16), ("verify", verify, 12)):
        cases.update({
            f"{name} no crs": (f(F), EARG), f"{name} count 0": (f(E, count=0), OK), f"{name} m 0": (f(E, mm=0), EDIM),
            f"{name} n 0": (f(E, nn=0), EDIM), f"{name} K 0": (f(E, kk=0), EDIM),
            f"{name} too many variables": (f(E, mm=(1 << 20)), EDIM)})
        for i in range(nargs):
            cases[f"{name} null argument {i}"] = (f(E, null=i), EARG)
    cases["simulate wrong key"] = (simulate(E, tk=wrong), EARG)
    assert all(o.raw == b"\xa5" * (1 << 13) for o in outs)        # nothing written by a refused call
    fresh.crs_load(crs_bytes(crs))
    cases["simulate under a binding crs"] = (simulate(F), EARG)
    fresh.close()
    assert all(o.raw == b"\xa5" * (1 << 13) for o in outs)
    assert simulate(E) == OK and prove(E) == OK and verify(E) == OK
    got = {k: v[0] for k, v in cases.items()}
    assert got == {k: v[1] for k, v in cases.items()}


def test_api_round_trip():
    """api.ZkPPE: prove / simulate / verify reproduce the C calls made with the same RNG stream"""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    from test_gpu_api_mirror import ReplayRng
    eng = gsb.Engine(0)
    rng = ReplayRng(93)
    crs, key = api.CRS.generate_hiding_crs_with_trapdoor(rng, eng)
    binding = api.CRS.generate_crs(ReplayRng(93), eng)
    crs_o = hiding_crs(ogs.generate_crs(*rng.log[:6]))
    m, n, K = 2, 3, 2
    c = ZkCase(m, n, K, crs_o, seed=3400, E=2)
    sts = [api.ZkPPE(cut(c.A[i * n * 96:(i + 1) * n * 96], 96), cut(c.B[i * m * 192:(i + 1) * m * 192], 192),
                     [[fr_b(g) for g in row] for row in c.gam[i]], list(zip(c.P[i * K:(i + 1) * K], c.Q[i * K:(i + 1) * K])))
           for i in range(2)]
    X = [cut(c.X[i * m * 96:(i + 1) * m * 96], 96) for i in range(2)]
    Y = [cut(c.Y[i * n * 192:(i + 1) * n * 192], 192) for i in range(2)]
    proofs = api.zk_prove_batch(sts, X, Y, crs, ReplayRng(7))
    r = ReplayRng(7)
    per = (m + K) * 2 + n * 2 + 4 + 2 * K      # R, S, T, T_1..T_K of one statement
    draws = [r.fr() for _ in range(2 * per)]
    part = lambda lo, hi: b"".join(b"".join(draws[i * per + lo:i * per + hi]) for i in range(2))
    a, b_, s = (m + K) * 2, (m + K) * 2 + n * 2, (m + K) * 2 + n * 2 + 4
    rnd = (part(0, a), part(a, b_), part(b_, s), part(s, per))
    want = eng.zk_ppe_prove_batch(2, m, n, K, *c.stmt(), c.X, c.Y, *rnd)
    p0 = proofs[0]
    assert b"".join(p0.xcoms.coms) == want[0][:(m + K) * 192] and b"".join(p0.ppe.pi) == want[2][:768]
    assert b"".join(b"".join(e.pi) for e in proofs[1].lin) == want[4][K * 768:]
    assert api.zk_verify_batch(sts, proofs, crs) == [True, True] and sts[0].verify(proofs[0], crs) is True
    assert sts[0].prove(X[0], Y[0], crs, ReplayRng(7)) == p0
    sims = api.zk_simulate_batch(sts, crs, key, ReplayRng(7))
    want = eng.zk_ppe_simulate_batch(2, m, n, K, *c.stmt(), *rnd, key.to_bytes())
    assert b"".join(b"".join(e.theta) for p in sims for e in p.lin) == want[5] and b"".join(sims[1].ycoms.coms) == want[1][n * 384:]
    assert api.zk_verify_batch(sts, sims, crs) == [True, True] and sims[0].xcoms.rand == []
    assert sts[0].verify(proofs[0], binding) is False
    with pytest.raises(gsb.GsError):
        sts[0].simulate(binding, key, ReplayRng(7))
    eng.close()
