"""gs_zk_ppe_rerandomize_batch on the GPU, through the C ABI and api.zk_rerandomize_batch.  A rerandomised real proof is
compared byte for byte with gs_zk_ppe_prove_batch under the combined randomness, a rerandomised simulated proof with
gs_zk_ppe_simulate_batch, and both with the composition of gs_rerandomize_batch on PPE' and on every L_k; the first and
last statement with the C oracle's prove.  Witnesses, constants and target pairs are multiples of the generators with
known discrete logs (bigcase.py, ZkCase of test_gpu_zk.py)."""
import ctypes
import random

import pytest

from bigcase import *  # noqa: F401,F403
from simulate_ref import hiding_crs
from test_gpu_zk import ONE, ZERO_FR, ZkCase, cut, oracle_prove

pytestmark = pytest.mark.gpu

OK, EDIM, EARG = 0, 1, 3
vp = ctypes.c_void_p


@pytest.fixture(scope="module")
def keys():
    crs, (_, _, _, _, t1, t2) = make_crs(4)
    return crs, hiding_crs(crs), t1, t2


@pytest.fixture(scope="module")
def eng():
    import groth_sahai_rs_b200 as gsb
    e = gsb.Engine(0)
    yield e
    e.close()


class Fresh:
    """fresh R', S', T', T'_k of E statements of shape (m, n, K), as Fr ints in the C ABI's layout"""

    def __init__(self, c, seed, zero=False):
        rng = SeededRng(seed)
        m, n, K, E = c.m, c.n, c.K, c.E
        d = (lambda k: [0] * k) if zero else (lambda k: fr_list(rng, k))
        self.xr, self.yr, self.Tr, self.Lr = d(E * (m + K) * 2), d(E * n * 2), d(E * 4), d(E * K * 2)

    def rand(self):
        return frs_b(self.xr), frs_b(self.yr), frs_b(self.Tr), frs_b(self.Lr)


def combined(c, f):
    """a ZkCase whose randomness is c's combined with the fresh f: R + R', S + S', T + T' + S'^T Gamma'^T R, T_k + T'_k"""
    m, n, K, E = c.m, c.n, c.K, c.E
    out = ZkCase.__new__(ZkCase)
    out.__dict__.update(c.__dict__)
    add = lambda a, b: [(x + y) % R for x, y in zip(a, b)]
    out.xr, out.yr, out.Lr = add(c.xr, f.xr), add(c.yr, f.yr), add(c.Lr, f.Lr)
    Tr = []
    for i in range(E):
        Rm = c.xr[i * (m + K) * 2:(i + 1) * (m + K) * 2]     # rows m.. of R meet Gamma''s zero rows
        S2, G = f.yr[i * n * 2:(i + 1) * n * 2], c.gam[i]
        for l in range(2):
            for j in range(2):
                sgr = sum(S2[t * 2 + l] * G[s][t] * Rm[s * 2 + j] for t in range(n) for s in range(m))
                Tr.append((c.Tr[i * 4 + l * 2 + j] + f.Tr[i * 4 + l * 2 + j] + sgr) % R)
    out.Tr = Tr
    return out


def rerand(eng, c, proof, f):
    return eng.zk_ppe_rerandomize_batch(c.E, c.m, c.n, c.K, c.A, c.B, c.G, b"".join(c.Q), *proof, *f.rand())


def composition(eng, c, proof, f, crs):
    """gs_rerandomize_batch of PPE' and of every L_k as MSMEG1 1 x 1 on ([c_{m+k}], [W2]) under row m + k of R', y_rand [0]"""
    m, n, K, E = c.m, c.n, c.K, c.E
    xc, yc, pi, th, lpi, lth = proof
    xr, yr, Tr, Lr = f.rand()
    ppe = eng.rerandomize_batch(0, E, m + K, n, *c.ppe_prime(), xc, yc, pi, th, xr, yr, Tr)
    la, lb, lg, _ = c.lin()
    zc = b"".join(xc[(i * (m + K) + m + k) * 192:][:192] for i in range(E) for k in range(K))
    zr = frs_b([f.xr[(i * (m + K) + m + k) * 2 + a] for i in range(E) for k in range(K) for a in range(2)])
    lin = eng.rerandomize_batch(1, E * K, 1, 1, la, lb, lg, zc, com2_b(ogs.w2(crs)) * E * K, lpi, lth, zr, ZERO_FR * E * K, Lr)
    # L_k's new x-commitments are PPE''s c'_{m+k}, its y-commitment stays W2
    assert lin[0] == b"".join(ppe[0][(i * (m + K) + m + k) * 192:][:192] for i in range(E) for k in range(K))
    assert lin[1] == com2_b(ogs.w2(crs)) * E * K
    return ppe + lin[2:]


def tiled(m, n, K, crs, seed, E, E0=32, true_targets=True):
    """E statements tiled from E0 distinct ones, with randomness of their own"""
    base = ZkCase(m, n, K, crs, seed=seed, E=E0, true_targets=true_targets)
    c = ZkCase.__new__(ZkCase)
    c.m, c.n, c.K, c.E = m, n, K, E
    tile = lambda b, per: b"".join(b[(i % E0) * per:(i % E0 + 1) * per] for i in range(E))
    c.A, c.X, c.B, c.Y, c.G = tile(base.A, n * 96), tile(base.X, m * 96), tile(base.B, m * 192), tile(base.Y, n * 192), \
        tile(base.G, m * n * 32)
    c.gam = [base.gam[i % E0] for i in range(E)]
    pick = lambda L: [L[(i % E0) * K + k] for i in range(E) for k in range(K)]
    c.P, c.negP, c.Q, c.negQ = pick(base.P), pick(base.negP), pick(base.Q), pick(base.negQ)
    rng = SeededRng(seed + 1)
    c.xr, c.yr, c.Tr, c.Lr = fr_list(rng, E * (m + K) * 2), fr_list(rng, E * n * 2), fr_list(rng, E * 4), fr_list(rng, E * K * 2)
    return c


def check_real(eng, c, crs, seed, oracle=True):
    """rerandomise c's real proofs: equal to the prover under the combined randomness and to the composition; accepted"""
    m, n, K, E = c.m, c.n, c.K, c.E
    proof = eng.zk_ppe_prove_batch(E, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())
    f = Fresh(c, seed)
    out = rerand(eng, c, proof, f)
    cc = combined(c, f)
    assert out == eng.zk_ppe_prove_batch(E, m, n, K, *cc.stmt(), cc.X, cc.Y, *cc.rand())
    assert out == composition(eng, c, proof, f, crs)
    if oracle:
        sizes = ((m + K) * 192, n * 384, 768, 384, K * 768, K * 192)
        for i in sorted({0, E - 1}):
            got = tuple(o[i * s:(i + 1) * s] for o, s in zip(out, sizes))
            assert got == oracle_prove(cc, crs_bytes(crs), i), f"statement {i}"
    assert eng.zk_ppe_verify_batch(E, m, n, K, *c.stmt(), *out) == b"\x01" * E
    assert eng.zk_ppe_verify_each_rand(E, m, n, K, *c.stmt(), *out) == b"\x01" * E
    return proof, out


@pytest.mark.parametrize("m,n,K", [(1, 1, 1), (4, 4, 1), (4, 4, 2), (4, 4, 3), (1, 4, 1)])
def test_real_proofs_equal_the_prover_under_the_combined_randomness(eng, keys, m, n, K):
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    c = ZkCase(m, n, K, crs, seed=7000 + 100 * m + 10 * n + K, E=3)
    proof, out = check_real(eng, c, crs, 7001 + 100 * m + 10 * n + K)
    assert all(a != b for a, b in zip(proof, out))


def test_lone_statement(eng, keys):
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    c = ZkCase(2, 3, 2, crs, seed=7100, E=1)
    check_real(eng, c, crs, 7101)


@pytest.mark.parametrize("K", [1, 2, 3])
def test_simulated_proofs_equal_the_simulator_under_the_combined_randomness(eng, keys, K):
    crs, hid, t1, t2 = keys
    eng.crs_load(crs_bytes(hid))
    m = n = 4
    c = ZkCase(m, n, K, hid, seed=7200 + K, E=3, true_targets=False)
    tkey = fr_b(t1) + fr_b(t2)
    sim = eng.zk_ppe_simulate_batch(c.E, m, n, K, *c.stmt(), *c.rand(), tkey)
    f = Fresh(c, 7210 + K)
    out = rerand(eng, c, sim, f)
    assert out == eng.zk_ppe_simulate_batch(c.E, m, n, K, *c.stmt(), *combined(c, f).rand(), tkey)
    assert out == composition(eng, c, sim, f, hid)
    assert eng.zk_ppe_verify_batch(c.E, m, n, K, *c.stmt(), *out) == b"\x01" * c.E
    assert eng.zk_ppe_verify_each_rand(c.E, m, n, K, *c.stmt(), *out) == b"\x01" * c.E
    eng.crs_load(crs_bytes(crs))
    assert eng.zk_ppe_verify_batch(c.E, m, n, K, *c.stmt(), *out) == b"\x00" * c.E


def test_zero_randomness_returns_the_input(eng, keys):
    crs, hid = keys[0], keys[1]
    for key in (crs, hid):
        eng.crs_load(crs_bytes(key))
        c = ZkCase(4, 4, 2, key, seed=7300, E=3)
        proof = eng.zk_ppe_prove_batch(c.E, 4, 4, 2, *c.stmt(), c.X, c.Y, *c.rand())
        assert rerand(eng, c, proof, Fresh(c, 0, zero=True)) == proof


def test_tampered_proofs_keep_their_verdicts(eng, keys):
    """512 statements, one tamper per statement from a mask (every proof element, an X and a Z commitment, a y commitment,
    the target pairs of another statement): the reject bitmaps of both verifiers are the same before and after"""
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    m, n, K, E = 2, 2, 2, 512
    c = tiled(m, n, K, crs, 7400, E)
    out = [bytearray(o) for o in eng.zk_ppe_prove_batch(E, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())]
    sizes = ((m + K) * 192, n * 384, 768, 384, K * 768, K * 192)
    P, Q = list(c.P), list(c.Q)
    mask = random.Random(7401).choices(range(9), k=E)
    for i, t in enumerate(mask):
        j = (i + 1) % E
        if t <= 5:          # 0: X commitment, 1: y commitment, 2: pi, 3: theta, 4: lin_pi, 5: lin_theta
            s = sizes[t]
            out[t][i * s:i * s + 192] = out[t][j * s:j * s + 192]
        elif t == 6:        # the commitment of Z_K
            at = i * sizes[0] + (m + K - 1) * 192
            out[0][at:at + 192] = out[0][j * sizes[0] + (m + K - 1) * 192:j * sizes[0] + (m + K) * 192]
        elif t == 7:        # target pairs exchanged with the next statement
            P[i * K:(i + 1) * K], Q[i * K:(i + 1) * K] = c.P[j * K:(j + 1) * K], c.Q[j * K:(j + 1) * K]
        # t == 8: untouched
    out = tuple(bytes(o) for o in out)
    stmt = (c.A, c.B, c.G, b"".join(P), b"".join(Q))
    before = eng.zk_ppe_verify_batch(E, m, n, K, *stmt, *out)
    assert before == bytes(1 if t == 8 else 0 for t in mask)
    assert eng.zk_ppe_verify_each_rand(E, m, n, K, *stmt, *out) == before
    new = eng.zk_ppe_rerandomize_batch(E, m, n, K, c.A, c.B, c.G, b"".join(Q), *out, *Fresh(c, 7402).rand())
    assert eng.zk_ppe_verify_batch(E, m, n, K, *stmt, *new) == before
    assert eng.zk_ppe_verify_each_rand(E, m, n, K, *stmt, *new) == before


def test_batch_across_the_rerandomisation_chunk(eng, keys):
    """32,769 statements: PPE' is rerandomised in two chunks of gs_rerandomize_batch (32,768 + 1)"""
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    c = tiled(1, 1, 1, crs, 7500, 32769)
    check_real(eng, c, crs, 7501)


@pytest.mark.parametrize("E", [4095, 4097])
def test_fixed_base_table_sizes(keys, E):
    """count * K * 2 = 8,190 and 8,194 L_k pi elements on a fresh engine: the G2 fixed-base tables of the L_k sums are
    the 8-bit and the 16-bit ones"""
    import groth_sahai_rs_b200 as gsb
    crs = keys[0]
    e = gsb.Engine(0)
    try:
        e.crs_load(crs_bytes(crs))
        c = tiled(1, 1, 1, crs, 7600 + E, E)
        check_real(e, c, crs, 7601 + E, oracle=False)
    finally:
        e.close()


def test_return_codes(eng, keys):
    import groth_sahai_rs_b200 as gsb
    crs, hid = keys[0], keys[1]
    eng.crs_load(crs_bytes(hid))
    lib = eng.lib
    m, n, K = 2, 2, 1
    c = ZkCase(m, n, K, hid, seed=7700)
    proof = eng.zk_ppe_prove_batch(1, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())
    ins = (c.A, c.B, c.G, b"".join(c.Q), *proof, *Fresh(c, 7701).rand())
    good = [ctypes.create_string_buffer(x, len(x)) for x in ins]
    outs = [ctypes.create_string_buffer(b"\xa5" * (1 << 13), 1 << 13) for _ in range(6)]
    P = [ctypes.cast(b, vp) for b in good]
    O = [ctypes.cast(o, vp) for o in outs]
    fresh = gsb.Engine(0)
    E, F = eng.h, fresh.h

    def call(h, count=1, mm=m, nn=n, kk=K, null=None):
        q = [None if i == null else x for i, x in enumerate(P + O)]
        return lib.gs_zk_ppe_rerandomize_batch(h, count, mm, nn, kk, *q)

    cases = {"no crs": (call(F), EARG), "count 0": (call(E, count=0), OK), "m 0": (call(E, mm=0), EDIM),
             "n 0": (call(E, nn=0), EDIM), "K 0": (call(E, kk=0), EDIM), "too many variables": (call(E, mm=(1 << 20)), EDIM),
             "too many target pairs": (call(E, kk=(1 << 20) + 1), EDIM)}
    for i in range(20):
        cases[f"null argument {i}"] = (call(E, null=i), EARG)
    fresh.close()
    assert all(o.raw == b"\xa5" * (1 << 13) for o in outs)        # nothing written by a refused call
    got = {k: v[0] for k, v in cases.items()}
    assert got == {k: v[1] for k, v in cases.items()}
    # no trapdoor needed: the same call under the binding and the hiding key
    assert call(E) == OK
    eng.crs_load(crs_bytes(crs))
    assert call(E) == OK


def test_api_round_trip():
    """api.zk_rerandomize_batch / ZkPPE.rerandomize reproduce the C call made with the same RNG stream and verify"""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    from test_gpu_api_mirror import ReplayRng
    eng = gsb.Engine(0)
    rng = ReplayRng(94)
    crs, key = api.CRS.generate_hiding_crs_with_trapdoor(rng, eng)
    crs_o = hiding_crs(ogs.generate_crs(*rng.log[:6]))
    m, n, K = 2, 3, 2
    c = ZkCase(m, n, K, crs_o, seed=7800, E=2)
    sts = [api.ZkPPE(cut(c.A[i * n * 96:(i + 1) * n * 96], 96), cut(c.B[i * m * 192:(i + 1) * m * 192], 192),
                     [[fr_b(g) for g in row] for row in c.gam[i]], list(zip(c.P[i * K:(i + 1) * K], c.Q[i * K:(i + 1) * K])))
           for i in range(2)]
    X = [cut(c.X[i * m * 96:(i + 1) * m * 96], 96) for i in range(2)]
    Y = [cut(c.Y[i * n * 192:(i + 1) * n * 192], 192) for i in range(2)]
    proofs = api.zk_prove_batch(sts, X, Y, crs, ReplayRng(7)) + api.zk_simulate_batch(sts[:1], crs, key, ReplayRng(8))
    sts3 = sts + sts[:1]
    new = api.zk_rerandomize_batch(sts3, proofs, crs, ReplayRng(9))
    assert api.zk_verify_batch(sts3, new, crs) == [True] * 3
    assert all(p.xcoms.rand == [] and p.ppe.rand == [] and p.lin[0].rand == [] for p in new)
    r = ReplayRng(9)
    per = (m + K) * 2 + n * 2 + 4 + 2 * K      # R', S', T', T'_1..T'_K of one statement
    draws = [r.fr() for _ in range(3 * per)]
    part = lambda lo, hi: b"".join(b"".join(draws[i * per + lo:i * per + hi]) for i in range(3))
    a, b_, s = (m + K) * 2, (m + K) * 2 + n * 2, (m + K) * 2 + n * 2 + 4
    cat = lambda f: b"".join(f(p) for p in proofs)
    st = lambda f: b"".join(f(s) for s in sts3)
    want = eng.zk_ppe_rerandomize_batch(
        3, m, n, K, st(lambda s: b"".join(s.a_consts)), st(lambda s: b"".join(s.b_consts)),
        st(lambda s: b"".join(b"".join(r) for r in s.gamma)), st(lambda s: b"".join(q for _, q in s.target_pairs)),
        cat(lambda p: b"".join(p.xcoms.coms)), cat(lambda p: b"".join(p.ycoms.coms)), cat(lambda p: b"".join(p.ppe.pi)),
        cat(lambda p: b"".join(p.ppe.theta)), cat(lambda p: b"".join(b"".join(e.pi) for e in p.lin)),
        cat(lambda p: b"".join(b"".join(e.theta) for e in p.lin)), part(0, a), part(a, b_), part(b_, s), part(s, per))
    assert b"".join(b"".join(p.xcoms.coms) for p in new) == want[0] and b"".join(b"".join(e.pi) for p in new for e in p.lin) == want[4]
    assert b"".join(b"".join(p.ppe.theta) for p in new) == want[3]
    one = sts[0].rerandomize(proofs[0], crs, ReplayRng(9))
    assert one == new[0] and sts[0].verify(one, crs) is True
    eng.close()
