"""gs_zk_ppe_verify_each_rand on the GPU, through the C ABI and api.zk_verify_each_randomized: one folded pairing product
and one final exponentiation per zk PPE statement.  Its verdicts are compared byte for byte with gs_zk_ppe_verify_batch's
on honest, simulated and tampered statements -- including errors on PPE''s theta_0 and L_1's theta that cancel when the
two equations share their weights -- in one pass and in many."""
import ctypes
import os
import random

import pytest

from bigcase import *  # noqa: F401,F403
from conv import com1_b, com1_i, g1_i
from simulate_ref import hiding_crs
from test_gpu_zk import ONE, ZkCase, cut

pytestmark = pytest.mark.gpu

OK, EDIM, EARG = 0, 1, 3
vp = ctypes.c_void_p


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


def rho_of(seed, count, K):
    return random.Random(seed).randbytes(8 * (2 * count * (1 + K) + 1))


def engine_with_batch_max(value):
    import groth_sahai_rs_b200 as gsb
    old = os.environ.get("GS_VERIFY_BATCH_MAX")
    os.environ["GS_VERIFY_BATCH_MAX"] = value
    try:
        return gsb.Engine(0)
    finally:
        os.environ.pop("GS_VERIFY_BATCH_MAX", None) if old is None else os.environ.__setitem__("GS_VERIFY_BATCH_MAX", old)


@pytest.mark.parametrize("m,n,K", [(1, 1, 1), (4, 4, 1), (4, 4, 2), (4, 4, 3), (1, 4, 1)])
def test_honest_real_proofs_are_accepted(eng, keys, m, n, K):
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    c = ZkCase(m, n, K, crs, seed=6000 + 100 * m + 10 * n + K, E=3)
    out = eng.zk_ppe_prove_batch(c.E, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())
    assert eng.zk_ppe_verify_each_rand(c.E, m, n, K, *c.stmt(), *out) == b"\x01" * c.E
    # the other statements' pairs: the targets no longer hold
    shifted = (c.A, c.B, c.G, b"".join(c.P[K:] + c.P[:K]), b"".join(c.Q[K:] + c.Q[:K]))
    assert eng.zk_ppe_verify_each_rand(c.E, m, n, K, *shifted, *out) == b"\x00" * c.E


@pytest.mark.parametrize("K", [1, 2])
def test_simulated_proofs_of_false_targets(eng, keys, K):
    crs, hid, t1, t2 = keys
    eng.crs_load(crs_bytes(hid))
    m = n = 4
    c = ZkCase(m, n, K, hid, seed=6100 + K, E=3, true_targets=False)
    out = eng.zk_ppe_simulate_batch(c.E, m, n, K, *c.stmt(), *c.rand(), fr_b(t1) + fr_b(t2))
    assert eng.zk_ppe_verify_each_rand(c.E, m, n, K, *c.stmt(), *out) == b"\x01" * c.E
    eng.crs_load(crs_bytes(crs))
    assert eng.zk_ppe_verify_each_rand(c.E, m, n, K, *c.stmt(), *out) == b"\x00" * c.E


def test_verdicts_match_the_exact_verifier_under_tampering(eng, keys):
    """The 6,000 statements of test_gpu_zk's tampering test (64 distinct ones tiled, one tamper per statement from a mask:
    every proof element, an X and a Z commitment, a y commitment, an L_k proved with y_rand 1, the target pairs of another
    statement), plus one more kind: +D on PPE''s theta_0 and -D on L_1's theta.  For two rho seeds the verdicts equal
    gs_zk_ppe_verify_batch's, and again with passes of 240 statements.  With L_k's weights set equal to PPE''s the
    cancelling tamper is accepted: the per-equation weights are read where the rho layout puts them."""
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
    bad_pi, bad_th = eng.prove_batch(1, E * K, 1, 1, la, lb, lg, b"".join(c.P), ONE * E * K, zr, ONE * E * K, frs_b(c.Lr))
    P, Q = list(c.P), list(c.Q)
    sizes = ((m + K) * 192, n * 384, 768, 384, K * 768, K * 192)
    D = tuple(g1_i(p) for p in g1_multiples(crs, [7, 11]))
    mask = random.Random(3202).choices(range(11), k=E)
    for i, t in enumerate(mask):
        j = (i + 1) % E
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
        elif t == 10:       # +D on PPE''s theta_0, -D on L_1's theta
            at, lt = i * 384, i * K * 192
            out[3][at:at + 192] = com1_b(ogs.com1_add(com1_i(bytes(out[3][at:at + 192])), D))
            out[5][lt:lt + 192] = com1_b(ogs.com1_add(com1_i(bytes(out[5][lt:lt + 192])), ogs.com1_neg(D)))
        # t == 9: untouched
    out = [bytes(o) for o in out]
    c.P, c.Q = P, Q
    exact = eng.zk_ppe_verify_batch(E, m, n, K, *c.stmt(), *out)
    assert all(exact[i] == (1 if t == 9 else 0) for i, t in enumerate(mask))
    for seed in (1, 2):
        assert eng.zk_ppe_verify_each_rand(E, m, n, K, *c.stmt(), *out, rho=rho_of(seed, E, K)) == exact, seed
    # every L_k weighted like its PPE': the cancelling tamper goes through, nothing else does
    words = rho_of(3, E, K)
    same = words[:16 * E] + b"".join(words[16 * i:16 * i + 16] * K for i in range(E)) + words[-8:]
    got = eng.zk_ppe_verify_each_rand(E, m, n, K, *c.stmt(), *out, rho=same)
    assert all(got[i] == (1 if t in (9, 10) else 0) for i, t in enumerate(mask))
    # passes of 240 statements, uploads of 4 * 240 / K = 480
    small = engine_with_batch_max("240")
    small.crs_load(crs_bytes(crs))
    assert small.zk_ppe_verify_each_rand(E, m, n, K, *c.stmt(), *out, rho=rho_of(1, E, K)) == exact
    small.close()


def test_lone_statement_empty_call_and_zero_rho(eng, keys):
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    m, n, K = 4, 4, 1
    c = ZkCase(m, n, K, crs, seed=6200, E=1)
    out = list(eng.zk_ppe_prove_batch(1, m, n, K, *c.stmt(), c.X, c.Y, *c.rand()))
    assert eng.zk_ppe_verify_each_rand(1, m, n, K, *c.stmt(), *out) == b"\x01"
    bad = out[:2] + [out[2][384:] + out[2][:384]] + out[3:]
    assert eng.zk_ppe_verify_batch(1, m, n, K, *c.stmt(), *bad) == b"\x00"
    assert eng.zk_ppe_verify_each_rand(1, m, n, K, *c.stmt(), *bad) == b"\x00"
    # an all-zero rho makes the check vacuous: everything is accepted
    assert eng.zk_ppe_verify_each_rand(1, m, n, K, *c.stmt(), *bad, rho=bytes(8 * (2 * (1 + K) + 1))) == b"\x01"
    assert eng.zk_ppe_verify_each_rand(0, m, n, K, *(b"",) * 11) == b""


def test_return_codes(eng, keys):
    import groth_sahai_rs_b200 as gsb
    crs = keys[0]
    eng.crs_load(crs_bytes(crs))
    lib = eng.lib
    m, n, K = 2, 2, 1
    c = ZkCase(m, n, K, crs, seed=6300)
    out = eng.zk_ppe_prove_batch(1, m, n, K, *c.stmt(), c.X, c.Y, *c.rand())
    good = [ctypes.create_string_buffer(x, len(x)) for x in (*c.stmt(), *out, rho_of(4, 1, K))]
    ok = ctypes.create_string_buffer(b"\xa5" * 64, 64)
    P = [ctypes.cast(b, vp) for b in good] + [ctypes.cast(ok, vp)]
    fresh = gsb.Engine(0)

    def verify(h, count=1, mm=m, nn=n, kk=K, null=None):
        return lib.gs_zk_ppe_verify_each_rand(h, count, mm, nn, kk, *[None if i == null else x for i, x in enumerate(P)])

    cases = {"no crs": (verify(fresh.h), EARG), "count 0": (verify(eng.h, count=0), OK), "m 0": (verify(eng.h, mm=0), EDIM),
             "n 0": (verify(eng.h, nn=0), EDIM), "K 0": (verify(eng.h, kk=0), EDIM),
             "too many variables": (verify(eng.h, mm=1 << 20), EDIM)}
    for i in range(13):
        cases[f"null argument {i}"] = (verify(eng.h, null=i), EARG)
    fresh.close()
    assert ok.raw == b"\xa5" * 64            # nothing written by a refused call
    assert verify(eng.h) == OK and ok.raw[:1] == b"\x01"
    got = {k: v[0] for k, v in cases.items()}
    assert got == {k: v[1] for k, v in cases.items()}


def test_api_equals_the_exact_verifier():
    """api.zk_verify_each_randomized on ZkPPE objects: the verdicts of api.zk_verify_batch"""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    from test_gpu_api_mirror import ReplayRng
    eng = gsb.Engine(0)
    rng = ReplayRng(95)
    crs = api.CRS.generate_crs(rng, eng)
    crs_o = ogs.generate_crs(*rng.log[:6])
    m, n, K, E = 2, 3, 2, 3
    c = ZkCase(m, n, K, crs_o, seed=6400, E=E)
    sts = [api.ZkPPE(cut(c.A[i * n * 96:(i + 1) * n * 96], 96), cut(c.B[i * m * 192:(i + 1) * m * 192], 192),
                     [[fr_b(g) for g in row] for row in c.gam[i]], list(zip(c.P[i * K:(i + 1) * K], c.Q[i * K:(i + 1) * K])))
           for i in range(E)]
    X = [cut(c.X[i * m * 96:(i + 1) * m * 96], 96) for i in range(E)]
    Y = [cut(c.Y[i * n * 192:(i + 1) * n * 192], 192) for i in range(E)]
    proofs = api.zk_prove_batch(sts, X, Y, crs, ReplayRng(8))
    proofs[1].ppe.pi = proofs[0].ppe.pi
    want = api.zk_verify_batch(sts, proofs, crs)
    assert want == [True, False, True]
    assert api.zk_verify_each_randomized(sts, proofs, crs) == want
    assert api.zk_verify_each_randomized(sts, proofs, crs, rho=rho_of(5, E, K)) == want
    assert api.zk_verify_each_randomized([], [], crs) == []
    with pytest.raises(ValueError):
        api.zk_verify_each_randomized(sts, proofs[:2], crs)
    eng.close()
