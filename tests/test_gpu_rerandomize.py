"""gs_rerandomize / gs_rerandomize_batch on the GPU.  Expected bytes are built without the engine: the C oracle's
reference-order commit + prove (bigcase) under the combined randomness R + R', S + S', T + T' + S'^T Gamma^T R, computed
here with Python integers mod r.  Every path of the proof-element MSMs is taken: the split lone call, one thread per
product (big batches, across the 32,768-proof chunk), the shared-commitment tables (many equations) and the bucket MSM
(one 1024 x 1024 statement)."""
import ctypes
import random

import pytest

from bigcase import *  # noqa: F401,F403

pytestmark = pytest.mark.gpu

OK, EDIM, EARG = 0, 1, 3
vp = ctypes.c_void_p


@pytest.fixture(scope="module")
def crs():
    return make_crs(1)[0]


@pytest.fixture(scope="module")
def eng(crs):
    import groth_sahai_rs_b200 as gsb
    e = gsb.Engine(0)
    e.crs_load(crs_bytes(crs))
    yield e
    e.close()


def ints(b):
    return [fr_i(b[32 * i:32 * (i + 1)]) for i in range(len(b) // 32)]


def mat(v, rows, cols):
    return [v[r * cols:(r + 1) * cols] for r in range(rows)]


def new_rand(seed, ty, m, n, reps=1, eqs=1):
    """(R', S' for `reps` commitment sets, T' for `eqs` equations) as int lists, C-ABI order"""
    r = random.Random(seed)
    cx, cy = cb.cx_of(ty), cb.cy_of(ty)
    draw = lambda k: [r.randrange(R) for _ in range(k)]
    return draw(reps * m * cx), draw(reps * n * cy), draw(eqs * cx * cy)


def combined(ty, m, n, gam, xr, yr, T, xr2, yr2, T2):
    """(R + R', S + S', T + T' + S'^T Gamma^T R) of one equation, flat int lists"""
    cx, cy = cb.cx_of(ty), cb.cy_of(ty)
    Rm, S2 = mat(xr, m, cx), mat(yr2, n, cy)
    G = mat(gam, m, n)
    sg = [[sum(S2[j][l] * G[k][j] for j in range(n)) % R for k in range(m)] for l in range(cy)]   # S'^T Gamma^T (cy x m)
    corr = [sum(sg[l][k] * Rm[k][i] for k in range(m)) % R for l in range(cy) for i in range(cx)]
    add = lambda a, b: [(x + y) % R for x, y in zip(a, b)]
    return add(xr, xr2), add(yr, yr2), add(add(T, T2), corr)


def expected_case(c, xr2, yr2, T2):
    """commit + prove of Case c under the combined randomness, by the C oracle"""
    xr, yr, T = combined(c.ty, c.m, c.n, ints(c.G), ints(c.xr), ints(c.yr), ints(c.Tr), xr2, yr2, T2)
    xc = cb.commit_x(c.ty, c.X, frs_b(xr), c.crsb, NT)
    yc = cb.commit_y(c.ty, c.Y, frs_b(yr), c.crsb, NT)
    pi, th = cb.prove(c.ty, c.m, c.n, c.A, c.B, c.G, c.X, c.Y, frs_b(xr), frs_b(yr), frs_b(T), c.crsb, NT)
    return xc, yc, pi, th


def rr_one(eng, c, xr2, yr2, T2):
    return eng.rerandomize(c.ty, c.m, c.n, c.A, c.B, c.G, c.xc, c.yc, c.pi, c.theta, frs_b(xr2), frs_b(yr2), frs_b(T2))


def flip_theta(th):
    t = bytearray(th)
    t[0:96], t[96:192] = th[96:192], th[0:96]
    return bytes(t)


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
@pytest.mark.parametrize("m,n", [(4, 4), (1, 3), (3, 1)])
def test_lone_call_equals_fresh_proof(eng, crs, ty, m, n):
    c = Case(ty, m, n, crs, seed=1000 + 10 * ty + m)
    xr2, yr2, T2 = new_rand(1100 + ty + m, ty, m, n)
    out = rr_one(eng, c, xr2, yr2, T2)
    assert out == expected_case(c, xr2, yr2, T2)
    assert out[0] != c.xc and out[2] != c.pi
    xc, yc, pi, th = out
    assert eng.verify(ty, m, n, c.A, c.B, c.G, c.T, xc, yc, pi, th) is True
    assert rr_one(eng, c, xr2, yr2, T2) == out                                # the same call twice: the same bytes
    # the batch entry point with count 1 and the lone one agree
    assert eng.rerandomize_batch(ty, 1, m, n, c.A, c.B, c.G, c.xc, c.yc, c.pi, c.theta, frs_b(xr2), frs_b(yr2), frs_b(T2)) == out


@pytest.mark.parametrize("ty", [0, 3])
def test_zero_randomness_and_tampered_input(eng, crs, ty):
    m = n = 4
    c = Case(ty, m, n, crs, seed=1200 + ty)
    cx, cy = cb.cx_of(ty), cb.cy_of(ty)
    assert rr_one(eng, c, [0] * (m * cx), [0] * (n * cy), [0] * (cx * cy)) == (c.xc, c.yc, c.pi, c.theta)
    bad = flip_theta(c.theta)
    assert eng.verify(ty, m, n, c.A, c.B, c.G, c.T, c.xc, c.yc, c.pi, bad) is False
    out = eng.rerandomize(ty, m, n, c.A, c.B, c.G, c.xc, c.yc, c.pi, bad, *[frs_b(v) for v in new_rand(1210 + ty, ty, m, n)])
    assert eng.verify(ty, m, n, c.A, c.B, c.G, c.T, *out) is False


def test_big_batch_one_thread_per_product(eng, crs):
    """32,768 + 512 independent 4 x 4 PPE proofs: one thread per product in the first chunk, the split path and two
    streams in the second; every output verifies, a sample is checked byte for byte, one tampered input stays rejected."""
    ty, m, n = 0, 4, 4
    count, distinct, bad = 32768 + 512, 16, 32768 + 7
    cases = [Case(ty, m, n, crs, seed=1300 + i) for i in range(distinct)]
    pick = lambda k: [cases[i % distinct].verify_arrays()[k] for i in range(count)]
    A, B, G, T, xc, yc, pi, th = [b"".join(pick(k)) for k in range(8)]
    thl = bytearray(th)
    o = bad * 2 * 192
    thl[o:o + 192] = flip_theta(th[o:o + 192])
    xr2, yr2, T2 = new_rand(1301, ty, m, n, reps=count, eqs=count)
    out = eng.rerandomize_batch(ty, count, m, n, A, B, G, xc, yc, pi, bytes(thl), frs_b(xr2), frs_b(yr2), frs_b(T2))
    ok = eng.verify_batch(ty, count, m, n, A, B, G, T, *out)
    assert ok == bytes(1 if i != bad else 0 for i in range(count))
    for i in (0, 5, 32767, 32768, count - 1):
        c = cases[i % distinct]
        want = expected_case(c, xr2[i * 8:(i + 1) * 8], yr2[i * 8:(i + 1) * 8], T2[i * 4:(i + 1) * 4])
        got = (out[0][i * m * 192:(i + 1) * m * 192], out[1][i * n * 384:(i + 1) * n * 384], out[2][i * 768:(i + 1) * 768],
               out[3][i * 384:(i + 1) * 384])
        assert got == want, f"proof {i}"


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_shared_commitments_statement(eng, crs, ty):
    """64 equations over one set of 64 x 64 commitments (the C4 shape): shared-base tables over the commitments and, on
    group-typed sides, the constants of all equations along one bucket structure."""
    m = n = E = 64
    st = Statement(ty, m, n, E, crs, seed=1400 + ty)
    cx, cy = cb.cx_of(ty), cb.cy_of(ty)
    xr2, yr2, T2 = new_rand(1410 + ty, ty, m, n, reps=1, eqs=E)
    out = eng.rerandomize_batch(ty, E, m, n, st.A, st.B, st.G, st.xc, st.yc, st.pi, st.theta, frs_b(xr2), frs_b(yr2),
                                frs_b(T2), shared_coms=True)
    G, xr, yr, T = ints(st.G), ints(st.xr), ints(st.yr), ints(st.Tr)
    Ts = []
    for e in range(E):
        k = cx * cy
        xrc, yrc, Te = combined(ty, m, n, G[e * m * n:(e + 1) * m * n], xr, yr, T[e * k:(e + 1) * k], xr2, yr2, T2[e * k:(e + 1) * k])
        Ts += Te
    want_x = cb.commit_x(ty, st.X, frs_b(xrc), st.crsb, NT)
    want_y = cb.commit_y(ty, st.Y, frs_b(yrc), st.crsb, NT)
    want_pi, want_th = cb.prove_batch(ty, E, m, n, st.A, st.B, st.G, st.X, st.Y, frs_b(xrc), frs_b(yrc), frs_b(Ts), True,
                                      st.crsb, NT)
    assert out == (want_x, want_y, want_pi, want_th)
    ok = eng.verify_batch(ty, E, m, n, st.A, st.B, st.G, st.T, out[0] * E, out[1] * E, out[2], out[3])
    assert ok == b"\x01" * E


def test_1024x1024_ppe_bucket_msm(eng, crs):
    c = Case(0, 1024, 1024, crs, seed=1500)
    xr2, yr2, T2 = new_rand(1501, 0, 1024, 1024)
    out = rr_one(eng, c, xr2, yr2, T2)
    assert out == expected_case(c, xr2, yr2, T2)
    assert eng.verify(0, 1024, 1024, c.A, c.B, c.G, c.T, *out) is True


def test_return_codes(eng):
    import groth_sahai_rs_b200 as gsb
    fresh = gsb.Engine(0)
    lib = eng.lib
    m = n = 4
    bufs = [ctypes.create_string_buffer(1 << 14) for _ in range(14)]
    p = [ctypes.cast(b, vp) for b in bufs]

    def call(h, ty=0, count=1, mm=m, nn=n, null=None):
        q = [None if i == null else x for i, x in enumerate(p)]
        return lib.gs_rerandomize_batch(h, ty, count, mm, nn, *q[:10], 0, *q[10:])

    E, F = eng.h, fresh.h
    cases = {
        "bad type": (call(E, ty=4), EARG),
        "negative type": (call(E, ty=-1), EARG),
        "no crs": (call(F), EARG),
        "count 0": (call(E, count=0), OK),
        "m 0": (call(E, mm=0), EDIM),
        "n 0": (call(E, nn=0), EDIM),
        "too many variables": (call(E, mm=(1 << 22) + 1), EDIM),
        "lone m 0": (lib.gs_rerandomize(E, 0, 0, n, *p), EDIM),
        "lone bad type": (lib.gs_rerandomize(E, 9, m, n, *p), EARG),
    }
    for i in range(14):
        cases[f"null argument {i}"] = (call(E, null=i), EARG)
    fresh.close()
    got = {k: v[0] for k, v in cases.items()}
    assert got == {k: v[1] for k, v in cases.items()}


@pytest.mark.parametrize("hiding", [False, True])
def test_api_round_trip(hiding):
    """serialize -> deserialize -> rerandomize -> verify through the host API, shared and independent commitments."""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    from test_gpu_api_mirror import ReplayRng, _equation
    eng = gsb.Engine(0)
    rng = ReplayRng(81)
    key = (api.CRS.generate_hiding_crs if hiding else api.CRS.generate_crs)(rng, eng)
    crs_o = ogs.generate_crs(*rng.log[:6])
    for ty in (0, 1, 2, 3):
        _, equ, xvars, yvars, _, _ = _equation(api, crs_o, ty, 90 + ty)
        cp = equ.commit_and_prove(xvars, yvars, key, ReplayRng(7))
        wire = (api.serialize_commit(cp.xcoms, eng), api.serialize_commit(cp.ycoms, eng),
                api.serialize_equ_proof(cp.equ_proofs[0], eng), api.serialize_equation(equ, eng))
        back = api.CProof(api.deserialize_commit(wire[0], 1, eng), api.deserialize_commit(wire[1], 2, eng),
                          [api.deserialize_equ_proof(wire[2], eng)])
        e2 = api.deserialize_equation(wire[3], ty, eng)
        rr = e2.rerandomize(back, key, ReplayRng(8))
        assert e2.verify(rr, key) is True
        assert rr.xcoms.coms != cp.xcoms.coms and rr.xcoms.rand == [] and rr.equ_proofs[0].rand == []
        assert api.deserialize_equ_proof(api.serialize_equ_proof(rr.equ_proofs[0], eng), eng) == rr.equ_proofs[0]
        # draw order: R' rows, S' rows, T' -- replaying it through rerandomize_batch gives the same bytes
        again = api.rerandomize_batch([e2], [back], key, ReplayRng(8))[0]
        assert again == rr
        # two equations sharing the commitments: one new set, shared by both returned proofs
        cp2 = api.CProof(cp.xcoms, cp.ycoms, [equ.prove(xvars, yvars, cp.xcoms, cp.ycoms, key, ReplayRng(9))])
        both = api.rerandomize_batch([equ, equ], [cp, cp2], key, ReplayRng(10), shared_commitments=True)
        assert both[0].xcoms.coms == both[1].xcoms.coms and both[0].ycoms.coms == both[1].ycoms.coms
        assert api.verify_batch([equ, equ], both, key) == [True, True]
    eng.close()
