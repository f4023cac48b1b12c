"""gs_extract on the GPU: commitments opened with the binding key's trapdoor.  Small and medium batches are committed by
the C oracle (bigcase) from known witnesses, with identity witnesses and zero randomness mixed in, and every extracted
point is compared by bytes.  Big batches (across the 2^16-element chunks, and the 2^20 + 2^20 C2 shape) are committed by
the engine.  Then the API round trip through rerandomisation, one-sided calls, every return code and repeatability."""
import ctypes
import random

import numpy as np
import pytest

from bigcase import *  # noqa: F401,F403
from oracle.bls12_381 import G1 as OG1, G2 as OG2

pytestmark = pytest.mark.gpu

OK, EARG = 0, 3
vp = ctypes.c_void_p


@pytest.fixture(scope="module")
def setup():
    import groth_sahai_rs_b200 as gsb
    crs, draws = make_crs(5)
    e = gsb.Engine(0)
    e.crs_load(crs_bytes(crs))
    yield e, crs, fr_b(draws[2]), fr_b(draws[3])
    e.close()


def _witnesses(rng, crs, n):
    """x, y scalars (every 7th zero: identity witnesses), their G1 / G2 points, and commitment randomness (every 5th
    row zero: c.0 = O)"""
    xs = [0 if i % 7 == 3 else rng.fr() for i in range(n)]
    ys = [0 if i % 7 == 5 else rng.fr() for i in range(n)]
    r2 = [[0, 0] if i % 5 == 1 else [rng.fr(), rng.fr()] for i in range(n)]
    r1 = [0 if i % 5 == 2 else rng.fr() for i in range(n)]
    return xs, ys, b"".join(g1_multiples(crs, xs)), b"".join(g2_multiples(crs, ys)), frs_b([v for r in r2 for v in r]), frs_b(r1)


@pytest.mark.parametrize("n", [1, 2, 127, 128, 129, 4097])
def test_four_kinds_return_the_witnesses(setup, n):
    eng, crs, a1, a2 = setup
    crsb = crs_bytes(crs)
    xs, ys, X, Y, rand2, rand1 = _witnesses(SeededRng(1000 + n), crs, n)
    # batch_commit_G1 / _G2 (PPE) and batch_commit_scalar_to_B1 / _B2 (Quad)
    xc, yc = cb.commit_x(0, X, rand2, crsb, NT), cb.commit_y(0, Y, rand2, crsb, NT)
    assert eng.extract(xc, a1, yc, a2) == (X, Y)
    xc, yc = cb.commit_x(3, frs_b(xs), rand1, crsb, NT), cb.commit_y(3, frs_b(ys), rand1, crsb, NT)
    assert eng.extract(xc, a1, yc, a2) == (X, Y)       # x g1, y g2 with g1 = p1, g2 = p2


def _random_frs(seed, k):
    """k Fr values in Montgomery bytes (< 2^248 < r), fast"""
    b = np.random.default_rng(seed).integers(0, 256, size=(k, 32), dtype=np.uint8)
    b[:, 31] = 0
    return b.tobytes()


def _tiled_points(crs, n, seed):
    """n G1 and n G2 witnesses cycling through 251 known multiples (identity included)"""
    rng = SeededRng(seed)
    ks = [0] + [rng.fr() for _ in range(250)]
    p1, p2 = g1_multiples(crs, ks), g2_multiples(crs, ks)
    return b"".join(p1[i % 251] for i in range(n)), b"".join(p2[i % 251] for i in range(n))


def test_chunked_batch(setup):
    """2 * 2^16 + 3 elements per side: three chunks on alternating streams; every element compared"""
    eng, crs, a1, a2 = setup
    n = 2 * (1 << 16) + 3
    X, Y = _tiled_points(crs, n, 51)
    xc = eng.batch_commit_g1(X, _random_frs(1, 2 * n))
    yc = eng.batch_commit_g2(Y, _random_frs(2, 2 * n))
    assert eng.extract(xc, a1, yc, a2) == (X, Y)


def test_c2_shape_sampled(setup):
    """2^20 G1 + 2^20 G2 commitments made by the engine from known witnesses; extract(commit(X)) == X on a sample"""
    eng, crs, a1, a2 = setup
    n = 1 << 20
    X, Y = _tiled_points(crs, n, 52)
    xc = eng.batch_commit_g1(X, _random_frs(3, 2 * n))
    yc = eng.batch_commit_g2(Y, _random_frs(4, 2 * n))
    ox, oy = eng.extract(xc, a1, yc, a2)
    assert len(ox) == n * 96 and len(oy) == n * 192
    idx = sorted(set(random.Random(7).sample(range(n), 4096)) | {0, n - 1, (1 << 16) - 1, 1 << 16})
    for i in idx:
        assert ox[96 * i:96 * (i + 1)] == X[96 * i:96 * (i + 1)], i
        assert oy[192 * i:192 * (i + 1)] == Y[192 * i:192 * (i + 1)], i


class _Rng:
    def __init__(self, seed): self.s = SeededRng(seed)
    def fr(self): return fr_b(self.s.fr())
    def g1(self): return g1_b(self.s.g1())
    def g2(self): return g2_b(self.s.g2())


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_api_commit_prove_rerandomise_extract(ty):
    """generate_crs_with_trapdoor -> commit_and_prove -> rerandomize_batch -> extract returns the witnesses"""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    eng = gsb.Engine(0)
    crs, key = api.CRS.generate_crs_with_trapdoor(_Rng(60 + ty), eng)
    assert crs.to_bytes() == api.CRS.generate_crs(_Rng(60 + ty), eng).to_bytes()       # the same draws
    assert api.ExtractionKey.from_bytes(key.to_bytes()) == key
    crs_o = ogs.CRS(u=[com1_i(c) for c in crs.u], v=[com2_i(c) for c in crs.v], g1_gen=g1_i(crs.g1_gen),
                    g2_gen=g2_i(crs.g2_gen), gt_gen=fp12_i(crs.gt_gen))
    m, n = 3, 2
    equ_o, xv, yv = random_instance(ty, m, n, crs_o, SeededRng(70 + ty))
    enc_x = lambda v: g1_b(v) if ty in (0, 1) else fr_b(v)
    enc_y = lambda v: g2_b(v) if ty in (0, 2) else fr_b(v)
    T = {0: fp12_b, 1: g1_b, 2: g2_b, 3: fr_b}[ty](equ_o.target)
    equ = (api.PPE, api.MSMEG1, api.MSMEG2, api.QuadEqu)[ty]([enc_x(a) if ty in (0, 1) else fr_b(a) for a in equ_o.a_consts],
                                                              [enc_y(b) if ty in (0, 2) else fr_b(b) for b in equ_o.b_consts],
                                                              [[fr_b(g) for g in row] for row in equ_o.gamma], T)
    rng = _Rng(80 + ty)
    proof = equ.commit_and_prove([enc_x(v) for v in xv], [enc_y(v) for v in yv], crs, rng)
    fresh = api.rerandomize_batch([equ], [proof], crs, rng)[0]
    assert fresh.xcoms.coms != proof.xcoms.coms and equ.verify(fresh, crs)
    want_x = [g1_b(v) if ty in (0, 1) else g1_b(g1_mul(crs_o.g1_gen, v)) for v in xv]
    want_y = [g2_b(v) if ty in (0, 2) else g2_b(g2_mul(crs_o.g2_gen, v)) for v in yv]
    for p in (proof, fresh):
        assert api.extract(p, ty, key, crs) == (want_x, want_y)
    ex1 = api.extract_G1 if ty in (0, 1) else api.extract_scalar_B1
    ex2 = api.extract_G2 if ty in (0, 2) else api.extract_scalar_B2
    assert ex1(fresh.xcoms, key, crs) == want_x and ex2(fresh.ycoms.coms, key, crs) == want_y
    eng.close()


def test_one_sided_calls(setup):
    eng, crs, a1, a2 = setup
    crsb = crs_bytes(crs)
    _, _, X, Y, rand2, _ = _witnesses(SeededRng(90), crs, 33)
    xc, yc = cb.commit_x(0, X, rand2, crsb, NT), cb.commit_y(0, Y, rand2, crsb, NT)
    assert eng.extract(xc, a1) == (X, b"")
    assert eng.extract(ycoms=yc, ykey=a2) == (b"", Y)
    # an empty side's key is not looked at
    assert eng.extract(xc, a1, b"", a1) == (X, b"") and eng.extract(b"", a2, yc, a2) == (b"", Y)


def _raw(eng, nx, xc, xk, ny, yc, yk, fill=0xAB):
    """gs_extract through ctypes with pre-filled outputs: (return code, out_x bytes, out_y bytes)"""
    ox = ctypes.create_string_buffer(bytes([fill]) * max(1, 96 * nx))
    oy = ctypes.create_string_buffer(bytes([fill]) * max(1, 192 * ny))
    keep = [ctypes.create_string_buffer(b) if b is not None else None for b in (xc, xk, yc, yk)]
    ptr = [ctypes.cast(k, vp) if k is not None else None for k in keep]
    rc = eng.lib.gs_extract(eng.h, nx, ptr[0], ptr[1], ny, ptr[2], ptr[3], ctypes.cast(ox, vp), ctypes.cast(oy, vp))
    return rc, ox.raw[:96 * nx], oy.raw[:192 * ny]


def test_return_codes(setup):
    import groth_sahai_rs_b200 as gsb
    eng, crs, a1, a2 = setup
    crsb = crs_bytes(crs)
    _, _, X, Y, rand2, _ = _witnesses(SeededRng(91), crs, 4)
    xc, yc = cb.commit_x(0, X, rand2, crsb, NT), cb.commit_y(0, Y, rand2, crsb, NT)
    fx, fy = b"\xab" * 4 * 96, b"\xab" * 4 * 192
    assert _raw(eng, 4, xc, a1, 4, yc, a2) == (OK, X, Y)
    assert _raw(eng, 0, None, None, 0, None, None)[0] == OK
    # no CRS loaded
    fresh = gsb.Engine(0)
    assert _raw(fresh, 4, xc, a1, 4, yc, a2) == (EARG, fx, fy)
    assert "no CRS" in fresh.lib.gs_last_error(fresh.h).decode()
    fresh.close()
    # a null pointer on a non-empty side
    assert _raw(eng, 4, None, a1, 4, yc, a2) == (EARG, fx, fy)
    assert _raw(eng, 4, xc, None, 0, None, None) == (EARG, fx, b"")
    assert _raw(eng, 0, None, None, 4, yc, None) == (EARG, b"", fy)
    # a wrong key on either side: nothing written on either side
    assert _raw(eng, 4, xc, a2, 4, yc, a2) == (EARG, fx, fy)
    assert "xkey" in eng.lib.gs_last_error(eng.h).decode()
    assert _raw(eng, 4, xc, a1, 4, yc, a1) == (EARG, fx, fy)
    assert "ykey" in eng.lib.gs_last_error(eng.h).decode()
    with pytest.raises(gsb.GsError) as ex:
        eng.extract(xc, a2)
    assert ex.value.code == EARG
    # the hiding CRS (u[1].1 - g1, v[1].1 - g2) has no extraction key: the right a1, a2 are rejected
    hid = ogs.CRS(u=[crs.u[0], (crs.u[1][0], OG1.add(crs.u[1][1], OG1.neg(crs.g1_gen)))],
                  v=[crs.v[0], (crs.v[1][0], OG2.add(crs.v[1][1], OG2.neg(crs.g2_gen)))],
                  g1_gen=crs.g1_gen, g2_gen=crs.g2_gen, gt_gen=crs.gt_gen)
    eng.crs_load(crs_bytes(hid))
    assert _raw(eng, 4, xc, a1, 0, None, None) == (EARG, fx, b"")
    assert _raw(eng, 0, None, None, 4, yc, a2) == (EARG, b"", fy)
    # a key validated (and cached) under one CRS is stale after another CRS is loaded, valid again after a reload
    eng.crs_load(crsb)
    assert _raw(eng, 4, xc, a1, 4, yc, a2) == (OK, X, Y)
    other, _ = make_crs(6)
    eng.crs_load(crs_bytes(other))
    assert _raw(eng, 4, xc, a1, 4, yc, a2) == (EARG, fx, fy)
    eng.crs_load(crsb)
    assert _raw(eng, 4, xc, a1, 4, yc, a2) == (OK, X, Y)


def test_repeatable(setup):
    eng, crs, a1, a2 = setup
    crsb = crs_bytes(crs)
    _, _, X, Y, rand2, _ = _witnesses(SeededRng(92), crs, 300)
    xc, yc = cb.commit_x(0, X, rand2, crsb, NT), cb.commit_y(0, Y, rand2, crsb, NT)
    first = eng.extract(xc, a1, yc, a2)
    assert first == (X, Y)
    for _ in range(3):
        assert eng.extract(xc, a1, yc, a2) == first
