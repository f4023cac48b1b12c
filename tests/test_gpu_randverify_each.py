"""gs_verify_each_rand (opt-in; the reference has no such mode): randomised PER-PROOF verification -- the four ComT entries
of every proof folded with that proof's random weights into one pairing product and one final exponentiation, nothing
multiplied across proofs.  Its verdicts must equal the exact verifier's (gs_verify_batch, itself byte-checked against
the CPU restatement in test_gpu_bigparity.py) byte for byte: honest batches of all four equation types, every single
change of a constant, Gamma entry, target, commitment or proof element at several positions, ragged shapes, several
passes, shared commitments, a big statement, a lone proof, and a 1 % tamper mask over a batch of thousands."""
import ctypes
import os
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


def rho_of(count, seed):
    return random.Random(seed).randbytes(8 * (2 * count + 1))


def batch_arrays(cases):
    return [b"".join(c.verify_arrays()[i] for c in cases) for i in range(8)]


def sizes_of(ty, m, n):
    return [n * cb.x_size(ty), m * cb.y_size(ty), m * n * 32, cb.target_size(ty), m * 192, n * 384, cb.cx_of(ty) * 384,
            cb.cy_of(ty) * 192]


def swap(buf, a, b, size):
    """exchange the `size`-byte records at byte offsets a and b"""
    out = bytearray(buf)
    out[a:a + size], out[b:b + size] = buf[b:b + size], buf[a:a + size]
    assert bytes(out) != bytes(buf), "tampering must change something"
    return bytes(out)


def tampered(ty, m, n, arrays, which, p, q):
    """arrays with ONE change in array `which` of proof p (targets: proofs p and q exchanged)."""
    sz = sizes_of(ty, m, n)
    bad = list(arrays)
    o = p * sz[which]
    if which == 0:      # two constants A_0 <-> A_1
        e = cb.x_size(ty)
        bad[0] = swap(arrays[0], o, o + e, e)
    elif which == 1:    # B_0 <-> B_1
        e = cb.y_size(ty)
        bad[1] = swap(arrays[1], o, o + e, e)
    elif which == 2:    # one bit of Gamma[1][1]
        g = bytearray(arrays[2])
        g[o + 32 * (n + 1)] ^= 1
        bad[2] = bytes(g)
    elif which == 3:    # the targets of two proofs exchanged
        bad[3] = swap(arrays[3], o, q * sz[3], sz[3])
    elif which == 4:    # commitments c_0 <-> c_1
        bad[4] = swap(arrays[4], o, o + 192, 192)
    elif which == 5:    # d_0 <-> d_1
        bad[5] = swap(arrays[5], o, o + 384, 384)
    elif which == 6:    # the two coordinates of pi_0
        bad[6] = swap(arrays[6], o, o + 192, 192)
    else:               # the two coordinates of theta_0
        bad[7] = swap(arrays[7], o, o + 96, 96)
    return bad


def check_equal(e, ty, count, m, n, arrays, seed, expect_bad=None):
    """gs_verify_each_rand's verdicts == gs_verify_batch's; returns them"""
    exact = e.verify_batch(ty, count, m, n, *arrays)
    each = e.verify_each_rand(ty, count, m, n, *arrays, rho=rho_of(count, seed))
    assert each == exact, f"type {ty} {m}x{n}: per-proof {each!r} vs exact {exact!r}"
    if expect_bad is not None:
        assert [i for i in range(count) if exact[i] == 0] == expect_bad, f"exact verdicts {exact!r}"
    return each


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_each_4x4_every_tampering(eng, crs, ty):
    count, m, n = 12, 4, 4
    cases = [Case(ty, m, n, crs, seed=3000 + 20 * ty + i, zero_frac=0.25 if i % 4 == 2 else 0.0) for i in range(count)]
    arrays = batch_arrays(cases)
    assert check_equal(eng, ty, count, m, n, arrays, 1) == b"\x01" * count
    assert eng.verify_each_rand(ty, count, m, n, *arrays) == b"\x01" * count                        # OS randomness
    assert eng.verify_each_rand(ty, count, m, n, *arrays, rho=bytes(8 * (2 * count + 1))) == b"\x01" * count  # vacuous
    for which in range(8):
        for p, q in ((0, 11), (5, 9), (11, 3)):
            bad = tampered(ty, m, n, arrays, which, p, q)
            check_equal(eng, ty, count, m, n, bad, 100 + 10 * which + p, sorted({p, q}) if which == 3 else [p])
    # all-zero weights accept even a bad batch (documented: the check is then vacuous)
    bad = tampered(ty, m, n, arrays, 7, 4, 0)
    assert eng.verify_each_rand(ty, count, m, n, *bad, rho=bytes(8 * (2 * count + 1))) == b"\x01" * count


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_each_single_proof(eng, crs, ty):
    m, n = 4, 4
    one = Case(ty, m, n, crs, seed=3100 + ty).verify_arrays()
    assert eng.verify_each_rand(ty, 1, m, n, *one, rho=rho_of(1, 20)) == b"\x01"
    for which in (2, 4, 6, 7):
        assert eng.verify_each_rand(ty, 1, m, n, *tampered(ty, m, n, one, which, 0, 0), rho=rho_of(1, 21 + which)) == b"\x00"


def test_each_ragged_shapes(eng, crs):
    for ty, m, n in ((0, 1, 1), (0, 7, 3), (1, 1, 5), (2, 6, 1), (3, 5, 9)):
        cases = [Case(ty, m, n, crs, seed=3200 + 10 * ty + m + i) for i in range(5)]
        arrays = batch_arrays(cases)
        check_equal(eng, ty, 5, m, n, arrays, 30, [])
        check_equal(eng, ty, 5, m, n, tampered(ty, m, n, arrays, 6, 2, 0), 31, [2])
        check_equal(eng, ty, 5, m, n, tampered(ty, m, n, arrays, 7, 4, 0), 32, [4])
        check_equal(eng, ty, 5, m, n, tampered(ty, m, n, arrays, 3, 1, 3), 33, [1, 3])


def test_each_several_passes(crs):
    """More proofs than one pass holds (GS_VERIFY_BATCH_MAX lowered for the test): passes of 40, 40, 20, each writing its
    own verdicts; bad proofs in the first, second and last pass."""
    import groth_sahai_rs_b200 as gsb
    old = os.environ.get("GS_VERIFY_BATCH_MAX")
    os.environ["GS_VERIFY_BATCH_MAX"] = "40"
    try:
        e = gsb.Engine(0)
    finally:
        os.environ.pop("GS_VERIFY_BATCH_MAX", None) if old is None else os.environ.__setitem__("GS_VERIFY_BATCH_MAX", old)
    e.crs_load(crs_bytes(crs))
    try:
        for ty in (0, 1, 2, 3):
            m, n = 4, 4
            cases = [Case(ty, m, n, crs, seed=3400 + 10 * ty + i) for i in range(6)]
            count = 100
            arrays = [b"".join(cases[i % 6].verify_arrays()[k] for i in range(count)) for k in range(8)]
            check_equal(e, ty, count, m, n, arrays, 40, [])
            bad = tampered(ty, m, n, arrays, 7, 97, 0)
            bad = tampered(ty, m, n, bad, 2, 3, 0)
            bad = tampered(ty, m, n, bad, 6, 41, 0)
            check_equal(e, ty, count, m, n, bad, 41, [3, 41, 97])
    finally:
        e.close()


def test_each_big_statement(eng, crs):
    """One 128 x 128 PPE: more pairs than one accumulator takes, so the proof's pairs are spread over several accumulators
    whose values are multiplied before its final exponentiation."""
    c = Case(0, 128, 128, crs, seed=3500)
    arrays = c.verify_arrays()
    assert eng.verify_each_rand(0, 1, 128, 128, *arrays, rho=rho_of(1, 50)) == b"\x01"
    assert eng.verify_each_rand(0, 1, 128, 128, *tampered(0, 128, 128, arrays, 2, 0, 0), rho=rho_of(1, 51)) == b"\x00"


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_each_shared_commitments(eng, crs, ty):
    """Equations over ONE witness set (the C4 shape): the statement MSM keeps its shared-base tables and both
    coordinates, the slots are folded afterwards."""
    E, m, n = 40, 8, 8
    st = Statement(ty, m, n, E, crs, seed=3600 + ty)
    arrays = st.verify_arrays()
    check_equal(eng, ty, E, m, n, arrays, 60, [])
    for which in (0, 2, 3, 6):
        bad = tampered(ty, m, n, arrays, which, 17, 30)
        check_equal(eng, ty, E, m, n, bad, 61 + which, [17, 30] if which == 3 else [17])


@pytest.mark.parametrize("ty", [0, 3])
def test_each_big_batch_tamper_mask(eng, crs, ty):
    """4,104 proofs with a random ~1 % of them tampered (every kind of change): the verdict bitmap equals the exact one."""
    m, n, reps = 3, 2, 342
    cases = [Case(ty, m, n, crs, seed=3700 + 20 * ty + i) for i in range(12)]
    count = 12 * reps
    arrays = [b"".join(c.verify_arrays()[k] for c in cases) * reps for k in range(8)]
    rng = random.Random(70 + ty)
    picks = sorted(rng.sample(range(count), count // 100))
    bad = arrays
    for i, p in enumerate(picks):
        bad = tampered(ty, m, n, bad, i % 8, p, (p + 1) % count)
    each = check_equal(eng, ty, count, m, n, bad, 72)
    assert each.count(0) >= len(picks)


def test_each_dev_equals_host(eng, crs):
    import torch
    ty, m, n, count = 0, 4, 4, 9
    arrays = batch_arrays([Case(ty, m, n, crs, seed=3800 + i) for i in range(count)])
    arrays = tampered(ty, m, n, arrays, 4, 6, 0)
    r = rho_of(count, 90)
    host = eng.verify_each_rand(ty, count, m, n, *arrays, rho=r)
    ts = [torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda() for b in arrays]
    out = torch.full((count,), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    eng.verify_each_rand_dev(ty, count, m, n, [t.data_ptr() for t in ts], out.data_ptr(), rho=r)
    torch.cuda.synchronize()
    assert bytes(out.cpu().numpy().tobytes()) == host
    assert host == b"\x01" * 6 + b"\x00" + b"\x01" * 2


def test_each_return_codes(eng, crs):
    import torch
    import groth_sahai_rs_b200 as gsb
    lib = eng.lib
    M = N = 4
    BIG = (1 << 20) + 1
    one = Case(0, M, N, crs, seed=3900).verify_arrays()
    keep = [ctypes.create_string_buffer(b, len(b)) for b in one]
    hp = [ctypes.cast(k, vp) for k in keep]
    ts = [torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda() for b in one]
    dp = [vp(t.data_ptr()) for t in ts]
    ok_h = ctypes.create_string_buffer(b"\x07" * 8, 8)
    okh = ctypes.cast(ok_h, vp)
    ok_d = torch.full((8,), 7, dtype=torch.uint8, device="cuda")
    okd = vp(ok_d.data_ptr())
    r = ctypes.create_string_buffer(rho_of(1, 95), 24)
    rp = ctypes.cast(r, vp)
    fresh = gsb.Engine(0)
    E, F = eng.h, fresh.h
    torch.cuda.synchronize()
    try:
        cases = {
            "bad type": (lib.gs_verify_each_rand(E, 4, 1, M, N, *hp, rp, okh), EARG),
            "no crs, count 0": (lib.gs_verify_each_rand(F, 0, 0, M, N, *hp, rp, okh), EARG),
            "no crs, count 1": (lib.gs_verify_each_rand(F, 0, 1, M, N, *hp, rp, okh), EARG),
            "count 0": (lib.gs_verify_each_rand(E, 0, 0, M, N, *hp, rp, okh), OK),
            "count 0, null rho and out": (lib.gs_verify_each_rand(E, 0, 0, M, N, *hp, None, None), OK),
            "m 0": (lib.gs_verify_each_rand(E, 0, 1, 0, N, *hp, rp, okh), EDIM),
            "m big": (lib.gs_verify_each_rand(E, 0, 1, BIG, N, *hp, rp, okh), EDIM),
            "null input": (lib.gs_verify_each_rand(E, 0, 1, M, N, *[None if j == 1 else p for j, p in enumerate(hp)], rp, okh),
                           EARG),
            "null rho": (lib.gs_verify_each_rand(E, 0, 1, M, N, *hp, None, okh), EARG),
            "null out": (lib.gs_verify_each_rand(E, 0, 1, M, N, *hp, rp, None), EARG),
            "dev bad type": (lib.gs_verify_each_rand_dev(E, 4, 1, M, N, *dp, rp, okd), EARG),
            "dev no crs, count 1": (lib.gs_verify_each_rand_dev(F, 0, 1, M, N, *dp, rp, okd), EARG),
            "dev count 0": (lib.gs_verify_each_rand_dev(E, 0, 0, M, N, *dp, rp, okd), OK),
            "dev count 0, null rho and out": (lib.gs_verify_each_rand_dev(E, 0, 0, M, N, *dp, None, None), OK),
            "dev m 0": (lib.gs_verify_each_rand_dev(E, 0, 1, 0, N, *dp, rp, okd), EDIM),
            "dev null rho": (lib.gs_verify_each_rand_dev(E, 0, 1, M, N, *dp, None, okd), EARG),
            "dev null out": (lib.gs_verify_each_rand_dev(E, 0, 1, M, N, *dp, rp, None), EARG),
        }
        torch.cuda.synchronize()
        wrong = {k: (got, want) for k, (got, want) in cases.items() if got != want}
        assert not wrong, f"(got, expected) return codes: {wrong}"
        # the empty calls wrote nothing
        torch.cuda.synchronize()
        assert ok_h.raw == b"\x07" * 8 and bytes(ok_d.cpu().numpy().tobytes()) == b"\x07" * 8
        assert lib.gs_verify_each_rand(E, 0, 1, M, N, *hp, rp, okh) == OK and ok_h.raw[:2] == b"\x01\x07"
    finally:
        fresh.close()


class ReplayRng:
    """host randomness in ABI bytes (as test_gpu_api_mirror.py)"""

    def __init__(self, seed):
        self.s = SeededRng(seed)
        self.log = []

    def fr(self):
        v = self.s.fr()
        self.log.append(v)
        return fr_b(v)

    def g1(self):
        p = self.s.g1()
        self.log.append(p)
        return g1_b(p)

    def g2(self):
        q = self.s.g2()
        self.log.append(q)
        return g2_b(q)


def _split_enc(b, ty, side):
    size = (96 if ty in (0, 1) else 32) if side == "A" else (192 if ty in (0, 2) else 32)
    return [b[i:i + size] for i in range(0, len(b), size)]


@pytest.mark.parametrize("ty", [0, 3])
def test_each_api(ty):
    """api.verify_each_randomized on CProof objects: the per-proof answers of api.verify_batch, honest or not; batches of
    mixed types or shapes are refused as verify_batch refuses them."""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    from oracle import gs as ogs
    eng = gsb.Engine(0)
    rng = ReplayRng(1)
    crs = api.CRS.generate_crs(rng, eng)
    crs_o = ogs.generate_crs(*rng.log[:6])
    cls = [api.PPE, api.MSMEG1, api.MSMEG2, api.QuadEqu][ty]
    eqs, proofs = [], []
    for i in range(5):
        equ_o, xv, yv = random_instance(ty, 2, 1, crs_o, SeededRng(60 + i), zero_frac=0.3)
        equ = cls(_split_enc(enc_A(ty, equ_o.a_consts), ty, "A"), _split_enc(enc_B(ty, equ_o.b_consts), ty, "B"),
                  [[fr_b(g) for g in row] for row in equ_o.gamma], enc_T(ty, equ_o.target))
        eqs.append(equ)
        proofs.append(equ.commit_and_prove(_split_enc(enc_A(ty, xv), ty, "A"), _split_enc(enc_B(ty, yv), ty, "B"), crs,
                                           ReplayRng(90 + i)))
    assert api.verify_each_randomized(eqs, proofs, crs) == [True] * 5
    ep = proofs[2].equ_proofs[0]
    bad = list(proofs)
    th0 = ep.theta[0][96:] + ep.theta[0][:96]                      # the two coordinates of theta_0 exchanged
    bad[2] = api.CProof(proofs[2].xcoms, proofs[2].ycoms, [api.EquProof(ep.pi, [th0] + ep.theta[1:], ty, ep.rand)])
    want = [True, True, False, True, True]
    assert api.verify_each_randomized(eqs, bad, crs, rho=rho_of(5, 7)) == want == api.verify_batch(eqs, bad, crs)
    with pytest.raises(ValueError):
        api.verify_each_randomized(eqs, [proofs[0], api.CProof(proofs[1].xcoms, proofs[1].ycoms, proofs[1].equ_proofs * 2)]
                                   + proofs[2:], crs)
    eng.close()
