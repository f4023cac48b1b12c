"""The verify entry points called directly through the C ABI (the Engine's Python size checks bypassed).

1. Return codes: every entry point answers a bad argument with the code below, whichever check comes first.  The codes
   are not all consistent with each other (with count 0, gs_verify_batch needs no CRS while gs_verify_batch_dev does;
   gs_verify_batch_rand accepts count 0 while gs_verify_batch_rand_dev rejects it); the table pins them as they are.
2. The device-buffer entry points give the verdicts of the host-buffer ones on the same honest + tampered batch."""
import ctypes

import pytest

from bigcase import *  # noqa: F401,F403

pytestmark = pytest.mark.gpu

OK, EDIM, EARG = 0, 1, 3
M = N = 4
BIG = (1 << 20) + 1
COMT = 4 * 576
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


@pytest.fixture(scope="module")
def fresh():
    """an Engine without a CRS"""
    import groth_sahai_rs_b200 as gsb
    e = gsb.Engine(0)
    yield e
    e.close()


def batch(ty, crs, count, seed, bad=None):
    """the eight verify arrays of `count` proofs; proof `bad` gets the two coordinates of its theta_0 exchanged"""
    arrays = [b"".join(Case(ty, M, N, crs, seed=seed + i).verify_arrays()[k] for i in range(count)) for k in range(8)]
    if bad is not None:
        th = bytearray(arrays[7])
        o = bad * cb.cy_of(ty) * 192
        th[o:o + 96], th[o + 96:o + 192] = arrays[7][o + 96:o + 192], arrays[7][o:o + 96]
        arrays[7] = bytes(th)
    return arrays


def host(bufs):
    """bytes -> keep-alive buffers and their addresses"""
    keep = [ctypes.create_string_buffer(b, max(1, len(b))) for b in bufs]
    return keep, [ctypes.cast(k, vp) for k in keep]


def dev(bufs):
    import torch
    ts = [torch.frombuffer(bytearray(b), dtype=torch.uint8).cuda() if b else torch.zeros(1, dtype=torch.uint8, device="cuda")
          for b in bufs]
    return ts, [vp(t.data_ptr()) for t in ts]


def rho(count):
    return ctypes.create_string_buffer(bytes(range(256)) * ((8 * (2 * count + 1)) // 256 + 1))


@pytest.fixture(scope="module")
def one(crs):
    """the arrays of one honest 4 x 4 PPE proof"""
    return batch(0, crs, 1, 3100)


def test_return_codes(eng, fresh, one):
    import torch
    from groth_sahai_rs_b200.ffi import ALLGATHER_FN
    lib = eng.lib
    hk, hp = host(one)
    dk, dp = dev(one)
    ok_h = ctypes.create_string_buffer(8)
    okh = ctypes.cast(ok_h, vp)
    ok_d = torch.zeros(8, dtype=torch.uint8, device="cuda")
    okd = vp(ok_d.data_ptr())
    part_h = ctypes.create_string_buffer(COMT)
    parth = ctypes.cast(part_h, vp)
    part_d = torch.zeros(COMT, dtype=torch.uint8, device="cuda")
    partd = vp(part_d.data_ptr())
    r = rho(1)
    rp = ctypes.cast(r, vp)
    never = ALLGATHER_FN(lambda u, s, d, b: 1)  # (no case below reaches an exchange)
    torch.cuda.synchronize()

    def with_null(ptrs, i):
        return [None if j == i else p for j, p in enumerate(ptrs)]

    E, F = eng.h, fresh.h
    cases = {
        # gs_verify_batch: a null output is checked first; no CRS is needed for count 0
        "batch bad type": (lib.gs_verify_batch(E, 4, 1, M, N, *hp, okh), EARG),
        "batch no crs, count 0": (lib.gs_verify_batch(F, 0, 0, M, N, *hp, okh), OK),
        "batch no crs, count 1": (lib.gs_verify_batch(F, 0, 1, M, N, *hp, okh), EARG),
        "batch count 0": (lib.gs_verify_batch(E, 0, 0, M, N, *hp, okh), OK),
        "batch m 0": (lib.gs_verify_batch(E, 0, 1, 0, N, *hp, okh), EDIM),
        "batch null out": (lib.gs_verify_batch(E, 0, 1, M, N, *hp, None), EARG),
        "batch null out, bad type": (lib.gs_verify_batch(E, 7, 1, M, N, *hp, None), EARG),
        "batch null out, m 0": (lib.gs_verify_batch(E, 0, 1, 0, N, *hp, None), EARG),
        "batch null out, count 0": (lib.gs_verify_batch(E, 0, 0, M, N, *hp, None), OK),
        "batch null input, m 0": (lib.gs_verify_batch(E, 0, 1, 0, N, *with_null(hp, 2), okh), EDIM),
        "batch null input, no crs": (lib.gs_verify_batch(F, 0, 1, M, N, *with_null(hp, 6), okh), EARG),
        # gs_verify_partial
        "partial bad type": (lib.gs_verify_partial(E, -1, 1, M, N, *hp, 0, 1, parth), EARG),
        "partial bad rank": (lib.gs_verify_partial(E, 0, 1, M, N, *hp, 2, 2, parth), EARG),
        "partial bad world": (lib.gs_verify_partial(E, 0, 1, M, N, *hp, 0, 0, parth), EARG),
        "partial bad rank, count 0": (lib.gs_verify_partial(E, 0, 0, M, N, *hp, -1, 2, parth), EARG),
        "partial no crs, count 0": (lib.gs_verify_partial(F, 0, 0, M, N, *hp, 0, 1, parth), OK),
        "partial no crs, count 1": (lib.gs_verify_partial(F, 0, 1, M, N, *hp, 0, 1, parth), EARG),
        "partial count 0": (lib.gs_verify_partial(E, 0, 0, M, N, *hp, 0, 1, parth), OK),
        "partial m 0": (lib.gs_verify_partial(E, 0, 1, 0, N, *hp, 0, 1, parth), EDIM),
        "partial n 0, bad rank": (lib.gs_verify_partial(E, 0, 1, M, 0, *hp, 3, 2, parth), EARG),
        "partial null out": (lib.gs_verify_partial(E, 0, 1, M, N, *hp, 0, 1, None), EARG),
        # gs_verify_finish (no CRS needed)
        "finish bad type": (lib.gs_verify_finish(E, 5, 1, 1, parth, hp[3], okh), EARG),
        "finish nparts 0": (lib.gs_verify_finish(E, 0, 1, 0, parth, hp[3], okh), EARG),
        "finish nparts 4097": (lib.gs_verify_finish(E, 0, 1, 4097, parth, hp[3], okh), EARG),
        "finish nparts 0, count 0": (lib.gs_verify_finish(E, 0, 0, 0, parth, hp[3], okh), EARG),
        "finish count 0": (lib.gs_verify_finish(E, 0, 0, 1, None, None, None), OK),
        "finish null partials": (lib.gs_verify_finish(E, 0, 1, 1, None, hp[3], okh), EARG),
        "finish null target": (lib.gs_verify_finish(E, 0, 1, 1, parth, None, okh), EARG),
        "finish null out": (lib.gs_verify_finish(E, 0, 1, 1, parth, hp[3], None), EARG),
        # gs_verify_sharded: the CRS is checked ahead of count 0, the length limit ahead of any read
        "sharded bad type": (lib.gs_verify_sharded(E, 4, 1, M, N, *hp, 0, 1, never, None, okh), EARG),
        "sharded bad rank": (lib.gs_verify_sharded(E, 0, 1, M, N, *hp, 1, 1, never, None, okh), EARG),
        "sharded no crs, count 0": (lib.gs_verify_sharded(F, 0, 0, M, N, *hp, 0, 1, never, None, okh), EARG),
        "sharded no crs, count 1": (lib.gs_verify_sharded(F, 0, 1, M, N, *hp, 0, 1, never, None, okh), EARG),
        "sharded count 0": (lib.gs_verify_sharded(E, 0, 0, M, N, *hp, 0, 1, never, None, okh), OK),
        "sharded m 0": (lib.gs_verify_sharded(E, 0, 1, 0, N, *hp, 0, 1, never, None, okh), EDIM),
        "sharded m big": (lib.gs_verify_sharded(E, 0, 1, BIG, N, *hp, 0, 1, never, None, okh), EDIM),
        "sharded n big, null input": (lib.gs_verify_sharded(E, 0, 1, M, BIG, *with_null(hp, 0), 0, 1, never, None, okh), EDIM),
        "sharded null input": (lib.gs_verify_sharded(E, 0, 1, M, N, *with_null(hp, 4), 0, 1, never, None, okh), EARG),
        "sharded null gamma": (lib.gs_verify_sharded(E, 0, 1, M, N, *with_null(hp, 2), 0, 1, never, None, okh), EARG),
        "sharded null out": (lib.gs_verify_sharded(E, 0, 1, M, N, *hp, 0, 1, never, None, None), EARG),
        "sharded null allgather": (lib.gs_verify_sharded(E, 0, 1, M, N, *hp, 0, 1, ALLGATHER_FN(), None, okh), EARG),
        # gs_verify_batch_rand: count 0 is an accepted (empty) batch
        "rand bad type": (lib.gs_verify_batch_rand(E, 4, 1, M, N, *hp, rp, okh), EARG),
        "rand no crs, count 0": (lib.gs_verify_batch_rand(F, 0, 0, M, N, *hp, rp, okh), EARG),
        "rand no crs, count 1": (lib.gs_verify_batch_rand(F, 0, 1, M, N, *hp, rp, okh), EARG),
        "rand m 0": (lib.gs_verify_batch_rand(E, 0, 1, 0, N, *hp, rp, okh), EDIM),
        "rand m big": (lib.gs_verify_batch_rand(E, 0, 1, BIG, N, *hp, rp, okh), EDIM),
        "rand m big, null rho": (lib.gs_verify_batch_rand(E, 0, 1, BIG, N, *hp, None, okh), EDIM),
        "rand null input": (lib.gs_verify_batch_rand(E, 0, 1, M, N, *with_null(hp, 1), rp, okh), EARG),
        "rand null rho": (lib.gs_verify_batch_rand(E, 0, 1, M, N, *hp, None, okh), EARG),
        "rand null out": (lib.gs_verify_batch_rand(E, 0, 1, M, N, *hp, rp, None), EARG),
        "rand null out, count 0": (lib.gs_verify_batch_rand(E, 0, 0, M, N, *hp, rp, None), EARG),
        # gs_verify_batch_dev / gs_verify_partial_dev: the CRS is checked ahead of count 0
        "batch_dev bad type": (lib.gs_verify_batch_dev(E, 4, 1, M, N, *dp, okd), EARG),
        "batch_dev no crs, count 0": (lib.gs_verify_batch_dev(F, 0, 0, M, N, *dp, okd), EARG),
        "batch_dev no crs, count 1": (lib.gs_verify_batch_dev(F, 0, 1, M, N, *dp, okd), EARG),
        "batch_dev count 0": (lib.gs_verify_batch_dev(E, 0, 0, M, N, *dp, okd), OK),
        "batch_dev m 0": (lib.gs_verify_batch_dev(E, 0, 1, 0, N, *dp, okd), EDIM),
        "batch_dev m big": (lib.gs_verify_batch_dev(E, 0, 1, BIG, N, *dp, okd), EDIM),
        "partial_dev bad type": (lib.gs_verify_partial_dev(E, 4, 1, M, N, *dp, 0, 1, partd), EARG),
        "partial_dev bad rank": (lib.gs_verify_partial_dev(E, 0, 1, M, N, *dp, 3, 3, partd), EARG),
        "partial_dev no crs, count 0": (lib.gs_verify_partial_dev(F, 0, 0, M, N, *dp, 0, 1, partd), EARG),
        "partial_dev no crs, count 1": (lib.gs_verify_partial_dev(F, 0, 1, M, N, *dp, 0, 1, partd), EARG),
        "partial_dev count 0": (lib.gs_verify_partial_dev(E, 0, 0, M, N, *dp, 0, 1, partd), OK),
        "partial_dev n 0": (lib.gs_verify_partial_dev(E, 0, 1, M, 0, *dp, 0, 1, partd), EDIM),
        "partial_dev n big": (lib.gs_verify_partial_dev(E, 0, 1, M, BIG, *dp, 0, 1, partd), EDIM),
        # gs_verify_finish_dev
        "finish_dev bad type": (lib.gs_verify_finish_dev(E, 4, 1, 1, partd, dp[3], okd), EARG),
        "finish_dev nparts 0": (lib.gs_verify_finish_dev(E, 0, 1, 0, partd, dp[3], okd), EARG),
        "finish_dev nparts 4097": (lib.gs_verify_finish_dev(E, 0, 1, 4097, partd, dp[3], okd), EARG),
        "finish_dev count 0": (lib.gs_verify_finish_dev(E, 0, 0, 1, partd, dp[3], okd), OK),
        # gs_verify_batch_rand_dev: count 0 is an error here
        "rand_dev bad type": (lib.gs_verify_batch_rand_dev(E, 4, 1, M, N, *dp, rp, okd), EARG),
        "rand_dev no crs, count 0": (lib.gs_verify_batch_rand_dev(F, 0, 0, M, N, *dp, rp, okd), EARG),
        "rand_dev no crs, count 1": (lib.gs_verify_batch_rand_dev(F, 0, 1, M, N, *dp, rp, okd), EARG),
        "rand_dev count 0": (lib.gs_verify_batch_rand_dev(E, 0, 0, M, N, *dp, rp, okd), EARG),
        "rand_dev m 0": (lib.gs_verify_batch_rand_dev(E, 0, 1, 0, N, *dp, rp, okd), EDIM),
        "rand_dev m big": (lib.gs_verify_batch_rand_dev(E, 0, 1, BIG, N, *dp, rp, okd), EDIM),
        "rand_dev m big, null rho": (lib.gs_verify_batch_rand_dev(E, 0, 1, BIG, N, *dp, None, okd), EDIM),
        "rand_dev null rho": (lib.gs_verify_batch_rand_dev(E, 0, 1, M, N, *dp, None, okd), EARG),
    }
    torch.cuda.synchronize()
    wrong = {k: (got, want) for k, (got, want) in cases.items() if got != want}
    assert not wrong, f"(got, expected) return codes: {wrong}"

    # what the accepted empty calls write: gs_verify_batch_rand reports an empty batch as valid
    ok_h[0] = b"\x07"
    assert lib.gs_verify_batch_rand(E, 0, 0, M, N, *hp, rp, okh) == OK and ok_h.raw[0] == 1
    # gs_verify_finish needs no CRS: a context without one finishes a partial product computed by another
    assert lib.gs_verify_partial(E, 0, 1, M, N, *hp, 0, 1, parth) == OK
    ok_h[0] = b"\x07"
    assert lib.gs_verify_finish(F, 0, 1, 1, parth, hp[3], okh) == OK and ok_h.raw[0] == 1
    part_d.copy_(torch.frombuffer(bytearray(part_h.raw), dtype=torch.uint8))
    ok_d.zero_()
    torch.cuda.synchronize()
    assert lib.gs_verify_finish_dev(F, 0, 1, 1, partd, dp[3], okd) == OK
    torch.cuda.synchronize()
    assert int(ok_d[0]) == 1


@pytest.mark.parametrize("ty", [0, 3])
@pytest.mark.parametrize("bad", [None, 2])
def test_dev_paths_match_host(eng, crs, ty, bad):
    """gs_verify_batch_dev, gs_verify_partial_dev (2 ranks) + gs_verify_finish_dev and gs_verify_batch_rand_dev on
    device copies give the verdicts of gs_verify_batch and gs_verify_batch_rand."""
    import torch
    lib = eng.lib
    count = 5
    arrays = batch(ty, crs, count, 3200 + 10 * ty, bad)
    want = eng.verify_batch(ty, count, M, N, *arrays)
    assert want == (b"\x01" * count if bad is None else b"\x01\x01\x00\x01\x01")
    r = rho(count)
    want_rand = eng.verify_batch_rand(ty, count, M, N, *arrays, rho=r.raw[:8 * (2 * count + 1)])
    assert want_rand is (bad is None)

    dk, dp = dev(arrays)
    ok = torch.full((count,), 7, dtype=torch.uint8, device="cuda")
    parts = torch.zeros(2 * count * COMT, dtype=torch.uint8, device="cuda")
    ok2 = torch.full((count,), 7, dtype=torch.uint8, device="cuda")
    ok1 = torch.full((1,), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    assert lib.gs_verify_batch_dev(eng.h, ty, count, M, N, *dp, vp(ok.data_ptr())) == OK
    for rank in range(2):
        assert lib.gs_verify_partial_dev(eng.h, ty, count, M, N, *dp, rank, 2, vp(parts.data_ptr() + rank * count * COMT)) == OK
    assert lib.gs_verify_finish_dev(eng.h, ty, count, 2, vp(parts.data_ptr()), dp[3], vp(ok2.data_ptr())) == OK
    assert lib.gs_verify_batch_rand_dev(eng.h, ty, count, M, N, *dp, ctypes.cast(r, vp), vp(ok1.data_ptr())) == OK
    torch.cuda.synchronize()
    assert bytes(ok.cpu().numpy()) == want
    assert bytes(ok2.cpu().numpy()) == want
    assert bool(ok1.item()) is want_rand
