"""Every GPU verifier against proofs that are wrong in exactly one ComT entry (entry_ref.py, confirmed by the oracle in
test_entry_oracle.py).  A verifier that compared fewer than four entries, permuted them, or weighted two of them alike in
the randomised fold would still pass tampers that change entry (1, 1), as every other tamper of the suite does; these
proofs leave that entry alone.  Checked: exact verdicts of gs_verify_batch / _dev, the final-exponentiated values of
gs_verify_partial (1 and several ranks) against the oracle's per-entry ratios, gs_verify_finish, gs_verify_sharded,
gs_verify_batch_rand, gs_verify_each_rand (with a proof built to cancel under one set of weights), gs_zk_ppe_verify_batch,
and the verify paths that big or lone batches take (passes, pass streams, halves, chunked accumulators, shared
commitments, bucket sums)."""
import os
import random
from contextlib import contextmanager

import pytest

from entry_ref import *  # noqa: F401,F403

pytestmark = pytest.mark.gpu

M = N = 2
KEYS = [False, True]
KEY_IDS = ["binding", "hiding"]


@pytest.fixture(scope="module")
def draws():
    return make_crs(1)[1]


@pytest.fixture(scope="module")
def eng():
    import groth_sahai_rs_b200 as gsb
    e = gsb.Engine(0)
    yield e
    e.close()


@contextmanager
def engine_with(key, **env):
    """a fresh Engine created under the GS_* settings `env` (read at creation), the environment restored after"""
    import groth_sahai_rs_b200 as gsb
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        e = gsb.Engine(0)
    finally:
        for k, v in old.items():
            os.environ.pop(k, None) if v is None else os.environ.__setitem__(k, v)
    e.crs_load(key.crsb)
    try:
        yield e
    finally:
        e.close()


def rho_of(count, seed):
    return random.Random(seed).randbytes(8 * (2 * count + 1))


def join(rows):
    return [b"".join(r[k] for r in rows) for k in range(8)]


def cancelling():
    return [[[1, 0], [0, R - 1]], [[0, 1], [R - 1, 0]]]


def planted_batch(key, ty, m, n, count, plant, seed):
    """count proofs of distinct honest cases (cycled), proof p replaced by a tamper of its case with error plant[p]"""
    cases = [Case(ty, m, n, key.crs, seed=seed + i) for i in range(min(count, 6))]
    rows = []
    for p in range(count):
        c = cases[p % len(cases)]
        rows.append(tamper(key, c, plant[p]) if p in plant else c.verify_arrays())
    return join(rows), bytes(0 if p in plant else 1 for p in range(count)), cases


def values_ok(e, key, ty, m, n, arrays, count, p, E):
    """the final-exponentiated entries of proof p's gs_verify_partial (one rank) are gt_gen^E (times the PPE target): the
    planted error sits where it was planted, whatever the shape"""
    return finish(e.verify_partial(ty, count, m, n, *arrays, 0, 1), p, count) == expected_values(key, ty, arrays, p, E)


def expected_values(key, ty, arrays, p, E):
    """the four final-exponentiated entries a partial of proof p must give: gt_gen^E, times the target in entry 3 (PPE)"""
    want = gt_of(key.crs, E or [[0, 0], [0, 0]])
    if ty == 0:
        want[3] = want[3] * fp12_i(arrays[3][576 * p:576 * (p + 1)])
    return want


@pytest.mark.parametrize("hiding", KEYS, ids=KEY_IDS)
@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_one_entry_errors_on_every_exact_path(eng, draws, ty, hiding):
    """single-entry errors (row / column errors where single entries are unreachable) and, where reachable, the two
    cancelling pairs, placed between honest proofs: exact verdicts on every exact path, and the VALUES of each entry"""
    import torch
    from test_gpu_scale import _sharded_on_one_gpu
    key = Key(draws, hiding)
    eng.crs_load(key.crsb)
    errs = errors(key, ty, lam=5) + (cancelling() if reachable(key, ty) else [])
    count = 2 * len(errs) + 1
    plant = {2 * k + 1: E for k, E in enumerate(errs)}
    arrays, want, _ = planted_batch(key, ty, M, N, count, plant, seed=6000 + 20 * ty + 10 * hiding)
    assert eng.verify_batch(ty, count, M, N, *arrays) == want
    dev = [torch.frombuffer(bytearray(a), dtype=torch.uint8).cuda() for a in arrays]
    ok = torch.full((count,), 7, dtype=torch.uint8, device="cuda")
    torch.cuda.synchronize()
    eng.verify_batch_dev(ty, count, M, N, [d.data_ptr() for d in dev], ok.data_ptr())
    torch.cuda.synchronize()
    assert bytes(ok.cpu().numpy()) == want
    # values, not just verdicts: this catches permuted entries too
    check = [0] + sorted(plant)
    for world in (1, 2, 3):
        parts = b"".join(eng.verify_partial(ty, count, M, N, *arrays, r, world) for r in range(world))
        for p in check:
            assert finish(parts, p, count) == expected_values(key, ty, arrays, p, plant.get(p)), (world, p)
        assert eng.verify_finish(ty, count, parts, arrays[3]) == want, world
    for world in (2, 3):
        assert _sharded_on_one_gpu(ty, count, M, N, arrays, key.crsb, world) == [want] * world
    # randomised: every batch with one such proof is rejected, each one is flagged on its own
    assert eng.verify_each_rand(ty, count, M, N, *arrays, rho=rho_of(count, 1)) == want
    sz = [len(a) // count for a in arrays]
    honest = [b"".join(a[s * p:s * (p + 1)] for p in range(count) if p not in plant) for a, s in zip(arrays, sz)]
    nh = count - len(plant)
    assert eng.verify_batch_rand(ty, nh, M, N, *honest, rho=rho_of(nh, 2)) is True
    for k, p in enumerate(sorted(plant)):
        one = [h + a[s * p:s * (p + 1)] for h, a, s in zip(honest, arrays, sz)]
        assert eng.verify_batch_rand(ty, nh + 1, M, N, *one, rho=rho_of(nh + 1, 3 + k)) is False, plant[p]


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_weight_cancelling_proof_pins_the_weights(eng, draws, ty):
    """A proof whose error cancels under the weights of one rho: the randomised verifiers accept it with that rho, as the
    documented fold (sigma_p = rho[2p], tau_p = rho[2p + 1] to 63 bits, beta = lo32 + hi32 |x| of rho[2 count]) requires,
    and reject it once a used bit changes; bit 63 of sigma_p and tau_p is unused.  The exact verifier rejects it."""
    key = Key(draws)
    eng.crs_load(key.crsb)
    count, p = 5, 2
    rho = rho_of(count, 700 + ty)
    E = weight_cancelling(*weights_of(rho, p, count))
    arrays, want, _ = planted_batch(key, ty, M, N, count, {p: E}, seed=7000 + 10 * ty)
    assert eng.verify_batch(ty, count, M, N, *arrays) == want
    assert eng.verify_each_rand(ty, count, M, N, *arrays, rho=rho) == b"\x01" * count
    assert eng.verify_batch_rand(ty, count, M, N, *arrays, rho=rho) is True
    for word, bit in ((2 * p, 0), (2 * p, 62), (2 * p + 1, 1), (2 * p + 1, 40), (2 * count, 0), (2 * count, 33),
                      (2 * count, 63)):
        r = flip_bit(rho, word, bit)
        assert eng.verify_each_rand(ty, count, M, N, *arrays, rho=r) == want, (word, bit)
        assert eng.verify_batch_rand(ty, count, M, N, *arrays, rho=r) is False, (word, bit)
    for word in (2 * p, 2 * p + 1):
        r = flip_bit(rho, word, 63)
        assert eng.verify_each_rand(ty, count, M, N, *arrays, rho=r) == b"\x01" * count
        assert eng.verify_batch_rand(ty, count, M, N, *arrays, rho=r) is True


def test_zk_statement_with_one_entry_error(eng, draws):
    """gs_zk_ppe_verify_batch: an error in one entry of the PPE' proof of the middle statement fails that statement only"""
    from test_gpu_zk import ZkCase
    key = Key(draws)
    eng.crs_load(key.crsb)
    m, n, K, S = 2, 2, 1, 3
    c = ZkCase(m, n, K, key.crs, seed=7100, E=S)
    out = list(eng.zk_ppe_prove_batch(S, m, n, K, *c.stmt(), c.X, c.Y, *c.rand()))
    stmt = list(c.stmt())
    assert eng.zk_ppe_verify_batch(S, m, n, K, *stmt, *out) == b"\x01" * S
    s, i, j = 1, 1, 0
    cl = key.com_x(0, c.xs[s * m + i], c.xr[(s * (m + K) + i) * 2:][:2])
    dl = key.com_y(0, c.ys[s * n + j], c.yr[(s * n + j) * 2:][:2])
    for e in (0, 2, 3, 1):
        g, pi, th = tamper_arrays(key, 0, m, n, stmt[2], out[2], out[3], cl, dl, unit(e, 3), s, i, j)
        bad = stmt[:2] + [g] + stmt[3:]
        assert eng.zk_ppe_verify_batch(S, m, n, K, *bad, out[0], out[1], pi, th, *out[4:]) == b"\x01\x00\x01", e
    # the last tamper's values: PPE' of statement s (x-variables X | Z, constants B | -Q, Gamma with K zero rows, target 1)
    a, b, _ = c.ppe_prime()
    cut = lambda buf, k: buf[s * k:(s + 1) * k]
    ppe = [cut(a, n * 96), cut(b, (m + K) * 192), cut(g, m * n * 32) + bytes(32 * n * K), fp12_b(FP12_ONE),
           cut(out[0], (m + K) * 192), cut(out[1], n * 384), cut(pi, 768), cut(th, 384)]
    assert values_ok(eng, key, 0, m + K, n, ppe, 1, 0, unit(1, 3))


@pytest.mark.parametrize("jac", [1, 0])
def test_lone_statement(draws, jac):
    """one 4 x 4 statement, both line walks of a lone statement"""
    key = Key(draws)
    with engine_with(key, GS_LONE_WALK_JAC=jac) as e:
        for ty in (0, 3):
            c = Case(ty, 4, 4, key.crs, seed=7200 + ty)
            assert e.verify(ty, 4, 4, *c.verify_arrays()) is True
            for k in range(4):
                bad = tamper(key, c, unit(k), i=k, j=3 - k)
                assert e.verify(ty, 4, 4, *bad) is False, (ty, k)
                if k == 2:
                    assert values_ok(e, key, ty, 4, 4, bad, 1, 0, unit(k)), ty


def test_batch_of_70_warps_and_halves(draws):
    """70 proofs, more than two warps, with GS_SPLIT_MIN = 64 (a batch that size or bigger is cut in two, halves of 64 and
    6 here) against GS_SPLIT_MIN = 0 (never cut): verify_batch runs the halves as pipelined host passes on alternating
    streams, verify_batch_dev as the two-stream passes inside one call.  Errors at the first and last proof of each warp
    and half; the cut is confirmed by the kernel launches it adds."""
    import torch
    key = Key(draws)
    pos = [0, 31, 32, 34, 35, 63, 64, 69]
    launches = {}
    for split in (64, 0):
        with engine_with(key, GS_SPLIT_MIN=split) as e:
            for ty in (0, 2):
                plant = {p: unit(k % 4, k + 1) for k, p in enumerate(pos)}
                arrays, want, _ = planted_batch(key, ty, M, N, 70, plant, seed=7300 + 10 * ty)
                n0 = e.launch_count
                assert e.verify_batch(ty, 70, M, N, *arrays) == want, (split, ty)
                dev = [torch.frombuffer(bytearray(a), dtype=torch.uint8).cuda() for a in arrays]
                ok = torch.full((70,), 7, dtype=torch.uint8, device="cuda")
                torch.cuda.synchronize()
                n1 = e.launch_count
                e.verify_batch_dev(ty, 70, M, N, [d.data_ptr() for d in dev], ok.data_ptr())
                torch.cuda.synchronize()
                launches[split, ty] = (n1 - n0, e.launch_count - n1)
                assert bytes(ok.cpu().numpy()) == want, (split, ty)
                assert e.verify_each_rand(ty, 70, M, N, *arrays, rho=rho_of(70, 9)) == want, (split, ty)
    for ty in (0, 2):
        assert all(a > b for a, b in zip(launches[64, ty], launches[0, ty])), launches


@pytest.mark.parametrize("streams", [2, 1])
def test_exact_passes_through_the_host_pipeline(draws, streams):
    """100 proofs in passes of 40 (GS_VERIFY_BATCH_MAX = 40): pipelined uploads and alternating pass streams (2), or one
    stream (1); errors at the first and last proof of every pass; the partials come back at the right offsets"""
    key = Key(draws)
    pos = [0, 39, 40, 79, 80, 99]
    with engine_with(key, GS_VERIFY_BATCH_MAX=40, GS_PASS_STREAMS=streams) as e:
        for ty in (0, 1):
            plant = {p: unit(k % 4, 2 + k) for k, p in enumerate(pos)}
            arrays, want, _ = planted_batch(key, ty, M, N, 100, plant, seed=7400 + 10 * ty)
            assert e.verify_batch(ty, 100, M, N, *arrays) == want, ty
            parts = e.verify_partial(ty, 100, M, N, *arrays, 0, 1)
            assert e.verify_finish(ty, 100, parts, arrays[3]) == want, ty
            for p in (39, 40, 41):
                assert finish(parts, p, 100) == expected_values(key, ty, arrays, p, plant.get(p)), (ty, p)


def test_chunked_64x64_statement(eng, draws):
    """one 64 x 64 PPE: the pairing product runs in accumulator chunks multiplied before the final exponentiation"""
    key = Key(draws)
    eng.crs_load(key.crsb)
    c = Case(0, 64, 64, key.crs, seed=7500)
    assert eng.verify(0, 64, 64, *c.verify_arrays()) is True
    for k in range(4):
        bad = tamper(key, c, unit(k, 11), i=63 - k, j=17 * k)
        assert eng.verify(0, 64, 64, *bad) is False, k
        if k == 1:
            assert finish(eng.verify_partial(0, 1, 64, 64, *bad, 0, 1), 0, 1) == expected_values(key, 0, bad, 0, unit(k, 11))


@pytest.mark.parametrize("ty", [0, 3])
def test_shared_commitment_statement(eng, draws, ty):
    """16 equations over ONE set of commitments (shared_x / shared_y slots): errors in one entry of the first and the last
    equation"""
    key = Key(draws)
    eng.crs_load(key.crsb)
    E, m, n = 16, 6, 6
    st = Statement(ty, m, n, E, key.crs, seed=7600 + ty)
    arrays = st.verify_arrays()
    assert eng.verify_batch(ty, E, m, n, *arrays) == b"\x01" * E
    for k in range(4):
        bad = tamper(key, st, unit(k, 4), eq=0, i=k, j=5 - k)
        bad = tamper(key, st, unit(3 - k, 9), eq=E - 1, i=5 - k, j=k, arrays=bad)
        want = b"\x00" + b"\x01" * (E - 2) + b"\x00"
        assert eng.verify_batch(ty, E, m, n, *bad) == want, k
        assert eng.verify_each_rand(ty, E, m, n, *bad, rho=rho_of(E, 20 + k)) == want, k
        assert eng.verify_batch_rand(ty, E, m, n, *bad, rho=rho_of(E, 30 + k)) is False, k
        if k == 1:
            parts = eng.verify_partial(ty, E, m, n, *bad, 0, 1)
            assert finish(parts, 0, E) == expected_values(key, ty, bad, 0, unit(1, 4))
            assert finish(parts, E - 1, E) == expected_values(key, ty, bad, E - 1, unit(2, 9))


def test_rand_bucket_sums(draws):
    """verify_batch_rand at and above GS_RAND_PIP_MIN (the pi / theta slots summed with the bucket method)"""
    key = Key(draws)
    ty, m, n = 0, 3, 2
    with engine_with(key, GS_RAND_PIP_MIN=4096) as e:
        cases = [Case(ty, m, n, key.crs, seed=7700 + i) for i in range(12)]
        rows = [cases[q % 12].verify_arrays() for q in range(4104)]
        assert e.verify_batch_rand(ty, 4104, m, n, *join(rows), rho=rho_of(4104, 40)) is True
        for count, p, k in ((4096, 4095, 0), (4104, 0, 2), (4104, 4103, 1)):
            bad = rows[:count]
            bad[p] = tamper(key, cases[p % 12], unit(k, 6))
            assert e.verify_batch_rand(ty, count, m, n, *join(bad), rho=rho_of(count, 41 + k)) is False, (count, p, k)
        assert values_ok(e, key, ty, m, n, bad[p], 1, 0, unit(k, 6))
