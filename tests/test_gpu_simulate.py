"""gs_simulate / gs_simulate_batch on the GPU.  Expected bytes are built without the engine: the C oracle's reference-order
commit + prove of the AUGMENTED equation (simulate_ref.py) with zero witnesses under the hiding key.  The statements have
random targets (PPE: target 1).  Every path of the proof-element MSMs is taken: the split lone call, one thread per
product (big batches, across the 32,768-proof chunk), the shared-scalar constant sums (many equations over one set of
commitments) and the bucket MSM (one 2048 x 2048 statement).  Every output is checked by the three GPU verifiers under
the hiding key."""
import ctypes
import random

import pytest

from bigcase import *  # noqa: F401,F403
from simulate_ref import hiding_crs

pytestmark = pytest.mark.gpu

OK, EDIM, EARG = 0, 1, 3
vp = ctypes.c_void_p


@pytest.fixture(scope="module")
def keys():
    crs, (_, _, _, _, t1, t2) = make_crs(2)
    return crs, hiding_crs(crs), t1, t2


@pytest.fixture(scope="module")
def eng(keys):
    import groth_sahai_rs_b200 as gsb
    e = gsb.Engine(0)
    e.crs_load(crs_bytes(keys[1]))
    yield e
    e.close()


def tkey_b(t1, t2):
    return fr_b(t1) + fr_b(t2)


class SimCase:
    """`E` statements of one type and shape with random targets, the simulator's randomness (one R, S for all with
    `shared`), and the augmented equations' byte arrays for the C oracle."""

    def __init__(self, ty, m, n, hid, seed, E=1, shared=False):
        rng = SeededRng(seed)
        self.ty, self.m, self.n, self.E, self.shared = ty, m, n, E, shared
        cx, cy = cb.cx_of(ty), cb.cy_of(ty)
        a = [fr_list(rng, n) for _ in range(E)]
        b = [fr_list(rng, m) for _ in range(E)]
        self.gam = [[fr_list(rng, n) for _ in range(m)] for _ in range(E)]
        tv = fr_list(rng, E)                                  # discrete logs of the targets (PPE: target 1)
        flat = lambda rows: [x for r in rows for x in r]
        self.A, self.B = bigcase_sides(hid, ty, flat(a), flat(b))
        self.G = b"".join(frmat_b(g) for g in self.gam)
        if ty == 0:
            self.T, self.negT = fp12_b(FP12_ONE) * E, None
        elif ty == 1:
            self.T, self.negT = b"".join(g1_multiples(hid, tv)), g1_multiples(hid, [(-v) % R for v in tv])
        elif ty == 2:
            self.T, self.negT = b"".join(g2_multiples(hid, tv)), g2_multiples(hid, [(-v) % R for v in tv])
        else:
            self.T, self.negT = frs_b(tv), [fr_b((-v) % R) for v in tv]
        reps = 1 if shared else E
        self.xr, self.yr = fr_list(rng, reps * m * cx), fr_list(rng, reps * n * cy)
        self.Tr = fr_list(rng, E * cx * cy)

    def args(self):
        return (self.A, self.B, self.G, self.T, frs_b(self.xr), frs_b(self.yr), frs_b(self.Tr))

    def expected(self, hid, t1, t2, e=None):
        """C oracle commit + prove of equation e's augmented statement (all equations as one shared batch when e is None)"""
        ty, m, n = self.ty, self.m, self.n
        cx, cy = cb.cx_of(ty), cb.cy_of(ty)
        es = range(self.E) if e is None else [e]
        k = 0 if self.shared else es[0]
        xr = self.xr[k * m * cx:(k + 1) * m * cx]
        yr = self.yr[k * n * cy:(k + 1) * n * cy]
        asz, bsz = cb.x_size(ty), cb.y_size(ty)
        A = [self.A[i * n * asz:(i + 1) * n * asz] for i in es]
        B = [self.B[i * m * bsz:(i + 1) * m * bsz] for i in es]
        G = [self.gam[i] for i in es]
        mm, nn = m, n
        if ty in (1, 3):      # one more y-variable: randomness [t2], constant -T1 / -t, a zero column of Gamma
            A = [a + self.negT[i] for a, i in zip(A, es)]
            G = [[r + [0] for r in g] for g in G]
            yr = yr + [t2]
            nn += 1
        if ty == 2:           # one more x-variable: randomness [t1], constant -T2, a zero row of Gamma
            B = [b + self.negT[i] for b, i in zip(B, es)]
            G = [g + [[0] * n] for g in G]
            xr = xr + [t1]
            mm += 1
        X, Y = bytes(mm * asz), bytes(nn * bsz)
        crsb = crs_bytes(hid)
        xc = cb.commit_x(ty, X, frs_b(xr), crsb, NT)[:m * 192]
        yc = cb.commit_y(ty, Y, frs_b(yr), crsb, NT)[:n * 384]
        Ts = frs_b([x for i in es for x in self.Tr[i * cx * cy:(i + 1) * cx * cy]])
        Gb = b"".join(frmat_b(g) for g in G) if ty != 0 else b"".join(self.G[i * m * n * 32:(i + 1) * m * n * 32] for i in es)
        if e is not None:
            pi, th = cb.prove(ty, mm, nn, A[0], B[0], Gb, X, Y, frs_b(xr), frs_b(yr), Ts, crsb, NT)
        else:
            pi, th = cb.prove_batch(ty, len(es), mm, nn, b"".join(A), b"".join(B), Gb, X, Y, frs_b(xr), frs_b(yr), Ts, True,
                                    crsb, NT)
        return xc, yc, pi, th


def bigcase_sides(crs, ty, a, b):
    A = b"".join(g1_multiples(crs, a)) if ty in (0, 1) else frs_b(a)
    B = b"".join(g2_multiples(crs, b)) if ty in (0, 2) else frs_b(b)
    return A, B


def verify_all(eng, c, out, target=None):
    """(gs_verify_batch bytes, gs_verify_batch_rand verdict, gs_verify_each_rand bytes) under the loaded key"""
    xc, yc, pi, th = out
    reps = c.E if c.shared else 1
    args = (c.ty, c.E, c.m, c.n, c.A, c.B, c.G, target or c.T, xc * reps, yc * reps, pi, th)
    rho = random.Random(c.E).randbytes(8 * (2 * c.E + 1))
    return eng.verify_batch(*args), eng.verify_batch_rand(*args, rho=rho), eng.verify_each_rand(*args, rho=rho)


def other_target(c, hid):
    """new targets for every statement (PPE: the GT generator instead of 1)"""
    if c.ty == 0:
        return fp12_b(hid.gt_gen) * c.E
    ks = [7 + i for i in range(c.E)]
    return {1: lambda: b"".join(g1_multiples(hid, ks)), 2: lambda: b"".join(g2_multiples(hid, ks)), 3: lambda: frs_b(ks)}[c.ty]()


def check_verifiers(eng, c, out, hid):
    ok, ok_rand, ok_each = verify_all(eng, c, out)
    assert ok == b"\x01" * c.E and ok_rand is True and ok_each == b"\x01" * c.E
    bad, bad_rand, bad_each = verify_all(eng, c, out, target=other_target(c, hid))
    assert bad == b"\x00" * c.E and bad_rand is False and bad_each == b"\x00" * c.E


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
@pytest.mark.parametrize("m,n", [(4, 4), (1, 3), (3, 1)])
def test_lone_call_equals_prove_of_the_augmented_equation(eng, keys, ty, m, n):
    _, hid, t1, t2 = keys
    c = SimCase(ty, m, n, hid, seed=2000 + 10 * ty + m)
    out = eng.simulate(ty, m, n, *c.args(), tkey_b(t1, t2))
    assert out == c.expected(hid, t1, t2, 0)
    assert eng.simulate(ty, m, n, *c.args(), tkey_b(t1, t2)) == out            # the same call twice: the same bytes
    assert eng.simulate_batch(ty, 1, m, n, *c.args(), tkey_b(t1, t2)) == out   # the batch entry point with count 1
    check_verifiers(eng, c, out, hid)


def test_big_batch_one_thread_per_product(eng, keys):
    """32,768 + 512 independent 4 x 4 MSMEG1 statements (target column on theta): one thread per product in the first
    chunk, the split path and two streams in the second; every output verifies, a sample is checked byte for byte."""
    _, hid, t1, t2 = keys
    ty, m, n, count = 1, 4, 4, 32768 + 512
    c = SimCase(ty, m, n, hid, seed=2100, E=count)
    out = eng.simulate_batch(ty, count, m, n, *c.args(), tkey_b(t1, t2))
    for i in (0, 5, 32767, 32768, count - 1):
        got = (out[0][i * m * 192:(i + 1) * m * 192], out[1][i * n * 384:(i + 1) * n * 384], out[2][i * 2 * 384:(i + 1) * 2 * 384],
               out[3][i * 192:(i + 1) * 192])
        assert got == c.expected(hid, t1, t2, i), f"proof {i}"
    check_verifiers(eng, c, out, hid)


@pytest.mark.parametrize("ty", [0, 1, 2, 3])
def test_shared_commitments_statement(eng, keys, ty):
    """256 equations over one set of 64 x 64 commitments: on group-typed sides the constants of all equations (and the
    targets, one more constant) are summed along one bucket structure (the shared-scalar path)."""
    _, hid, t1, t2 = keys
    m = n = 64
    c = SimCase(ty, m, n, hid, seed=2200 + ty, E=256, shared=True)
    out = eng.simulate_batch(ty, c.E, m, n, *c.args(), tkey_b(t1, t2), shared_coms=True)
    assert out == c.expected(hid, t1, t2)
    check_verifiers(eng, c, out, hid)


def test_2048x2048_ppe_bucket_msm(eng, keys):
    _, hid, t1, t2 = keys
    c = SimCase(0, 2048, 2048, hid, seed=2300)
    out = eng.simulate(0, 2048, 2048, *c.args(), tkey_b(t1, t2))
    assert out == c.expected(hid, t1, t2, 0)
    check_verifiers(eng, c, out, hid)


def test_return_codes_and_key_cache(eng, keys):
    import groth_sahai_rs_b200 as gsb
    crs, hid, t1, t2 = keys
    lib = eng.lib
    m = n = 4
    c = SimCase(1, m, n, hid, seed=2400)
    good = [ctypes.create_string_buffer(x, len(x)) for x in c.args()]
    key = ctypes.create_string_buffer(tkey_b(t1, t2), 64)
    outs = [ctypes.create_string_buffer(b"\xa5" * (1 << 14), 1 << 14) for _ in range(4)]
    p = [ctypes.cast(b, vp) for b in good] + [ctypes.cast(key, vp)] + [ctypes.cast(o, vp) for o in outs]

    def call(h, ty=1, count=1, mm=m, nn=n, null=None, tk=None, tgt=None):
        q = [None if i == null else x for i, x in enumerate(p)]
        if tk is not None:
            q[7] = ctypes.cast(tk, vp)
        if tgt is not None:
            q[3] = ctypes.cast(tgt, vp)
        return lib.gs_simulate_batch(h, ty, count, mm, nn, *q[:7], 0, *q[7:])

    fresh = gsb.Engine(0)
    E, F = eng.h, fresh.h
    wrong = ctypes.create_string_buffer(tkey_b(t1, (t2 + 1) % R), 64)
    swapped = ctypes.create_string_buffer(tkey_b(t2, t1), 64)
    ppe_t = ctypes.create_string_buffer(fp12_b(hid.gt_gen), 576)
    cases = {
        "bad type": (call(E, ty=4), EARG),
        "negative type": (call(E, ty=-1), EARG),
        "no crs": (call(F), EARG),
        "count 0": (call(E, count=0), OK),
        "m 0": (call(E, mm=0), EDIM),
        "n 0": (call(E, nn=0), EDIM),
        "too many variables": (call(E, mm=(1 << 22) + 1), EDIM),
        "wrong key": (call(E, tk=wrong), EARG),
        "swapped key": (call(E, tk=swapped), EARG),
        "ppe target not 1": (call(E, ty=0, tgt=ppe_t), EARG),
    }
    for i in range(12):
        cases[f"null argument {i}"] = (call(E, null=i), EARG)
    assert all(o.raw == b"\xa5" * (1 << 14) for o in outs)        # nothing written by a refused call
    assert lib.gs_simulate(E, 1, 0, n, *p) == EDIM and lib.gs_simulate(E, 9, m, n, *p) == EARG
    # the key is cached per CRS: a binding CRS of the same draws refuses it after gs_crs_load, the hiding one takes it again
    assert call(E) == OK
    fresh.crs_load(crs_bytes(crs))
    cases["binding crs"] = (call(F), EARG)
    eng.crs_load(crs_bytes(crs))
    cases["cached key after loading the binding crs"] = (call(E), EARG)
    eng.crs_load(crs_bytes(hid))
    cases["hiding crs reloaded"] = (call(E), OK)
    fresh.close()
    got = {k: v[0] for k, v in cases.items()}
    assert got == {k: v[1] for k, v in cases.items()}


def test_api_round_trip():
    """generate_hiding_crs_with_trapdoor -> simulate -> serialize -> verify through the host API; the trapdoor generator
    makes exactly generate_hiding_crs's draws."""
    import groth_sahai_rs_b200 as gsb
    from groth_sahai_rs_b200 import api
    from test_gpu_api_mirror import ReplayRng
    eng = gsb.Engine(0)
    crs, key = api.CRS.generate_hiding_crs_with_trapdoor(ReplayRng(91), eng)
    assert crs == api.CRS.generate_hiding_crs(ReplayRng(91), eng)
    rng = ReplayRng(91)
    api.CRS.generate_hiding_crs(rng, eng)
    assert key == api.SimulationKey(fr_b(rng.log[4]), fr_b(rng.log[5]))
    assert api.SimulationKey.from_bytes(key.to_bytes()) == key
    binding, _ = api.CRS.generate_crs_with_trapdoor(ReplayRng(91), eng)
    crs_o = hiding_crs(ogs.generate_crs(*rng.log[:6]))
    for ty in (0, 1, 2, 3):
        c = SimCase(ty, 2, 3, crs_o, seed=2500 + ty, E=2)
        cls = [api.PPE, api.MSMEG1, api.MSMEG2, api.QuadEqu][ty]
        asz, bsz, tsz = cb.x_size(ty), cb.y_size(ty), cb.target_size(ty)
        eqs = [cls([c.A[(e * 3 + j) * asz:(e * 3 + j + 1) * asz] for j in range(3)],
                   [c.B[(e * 2 + i) * bsz:(e * 2 + i + 1) * bsz] for i in range(2)],
                   [[fr_b(g) for g in row] for row in c.gam[e]], c.T[e * tsz:(e + 1) * tsz]) for e in range(2)]
        cp = eqs[0].simulate(crs, key, ReplayRng(7))
        assert eqs[0].verify(cp, crs) is True and cp.xcoms.rand == [] and cp.equ_proofs[0].rand == []
        assert api.simulate_batch([eqs[0]], crs, key, ReplayRng(7))[0] == cp
        back = api.CProof(api.deserialize_commit(api.serialize_commit(cp.xcoms, eng), 1, eng),
                          api.deserialize_commit(api.serialize_commit(cp.ycoms, eng), 2, eng),
                          [api.deserialize_equ_proof(api.serialize_equ_proof(cp.equ_proofs[0], eng), eng)])
        assert eqs[0].verify(back, crs) is True
        both = api.simulate_batch(eqs, crs, key, ReplayRng(8), shared_commitments=True)
        assert both[0].xcoms.coms == both[1].xcoms.coms
        assert api.verify_batch(eqs, both, crs) == [True, True]
        assert eqs[0].verify(cp, binding) is False
        with pytest.raises(gsb.GsError):
            eqs[0].simulate(binding, key, ReplayRng(7))
    eng.close()
