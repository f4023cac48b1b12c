"""Zero knowledge for PPE targets given as pairs, on the big-integer oracle (no CUDA): the augmented statement of
gs_zk_ppe_*_batch (zk_ref.py) is complete, sound where the fixed delta commitment W2 matters, and simulatable for target
pairs nobody knows a witness for."""
import pytest

from gsutil import SeededRng, make_crs
from oracle import gs as ogs
from oracle.bls12_381 import G1, R, g1_mul, g2_mul
from simulate_ref import hiding_crs
import zk_ref


@pytest.fixture(scope="module")
def keys():
    crs, (p1, p2, a1, a2, t1, t2) = make_crs(6)
    return crs, hiding_crs(crs), t1, t2


def draws(m, n, K, rng):
    """R ((m + K) x 2), S (n x 2), T (2 x 2), T_1..T_K (1 x 2): the engine's order"""
    d = lambda r, c: [[rng.fr() for _ in range(c)] for _ in range(r)]
    return d(m + K, 2), d(n, 2), d(2, 2), [d(1, 2) for _ in range(K)]


def satisfied(m, n, K, crs, rng):
    """a random PPE with witnesses, and K pairs whose pairing product is its value (the last pair absorbs the rest);
    also the discrete logs q_k of the Q_k"""
    g1, g2 = crs.g1_gen, crs.g2_gen
    xs, ys = [rng.fr() for _ in range(m)], [rng.fr() for _ in range(n)]
    a, b = [rng.fr() for _ in range(n)], [rng.fr() for _ in range(m)]
    gam = [[rng.fr() for _ in range(n)] for _ in range(m)]
    val = (sum(a[j] * ys[j] for j in range(n)) + sum(xs[i] * b[i] for i in range(m)) +
           sum(gam[i][j] * xs[i] * ys[j] for i in range(m) for j in range(n))) % R
    ps, qs = [rng.fr() for _ in range(K)], [rng.fr() for _ in range(K - 1)]
    rest = (val - sum(p * q for p, q in zip(ps, qs))) % R
    qs.append(rest * pow(ps[-1], -1, R) % R)
    pairs = [(g1_mul(g1, p), g2_mul(g2, q)) for p, q in zip(ps, qs)]
    return ([g1_mul(g1, v) for v in a], [g2_mul(g2, v) for v in b], gam, pairs,
            [g1_mul(g1, v) for v in xs], [g2_mul(g2, v) for v in ys], qs)


SHAPES = [(1, 1, 1), (1, 1, 2), (2, 2, 1), (2, 2, 2)]


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_real_proofs_verify_and_forged_delta_fails_under_the_binding_key(keys, m, n, K):
    crs = keys[0]
    rng = SeededRng(1000 + 100 * m + 10 * n + K)
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    R_, S, T, Ts = draws(m, n, K, rng)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, R_, S, T, Ts)
    assert zk_ref.verify(a, b, gam, pairs, proof, crs)
    # any other commitment of delta: 2 W2 (delta = 2), or W2 + r v[0] (delta = 1, but not the fixed commitment)
    w2 = ogs.w2(crs)
    assert not zk_ref.verify(a, b, gam, pairs, proof, crs, delta_com=ogs.com2_scalar_mul(w2, 2))
    assert not zk_ref.verify(a, b, gam, pairs, proof, crs, delta_com=ogs.com2_add(w2, ogs.com2_scalar_mul(crs.v[0], 5)))


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_z_other_than_p_fails_under_the_binding_key(keys, m, n, K):
    """the prover run with Z_K = P_K + g1 instead of P_K: L_K (and PPE') reject, delta's commitment being W2"""
    crs = keys[0]
    rng = SeededRng(1100 + 100 * m + 10 * n + K)
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    Z = [p for p, _ in pairs]
    Z[-1] = G1.add(Z[-1], crs.g1_gen)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(m, n, K, rng), Z=Z)
    assert not zk_ref.verify(a, b, gam, pairs, proof, crs)


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_simulated_proofs_of_false_targets_verify_under_the_hiding_key_only(keys, m, n, K):
    crs, hid, t1, t2 = keys
    rng = SeededRng(1200 + 100 * m + 10 * n + K)
    a, b, gam, pairs, _, _, _ = satisfied(m, n, K, hid, rng)
    pairs = [(g1_mul(hid.g1_gen, rng.fr()), g2_mul(hid.g2_gen, rng.fr())) for _ in range(K)]   # no known witness
    R_, S, T, Ts = draws(m, n, K, rng)
    sim = zk_ref.simulate(a, b, gam, pairs, hid, t1, t2, R_, S, T, Ts)
    assert zk_ref.verify(a, b, gam, pairs, sim, hid)
    assert not zk_ref.verify(a, b, gam, pairs, sim, crs)
    # each simulated L_k is the oracle prove with Z_k = O, delta = 0 under randomness t2
    ppe, lins = zk_ref.augmented(a, b, gam, pairs)
    for k, L in enumerate(lins):
        xc = ogs.commit_and_prove(L, [None], [0], hid, [R_[m + k]], [[t2]], Ts[k])
        assert xc.xcoms.coms[0] == sim[0].coms[m + k] and xc.ycoms.coms[0] == ogs.w2(hid)
        assert (xc.equ_proofs[0].pi, xc.equ_proofs[0].theta) == (sim[3][k].pi, sim[3][k].theta)


@pytest.mark.parametrize("m,n", [(1, 1), (2, 2)])
def test_z_that_satisfies_ppe_prime_but_not_p_is_caught_by_the_linear_equations(keys, m, n):
    """Z_1 = P_1 + a g1, Z_2 = P_2 + b g1 with a q_1 + b q_2 = 0: PPE' alone holds for this Z (the target shifts cancel),
    so only the equations Z_k - delta P_k = O, with delta fixed by W2, reject the proof under the binding key"""
    crs = keys[0]
    rng = SeededRng(1300 + 10 * m + n)
    a, b, gam, pairs, X, Y, qs = satisfied(m, n, 2, crs, rng)
    s = rng.fr()
    shift = [s, (-s * qs[0] * pow(qs[1], -1, R)) % R]
    Z = [G1.add(p, g1_mul(crs.g1_gen, d)) for (p, _), d in zip(pairs, shift)]
    xcoms, ycoms, pf, lin = proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(m, n, 2, rng), Z=Z)
    ppe, lins = zk_ref.augmented(a, b, gam, pairs)
    assert ogs.verify(ppe, ogs.CProof(xcoms, ycoms, [pf]), crs)
    for k, L in enumerate(lins):
        xc, yc = zk_ref.lin_coms(xcoms, m, k, crs)
        assert not ogs.verify(L, ogs.CProof(xc, yc, [lin[k]]), crs)
    assert not zk_ref.verify(a, b, gam, pairs, proof, crs)


def test_empty_batches_are_empty_lists():
    """the C ABI returns GS_OK for count 0; the host API returns no proofs / verdicts without touching an engine"""
    from groth_sahai_rs_b200 import api
    assert api.zk_prove_batch([], [], [], None, None) == []
    assert api.zk_simulate_batch([], None, None, None) == []
    assert api.zk_verify_batch([], [], None) == []
