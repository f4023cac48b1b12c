"""Rerandomisation of zero-knowledge PPE proofs on the big-integer oracle (no CUDA): the formulas of
gs_zk_ppe_rerandomize_batch (zk_rerand_ref.py) give exactly the real prover's or the simulator's proof under the combined
randomness, keep a bad proof bad, and need ONE R' row per Z_k for PPE' and L_k together."""
import pytest

from gsutil import SeededRng, make_crs
from oracle import gs as ogs
from oracle.bls12_381 import g1_mul, g2_mul
from simulate_ref import hiding_crs
from test_zk_oracle import draws, satisfied
import rerand_ref
import zk_ref
import zk_rerand_ref


@pytest.fixture(scope="module")
def keys():
    crs, (p1, p2, a1, a2, t1, t2) = make_crs(8)
    return crs, hiding_crs(crs), t1, t2


SHAPES = [(1, 1, 1), (1, 1, 2), (2, 2, 1), (2, 2, 2)]


def same(p, q):
    """the same commitments, PPE' proof and L_k proofs"""
    return (p[0].coms == q[0].coms and p[1].coms == q[1].coms and (p[2].pi, p[2].theta) == (q[2].pi, q[2].theta) and
            [(e.pi, e.theta) for e in p[3]] == [(e.pi, e.theta) for e in q[3]])


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_rerandomised_real_proof_is_the_fresh_proof_under_the_combined_randomness(keys, m, n, K):
    crs = keys[0]
    rng = SeededRng(2000 + 100 * m + 10 * n + K)
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    rands, rands2 = draws(m, n, K, rng), draws(m, n, K, rng)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *rands)
    out = zk_rerand_ref.rerandomize(a, b, gam, pairs, proof, crs, *rands2)
    fresh = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *zk_rerand_ref.combined(a, b, gam, pairs, rands, rands2))
    assert same(out, fresh)
    assert out[0].coms != proof[0].coms and out[3][0].pi != proof[3][0].pi
    assert zk_ref.verify(a, b, gam, pairs, out, crs)


@pytest.mark.parametrize("m,n,K", SHAPES)
def test_rerandomised_simulated_proof_is_the_simulation_under_the_combined_randomness(keys, m, n, K):
    crs, hid, t1, t2 = keys
    rng = SeededRng(2100 + 100 * m + 10 * n + K)
    a, b, gam, _, _, _, _ = satisfied(m, n, K, hid, rng)
    pairs = [(g1_mul(hid.g1_gen, rng.fr()), g2_mul(hid.g2_gen, rng.fr())) for _ in range(K)]   # no known witness
    rands, rands2 = draws(m, n, K, rng), draws(m, n, K, rng)
    sim = zk_ref.simulate(a, b, gam, pairs, hid, t1, t2, *rands)
    out = zk_rerand_ref.rerandomize(a, b, gam, pairs, sim, hid, *rands2)
    fresh = zk_ref.simulate(a, b, gam, pairs, hid, t1, t2, *zk_rerand_ref.combined(a, b, gam, pairs, rands, rands2))
    assert same(out, fresh)
    assert zk_ref.verify(a, b, gam, pairs, out, hid)
    assert not zk_ref.verify(a, b, gam, pairs, out, crs)


def test_fixed_base_lin_terms_equal_the_generic_rerandomisation(keys):
    """L_k's fixed-base formula is gs_rerandomize of the MSMEG1 equation on ([c_{m+k}], [W2]) with x_rand = row m + k of
    R' and y_rand [0]; the x-commitment it returns is PPE''s c'_{m+k}"""
    crs = keys[0]
    m, n, K = 2, 2, 2
    rng = SeededRng(2200)
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(m, n, K, rng))
    R2, S2, T2, Ts2 = draws(m, n, K, rng)
    out = zk_rerand_ref.rerandomize(a, b, gam, pairs, proof, crs, R2, S2, T2, Ts2)
    _, lins = zk_ref.augmented(a, b, gam, pairs)
    for k, L in enumerate(lins):
        xc, yc = zk_ref.lin_coms(proof[0], m, k, crs)
        gen = rerand_ref.rerandomize(L, ogs.CProof(xc, yc, [proof[3][k]]), crs, [R2[m + k]], [[0]], Ts2[k])
        assert gen.ycoms.coms == [ogs.w2(crs)] and gen.xcoms.coms == [out[0].coms[m + k]]
        assert (gen.equ_proofs[0].pi, gen.equ_proofs[0].theta) == (out[3][k].pi, out[3][k].theta)


@pytest.mark.parametrize("m,n,K", [(1, 1, 1), (2, 2, 2)])
@pytest.mark.parametrize("where", ["ppe_theta", "lin_pi"])
def test_tampered_proof_is_still_rejected(keys, m, n, K, where):
    """the verification error of a tampered element survives rerandomisation"""
    crs = keys[0]
    rng = SeededRng(2300 + 100 * m + 10 * n + K + (0 if where == "ppe_theta" else 5))
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    xc, yc, pf, lin = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(m, n, K, rng))
    if where == "ppe_theta":
        pf = ogs.EquProof(pf.pi, [ogs.com1_add(pf.theta[0], (None, crs.g1_gen))] + pf.theta[1:], pf.equ_type, [])
    else:
        e = lin[-1]
        lin = lin[:-1] + [ogs.EquProof([e.pi[0], ogs.com2_add(e.pi[1], (None, crs.g2_gen))], e.theta, e.equ_type, [])]
    bad = (xc, yc, pf, lin)
    assert not zk_ref.verify(a, b, gam, pairs, bad, crs)
    out = zk_rerand_ref.rerandomize(a, b, gam, pairs, bad, crs, *draws(m, n, K, rng))
    assert not zk_ref.verify(a, b, gam, pairs, out, crs)


@pytest.mark.parametrize("m,n,K", [(1, 1, 1), (2, 2, 2)])
def test_separate_rerandomisation_of_the_linear_equations_is_rejected(keys, m, n, K):
    """L_k rerandomised with its own R' row for Z_k -- as a call on L_k alone would -- while PPE' moves c_{m+k} by
    another: L_k no longer verifies on the shared commitment, so the whole proof is rejected"""
    crs = keys[0]
    rng = SeededRng(2400 + 100 * m + 10 * n + K)
    a, b, gam, pairs, X, Y, _ = satisfied(m, n, K, crs, rng)
    proof = zk_ref.prove(a, b, gam, pairs, X, Y, crs, *draws(m, n, K, rng))
    R2, S2, T2, Ts2 = draws(m, n, K, rng)
    other = [[rng.fr(), rng.fr()] for _ in range(K)]
    out = zk_rerand_ref.rerandomize(a, b, gam, pairs, proof, crs, R2, S2, T2, Ts2, lin_rows=other)
    ppe, lins = zk_ref.augmented(a, b, gam, pairs)
    assert ogs.verify(ppe, ogs.CProof(out[0], out[1], [out[2]]), crs)
    assert not zk_ref.verify(a, b, gam, pairs, out, crs)
    assert zk_ref.verify(a, b, gam, pairs, zk_rerand_ref.rerandomize(a, b, gam, pairs, proof, crs, R2, S2, T2, Ts2), crs)


def test_empty_batch_is_an_empty_list():
    """the host API returns no proofs without touching an engine"""
    from groth_sahai_rs_b200 import api
    assert api.zk_rerandomize_batch([], [], None, None) == []
