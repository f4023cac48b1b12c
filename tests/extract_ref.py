"""Big-integer restatement of extraction with the binding key (gs_extract), on the oracle's types: the reference the
extraction tests compare against.  TEST INFRASTRUCTURE ONLY, like oracle/.

generate_crs(p1, p2, a1, a2, t1, t2) gives u[0] = (p1, a1 p1), u[1] = t1 u[0] (v likewise with a2), so every commitment
under that key has c.1 = X + a1 c.0 and
    X = c.1 - a1 c.0                 (batch_commit_G1;  batch_commit_scalar_to_B1 gives x p1)
    Y = d.1 - a2 d.0                 (batch_commit_G2;  batch_commit_scalar_to_B2 gives y p2)
A key matches a CRS iff it opens u[0] and u[1] (v[0] and v[1]) to the identity."""
from oracle import gs as ogs
from oracle.bls12_381 import G1, G2, g1_mul, g2_mul


def extract_g1(com, a1):
    return G1.add(com[1], G1.neg(g1_mul(com[0], a1)))


def extract_g2(com, a2):
    return G2.add(com[1], G2.neg(g2_mul(com[0], a2)))


def key_matches(crs: ogs.CRS, a1, a2):
    """(G1 side, G2 side): does the key open the CRS's own commitments to the identity?"""
    return (all(extract_g1(u, a1) is None for u in crs.u), all(extract_g2(v, a2) is None for v in crs.v))
