"""Parity cases at the BASELINE.json shapes, built WITHOUT the engine under test: witnesses and constants are
multiples of the CRS generators computed by the C oracle (oracle/gs_oracle.c, host threads), commitments and proofs
come from the C restatement of the reference (`gsref_prove`, reference evaluation order), so a GPU result can be
byte-compared with them at 4x4, 64x64, 128x128 and 1024x1024.  Everything is in C-ABI bytes."""
from gsutil import *  # noqa: F401,F403
from oracle import cbaseline as cb

NT = cb.host_cores()


def fr_list(rng, k, zero_frac=0.0):
    return [0 if (zero_frac and rng.r.random() < zero_frac) else rng.fr() for _ in range(k)]


def g1_multiples(crs, ks):
    out = cb.g1_mul_batch(g1_b(crs.g1_gen), frs_b(ks), NT)
    return [out[96 * i:96 * (i + 1)] for i in range(len(ks))]


def g2_multiples(crs, ks):
    out = cb.g2_mul_batch(g2_b(crs.g2_gen), frs_b(ks), NT)
    return [out[192 * i:192 * (i + 1)] for i in range(len(ks))]


def _enc_side1(crs, ty, ks):
    return b"".join(g1_multiples(crs, ks)) if ty in (0, 1) else frs_b(ks)


def _enc_side2(crs, ty, ks):
    return b"".join(g2_multiples(crs, ks)) if ty in (0, 2) else frs_b(ks)


def _target(crs, ty, val):
    if ty == 0:
        return fp12_b(crs.gt_gen.pow(val))
    if ty == 1:
        return g1_multiples(crs, [val])[0]
    if ty == 2:
        return g2_multiples(crs, [val])[0]
    return fr_b(val)


def _value(a, b, gam, xs, ys):
    m, n = len(xs), len(ys)
    row = [sum(gam[i][j] * ys[j] for j in range(n)) % R for i in range(m)]
    return (sum(a[j] * ys[j] for j in range(n)) + sum(xs[i] * (b[i] + row[i]) for i in range(m))) % R


class Case:
    """One satisfied equation with its witnesses, randomness and the REFERENCE-ORDER commitments and proof."""

    def __init__(self, ty, m, n, crs, seed, zero_frac=0.0, prove=True, collide=False):
        rng = SeededRng(seed)
        self.ty, self.m, self.n, self.crs, self.crsb = ty, m, n, crs, crs_bytes(crs)
        cx, cy = cb.cx_of(ty), cb.cy_of(ty)
        xs, ys = fr_list(rng, m), fr_list(rng, n)
        a, b = fr_list(rng, n, zero_frac), fr_list(rng, m, zero_frac)
        gam = [fr_list(rng, n, zero_frac) for _ in range(m)]
        if collide and n >= 4:
            # y_1 = y_0 and y_2 = -y_0 with equal Gamma columns: inside an MSM the three terms carry the same scalar, so a
            # bucket / table sees P + P and P + (-P); scalars 1 and r - 1 ride along
            ys[1], ys[2] = ys[0], (-ys[0]) % R
            for row in gam:
                row[1] = row[2] = row[0]
            gam[0][3], gam[m - 1][3] = 1, R - 1
        self.xs, self.ys, self.a, self.b, self.gam = xs, ys, a, b, gam     # the discrete logs (tests/entry_ref.py)
        self.A, self.B = _enc_side1(crs, ty, a), _enc_side2(crs, ty, b)
        self.X, self.Y = _enc_side1(crs, ty, xs), _enc_side2(crs, ty, ys)
        self.G = frmat_b(gam)
        self.T = _target(crs, ty, _value(a, b, gam, xs, ys))
        self.xr, self.yr = frs_b(fr_list(rng, m * cx)), frs_b(fr_list(rng, n * cy))
        self.Tr = frs_b(fr_list(rng, cx * cy))
        if prove:
            self.xc = cb.commit_x(ty, self.X, self.xr, self.crsb, NT)
            self.yc = cb.commit_y(ty, self.Y, self.yr, self.crsb, NT)
            self.pi, self.theta = cb.prove(ty, m, n, self.A, self.B, self.G, self.X, self.Y, self.xr, self.yr, self.Tr,
                                           self.crsb, NT)

    def prove_args(self):
        return [self.A, self.B, self.G, self.X, self.Y, self.xr, self.yr, self.Tr]

    def verify_arrays(self):
        return [self.A, self.B, self.G, self.T, self.xc, self.yc, self.pi, self.theta]


class Statement:
    """E satisfied equations of one type over ONE set of variables (the C4 shape), proofs by the C oracle."""

    def __init__(self, ty, m, n, E, crs, seed, prove=True):
        rng = SeededRng(seed)
        self.ty, self.m, self.n, self.E, self.crs, self.crsb = ty, m, n, E, crs, crs_bytes(crs)
        cx, cy = cb.cx_of(ty), cb.cy_of(ty)
        xs, ys = fr_list(rng, m), fr_list(rng, n)
        a = [fr_list(rng, n) for _ in range(E)]
        b = [fr_list(rng, m) for _ in range(E)]
        gam = [[fr_list(rng, n) for _ in range(m)] for _ in range(E)]
        flat = lambda rows: [x for r in rows for x in r]
        self.xs, self.ys, self.a, self.b, self.gam = xs, ys, a, b, gam
        self.X, self.Y = _enc_side1(crs, ty, xs), _enc_side2(crs, ty, ys)
        self.A, self.B = _enc_side1(crs, ty, flat(a)), _enc_side2(crs, ty, flat(b))     # [E][n], [E][m]
        self.G = b"".join(frmat_b(g) for g in gam)
        vals = [_value(a[e], b[e], gam[e], xs, ys) for e in range(E)]
        if ty == 0:
            self.T = b"".join(fp12_b(crs.gt_gen.pow(v)) for v in vals)
        elif ty == 1:
            self.T = b"".join(g1_multiples(crs, vals))
        elif ty == 2:
            self.T = b"".join(g2_multiples(crs, vals))
        else:
            self.T = frs_b(vals)
        self.xr, self.yr = frs_b(fr_list(rng, m * cx)), frs_b(fr_list(rng, n * cy))
        self.Tr = frs_b(fr_list(rng, E * cx * cy))
        if prove:
            self.xc = cb.commit_x(ty, self.X, self.xr, self.crsb, NT)
            self.yc = cb.commit_y(ty, self.Y, self.yr, self.crsb, NT)
            self.pi, self.theta = cb.prove_batch(ty, E, m, n, self.A, self.B, self.G, self.X, self.Y, self.xr, self.yr,
                                                 self.Tr, True, self.crsb, NT)

    def verify_arrays(self):
        """gs_verify_batch layout: the shared commitments repeated per equation."""
        return [self.A, self.B, self.G, self.T, self.xc * self.E, self.yc * self.E, self.pi, self.theta]
