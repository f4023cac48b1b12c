"""Host-side mirror of the reference's Rust API for the hot path (same names, argument
meaning and error behaviour), over the C ABI.  Every arithmetic step runs on the GPU.

Reference surface mirrored (paths relative to /root/reference):
  generator.rs:25-42     AbstractCrs::generate_crs, CRS{u, v, g1_gen, g2_gen, gt_gen}
  prover/commit.rs       Commit1/Commit2 (+append), commit_G1, batch_commit_G1, commit_scalar_to_B1,
                         batch_commit_scalar_to_B1 and the four G2/B2 mirrors
  prover/prove.rs        Provable::{commit_and_prove, prove}, EquProof, CProof
  statement.rs           EquType, PPE, MSMEG1, MSMEG2, QuadEqu
  verifier.rs            Verifiable::verify
  data_structures.rs     ComT::{pairing, pairing_sum, linear_map_*}, Mat::{left_mul, right_mul, ...}

Elements are `bytes` in the C-ABI encoding (arkworks Montgomery limbs; see include/gs_b200.h):
Fr 32 B, G1 96 B, G2 192 B, GT 576 B; Com1 = (G1, G1) and Com2 = (G2, G2) are 192 / 384 B
strings; a Matrix<Fr> is a list of rows of Fr.  `rng` is any object with a method
``fr() -> bytes`` (and ``g1()``, ``g2()`` for generate_crs); draws happen on the host in the
reference's order, which makes every output reproducible bit-for-bit.
The reference signals misuse by assert!/panic; here those are AssertionError / GsError.
"""
from dataclasses import dataclass, field
from typing import List, Tuple

from . import ffi
from .ffi import Engine, GsError

FR, G1, G2, GT = ffi.FR, ffi.G1, ffi.G2, ffi.GT
G1_ZERO, G2_ZERO = bytes(G1), bytes(G2)


class EquType:  # statement.rs:42-50, serialised as one byte :68-73
    PairingProduct, MultiScalarG1, MultiScalarG2, Quadratic = 0, 1, 2, 3


_default_engine = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(0)
    return _default_engine


def _split(b, size):
    return [b[i:i + size] for i in range(0, len(b), size)]


def _flat(m):
    return b"".join(x for row in m for x in row)


# ---------------------------------------------------------------- CRS  (generator.rs)
@dataclass
class ExtractionKey:
    """The trapdoor of a binding CRS: a1, a2 of generate_crs (Fr bytes), with u[0] = (p1, a1 p1), v[0] = (p2, a2 p2).
    Whoever holds it opens every commitment made under that CRS (extract_G1 and the other extract functions)."""
    a1: bytes
    a2: bytes

    def to_bytes(self) -> bytes:
        return self.a1 + self.a2

    @staticmethod
    def from_bytes(b: bytes) -> "ExtractionKey":
        if len(b) != 2 * FR:
            raise ValueError(f"ExtractionKey: {len(b)} bytes, expected {2 * FR}")
        return ExtractionKey(b[:FR], b[FR:])


@dataclass
class CRS:
    u: List[bytes]       # 2 x Com1
    v: List[bytes]       # 2 x Com2
    g1_gen: bytes
    g2_gen: bytes
    gt_gen: bytes
    engine: Engine = field(default=None, repr=False, compare=False)

    @staticmethod
    def generate_crs(rng, engine: Engine = None) -> "CRS":
        """generator.rs:81-118; RNG order p1 <- G1, p2 <- G2, a1, a2, t1, t2 <- Fr (:86-93)."""
        return CRS.generate_crs_with_trapdoor(rng, engine)[0]

    @staticmethod
    def generate_crs_with_trapdoor(rng, engine: Engine = None) -> "Tuple[CRS, ExtractionKey]":
        """generate_crs that also returns the binding key's trapdoor (a1, a2) instead of dropping it (not in the reference;
        ExtGen of Groth & Sahai, EUROCRYPT 2008).  Exactly generate_crs's draws: the same rng state gives the same CRS."""
        eng = engine or default_engine()
        p1, p2 = rng.g1(), rng.g2()
        a1, a2, t1, t2 = rng.fr(), rng.fr(), rng.fr(), rng.fr()
        return CRS.from_bytes(eng.crs_generate(p1, p2, a1, a2, t1, t2), eng, loaded=True), ExtractionKey(a1, a2)

    @staticmethod
    def generate_hiding_crs(rng, engine: Engine = None) -> "CRS":
        """The simulated (perfectly hiding) key of generator.rs:62-77 -- dead code upstream (`#[allow(dead_code)]`),
        offered here because it is what a zero-knowledge simulator needs (SURVEY.md §8f.4).  Same RNG draws as
        generate_crs; the only difference is the last entry of each key: u[1].1 = t1*q1 - g1, v[1].1 = t2*q2 - g2,
        i.e. u[1] - iota_1(g1) and v[1] - iota_2(g2) on the device (gs_com1_sub / gs_com2_sub)."""
        crs = CRS.generate_crs(rng, engine)
        u1 = Com1.sub(crs.u[1], Com1.linear_map(crs.g1_gen), crs.engine)
        v1 = Com2.sub(crs.v[1], Com2.linear_map(crs.g2_gen), crs.engine)
        return CRS.from_bytes(crs.u[0] + u1 + crs.v[0] + v1 + crs.g1_gen + crs.g2_gen + crs.gt_gen, crs.engine)

    def to_bytes(self) -> bytes:
        return b"".join(self.u) + b"".join(self.v) + self.g1_gen + self.g2_gen + self.gt_gen

    @staticmethod
    def from_bytes(b: bytes, engine: Engine = None, loaded=False) -> "CRS":
        eng = engine or default_engine()
        o = 0
        u = [b[0:192], b[192:384]]
        v = [b[384:768], b[768:1152]]
        o = 1152
        crs = CRS(u, v, b[o:o + G1], b[o + G1:o + G1 + G2], b[o + G1 + G2:o + G1 + G2 + GT], eng)
        if not loaded:
            eng.crs_load(b)
        eng._loaded_crs = b
        return crs

    def _use(self) -> Engine:
        """Make this key the engine's current one (any `&CRS` argument of the reference)."""
        b = self.to_bytes()
        if getattr(self.engine, "_loaded_crs", None) != b:
            self.engine.crs_load(b)
            self.engine._loaded_crs = b
        return self.engine


# ---------------------------------------------------------------- commitments  (prover/commit.rs)
@dataclass
class _Commit:
    coms: List[bytes]
    rand: List[List[bytes]]   # Matrix<Fr>

    def append(self, other):   # Commit::append :42-51
        self.coms.extend(other.coms)
        self.rand.extend(other.rand)


class Commit1(_Commit):
    pass


class Commit2(_Commit):
    pass


def batch_commit_G1(xvars, key: CRS, rng) -> Commit1:            # :78-100
    rand = [[rng.fr(), rng.fr()] for _ in xvars]                 # row-major draws :85-88
    out = key._use().batch_commit_g1(b"".join(xvars), _flat(rand))
    return Commit1(_split(out, 192), rand)


def batch_commit_G2(yvars, key: CRS, rng) -> Commit2:            # :178-200
    rand = [[rng.fr(), rng.fr()] for _ in yvars]
    out = key._use().batch_commit_g2(b"".join(yvars), _flat(rand))
    return Commit2(_split(out, 384), rand)


def batch_commit_scalar_to_B1(scalar_xvars, key: CRS, rng) -> Commit1:   # :125-156
    rand = [[rng.fr()] for _ in scalar_xvars]
    out = key._use().batch_commit_scalar_b1(b"".join(scalar_xvars), _flat(rand))
    return Commit1(_split(out, 192), rand)


def batch_commit_scalar_to_B2(scalar_yvars, key: CRS, rng) -> Commit2:   # :225-256
    rand = [[rng.fr()] for _ in scalar_yvars]
    out = key._use().batch_commit_scalar_b2(b"".join(scalar_yvars), _flat(rand))
    return Commit2(_split(out, 384), rand)


def commit_G1(xvar, key, rng): return batch_commit_G1([xvar], key, rng)                       # :59-75
def commit_G2(yvar, key, rng): return batch_commit_G2([yvar], key, rng)                       # :159-175
def commit_scalar_to_B1(x, key, rng): return batch_commit_scalar_to_B1([x], key, rng)         # :103-122
def commit_scalar_to_B2(y, key, rng): return batch_commit_scalar_to_B2([y], key, rng)         # :203-222


# ---------------------------------------------------------------- proofs  (prover/prove.rs)
@dataclass
class EquProof:               # :55-61
    pi: List[bytes]
    theta: List[bytes]
    equ_type: int
    rand: List[List[bytes]]


@dataclass
class CProof:                 # :64-69
    xcoms: Commit1
    ycoms: Commit2
    equ_proofs: List[EquProof]


@dataclass
class _Equation:
    a_consts: List[bytes]
    b_consts: List[bytes]
    gamma: List[List[bytes]]
    target: bytes
    equ_type = None

    def get_type(self): return self.equ_type

    def _cx(self): return 2 if self.equ_type in (0, 1) else 1
    def _cy(self): return 2 if self.equ_type in (0, 2) else 1

    def prove(self, xvars, yvars, xcoms, ycoms, crs: CRS, rng) -> EquProof:
        # the reference's dimension asserts (prove.rs:106-114 and mirrors)
        assert len(xvars) == len(xcoms.rand) and len(self.gamma) == len(xcoms.rand)
        assert len(xcoms.rand[0]) == self._cx()
        assert len(yvars) == len(ycoms.rand) and len(self.gamma[0]) == len(ycoms.rand)
        assert len(ycoms.rand[0]) == self._cy()
        m, n = len(xvars), len(yvars)
        cx, cy = self._cx(), self._cy()
        pf_rand = [[rng.fr() for _ in range(cx)] for _ in range(cy)]    # T, row-major (:123-126 etc.)
        pi, theta = crs._use().prove(self.equ_type, m, n, b"".join(self.a_consts), b"".join(self.b_consts),
                                     _flat(self.gamma), b"".join(xvars), b"".join(yvars),
                                     _flat(xcoms.rand), _flat(ycoms.rand), _flat(pf_rand))
        return EquProof(_split(pi, 384), _split(theta, 192), self.equ_type, pf_rand)

    def commit_and_prove(self, xvars, yvars, crs: CRS, rng) -> CProof:
        # RNG order: x commitments, y commitments, then T (prove.rs:82-88)
        xc = (batch_commit_G1 if self.equ_type in (0, 1) else batch_commit_scalar_to_B1)(xvars, crs, rng)
        yc = (batch_commit_G2 if self.equ_type in (0, 2) else batch_commit_scalar_to_B2)(yvars, crs, rng)
        return CProof(xc, yc, [self.prove(xvars, yvars, xc, yc, crs, rng)])

    def rerandomize(self, com_proof: CProof, crs: CRS, rng) -> CProof:
        """A fresh-looking CProof of the same statement from `com_proof` alone, without the witnesses or the old randomness
        (not in the reference; see rerandomize_batch).  RNG order: R' rows, S' rows, then T', row-major."""
        return rerandomize_batch([self], [com_proof], crs, rng)[0]

    def verify(self, com_proof: CProof, crs: CRS) -> bool:              # verifier.rs:23-157
        assert len(com_proof.equ_proofs) == 1
        ep = com_proof.equ_proofs[0]
        assert self.get_type() == ep.equ_type
        m, n = len(com_proof.xcoms.coms), len(com_proof.ycoms.coms)
        # pairing_sum's assert_eq!(x_vec.len(), y_vec.len()) (data_structures.rs:495) and left_mul's (:705)
        assert len(self.a_consts) == n and len(self.b_consts) == m
        assert len(self.gamma) == m and all(len(r) == n for r in self.gamma)
        return crs._use().verify(self.equ_type, m, n, b"".join(self.a_consts), b"".join(self.b_consts),
                                 _flat(self.gamma), self.target, b"".join(com_proof.xcoms.coms),
                                 b"".join(com_proof.ycoms.coms), b"".join(ep.pi), b"".join(ep.theta))


class PPE(_Equation):
    equ_type = EquType.PairingProduct


class MSMEG1(_Equation):
    equ_type = EquType.MultiScalarG1


class MSMEG2(_Equation):
    equ_type = EquType.MultiScalarG2


class QuadEqu(_Equation):
    equ_type = EquType.Quadratic


def prove_batch(equations, xvars, yvars, xcoms, ycoms, crs: CRS, rng) -> List[EquProof]:
    """Provable::prove for many equations of one type over the SAME committed variables (a multi-equation
    statement, statement.rs:109) in one GPU pass.  T is drawn equation by equation in the reference's order."""
    assert equations
    e0 = equations[0]
    ty, cx, cy = e0.equ_type, e0._cx(), e0._cy()
    m, n = len(xvars), len(yvars)
    for e in equations:
        assert e.equ_type == ty and len(e.gamma) == m and len(e.gamma[0]) == n
    assert len(xcoms.rand) == m and len(ycoms.rand) == n and len(xcoms.rand[0]) == cx and len(ycoms.rand[0]) == cy
    rands = [[[rng.fr() for _ in range(cx)] for _ in range(cy)] for _ in equations]
    pi, th = crs._use().prove_batch(ty, len(equations), m, n, b"".join(b"".join(e.a_consts) for e in equations),
                                    b"".join(b"".join(e.b_consts) for e in equations), b"".join(_flat(e.gamma) for e in equations),
                                    b"".join(xvars), b"".join(yvars), _flat(xcoms.rand), _flat(ycoms.rand),
                                    b"".join(_flat(r) for r in rands), shared_vars=True)
    ps, ts = _split(pi, 384 * cx), _split(th, 192 * cy)
    return [EquProof(_split(p, 384), _split(t, 192), ty, r) for p, t, r in zip(ps, ts, rands)]


def rerandomize_batch(equations, proofs, crs: CRS, rng, shared_commitments: bool = False) -> List[CProof]:
    """Rerandomisation of committed proofs (Belenkiy et al., CRYPTO 2009; not in the reference): every (equation, CProof)
    pair becomes a CProof of the same statement that is distributed exactly as a fresh commit_and_prove, computed from the
    proof alone in one GPU pass (gs_rerandomize_batch).  One type and one shape per batch.

    Fresh randomness is drawn per proof in commit_and_prove's order: R' (m x cx) rows, then S' (n x cy) rows, then T'
    (cy x cx), row-major.  With shared_commitments every CProof must hold the same commitments (a multi-equation statement
    over one set of variables): R' and S' are drawn once, then T' equation by equation, and the returned CProofs share the
    new commitments.  The openings are not known to the rerandomiser, so the returned Commit*.rand and EquProof.rand are
    empty matrices."""
    assert len(equations) == len(proofs) and equations
    ty = equations[0].equ_type
    m, n = len(proofs[0].xcoms.coms), len(proofs[0].ycoms.coms)
    for e, p in zip(equations, proofs):
        if e.equ_type != ty or len(p.xcoms.coms) != m or len(p.ycoms.coms) != n:
            raise ValueError("rerandomize_batch: every (equation, proof) must have the same type and shape")
        if len(p.equ_proofs) != 1 or p.equ_proofs[0].equ_type != ty:
            raise ValueError("rerandomize_batch: exactly one EquProof of the equation's type per CProof")
        if len(e.a_consts) != n or len(e.b_consts) != m or len(e.gamma) != m or any(len(r) != n for r in e.gamma):
            raise ValueError("rerandomize_batch: constants / Gamma do not match the number of variables")
        if shared_commitments and (p.xcoms.coms != proofs[0].xcoms.coms or p.ycoms.coms != proofs[0].ycoms.coms):
            raise ValueError("rerandomize_batch: shared_commitments needs the same commitments in every CProof")
    cx, cy = equations[0]._cx(), equations[0]._cy()
    draw = lambda rows, cols: [[rng.fr() for _ in range(cols)] for _ in range(rows)]
    if shared_commitments:
        R, S = draw(m, cx), draw(n, cy)
        Rs, Ss, Ts = [R], [S], [draw(cy, cx) for _ in equations]
    else:
        Rs, Ss, Ts = [], [], []
        for _ in equations:
            Rs.append(draw(m, cx))
            Ss.append(draw(n, cy))
            Ts.append(draw(cy, cx))
    coms = proofs[:1] if shared_commitments else proofs
    cat = lambda f, items: b"".join(f(x) for x in items)
    xc, yc, pi, th = crs._use().rerandomize_batch(
        ty, len(equations), m, n, cat(lambda e: b"".join(e.a_consts), equations), cat(lambda e: b"".join(e.b_consts), equations),
        cat(lambda e: _flat(e.gamma), equations), cat(lambda p: b"".join(p.xcoms.coms), coms),
        cat(lambda p: b"".join(p.ycoms.coms), coms), cat(lambda p: b"".join(p.equ_proofs[0].pi), proofs),
        cat(lambda p: b"".join(p.equ_proofs[0].theta), proofs), cat(_flat, Rs), cat(_flat, Ss), cat(_flat, Ts),
        shared_coms=shared_commitments)
    xcs, ycs = _split(xc, 192 * m), _split(yc, 384 * n)
    pis, ths = _split(pi, 384 * cx), _split(th, 192 * cy)
    out = []
    for k in range(len(equations)):
        j = 0 if shared_commitments else k
        out.append(CProof(Commit1(_split(xcs[j], 192), []), Commit2(_split(ycs[j], 384), []),
                          [EquProof(_split(pis[k], 384), _split(ths[k], 192), ty, [])]))
    return out


# ---------------------------------------------------------------- extraction with the binding key (not in the reference)
# X = c.1 - a1 c.0 for a commitment under a binding CRS (u[0] = (p1, a1 p1), u[1] = t1 u[0]); scalar commitments give x p1
# (x itself cannot be recovered), the G2 side likewise with a2 (gs_extract).  The key is checked against the engine's
# current CRS -- `crs` when given, else the one loaded last -- and a mismatch raises GsError; a hiding CRS has no key.
def _coms_of(coms): return coms.coms if isinstance(coms, _Commit) else list(coms)


def _extract_engine(crs): return crs._use() if crs is not None else default_engine()


def extract_G1(coms, key: ExtractionKey, crs: CRS = None) -> List[bytes]:
    """The committed G1 values of a Commit1 (batch_commit_G1) or of a list of Com1."""
    return _split(_extract_engine(crs).extract(b"".join(_coms_of(coms)), key.a1)[0], G1)


def extract_G2(coms, key: ExtractionKey, crs: CRS = None) -> List[bytes]:
    """The committed G2 values of a Commit2 (batch_commit_G2) or of a list of Com2."""
    return _split(_extract_engine(crs).extract(ycoms=b"".join(_coms_of(coms)), ykey=key.a2)[1], G2)


def extract_scalar_B1(coms, key: ExtractionKey, crs: CRS = None) -> List[bytes]:
    """x * g1 for every commitment of a scalar x (batch_commit_scalar_to_B1)."""
    return extract_G1(coms, key, crs)


def extract_scalar_B2(coms, key: ExtractionKey, crs: CRS = None) -> List[bytes]:
    """y * g2 for every commitment of a scalar y (batch_commit_scalar_to_B2)."""
    return extract_G2(coms, key, crs)


def extract(com_proof: CProof, equ_type: int, key: ExtractionKey, crs: CRS = None) -> Tuple[List[bytes], List[bytes]]:
    """Both sides of a CProof in one GPU call: (x values, y values).  Group-typed sides (x of PPE / MSMEG1, y of PPE /
    MSMEG2) give the witnesses themselves; scalar-typed sides give x * g1 / y * g2."""
    if equ_type not in (0, 1, 2, 3):
        raise ValueError(f"extract: bad equation type {equ_type}")
    xs, ys = _extract_engine(crs).extract(b"".join(com_proof.xcoms.coms), key.a1, b"".join(com_proof.ycoms.coms), key.a2)
    return _split(xs, G1), _split(ys, G2)


def verify_batch(equations, proofs, crs: CRS, randomized: bool = False, rho: bytes = None) -> List[bool]:
    """Many independent (equation, CProof) pairs of one type and shape in one GPU pass.

    randomized=True (opt-in, SURVEY.md 8f.4; not in the reference): first ONE randomised check of the whole batch
    (gs_verify_batch_rand: a single folded pairing product, one final exponentiation); if it accepts, every proof is
    reported valid (error <= 2^-62 over `rho`, drawn from the OS CSPRNG when not given); if it rejects, the exact
    per-proof verification below runs and says which proofs failed.  Inputs must be group members (deserialised values
    are), PPE targets members of GT."""
    ty, m, n, arrays = _batch_arrays(equations, proofs, "verify_batch")
    if randomized and crs._use().verify_batch_rand(ty, len(equations), m, n, *arrays, rho=rho):
        return [True] * len(equations)
    ok = crs._use().verify_batch(ty, len(equations), m, n, *arrays)
    return [b == 1 for b in ok]


def _batch_arrays(equations, proofs, name):
    """(type, m, n, the eight C-ABI arrays) of a batch of one type and shape; ValueError names `name`."""
    assert len(equations) == len(proofs) and equations
    ty = equations[0].equ_type
    m, n = len(proofs[0].xcoms.coms), len(proofs[0].ycoms.coms)
    for e, p in zip(equations, proofs):     # one type and one shape per batch: a mixed batch would be mis-sliced silently
        if e.equ_type != ty or len(p.xcoms.coms) != m or len(p.ycoms.coms) != n:
            raise ValueError(f"{name}: every (equation, proof) must have the same type and shape")
        if len(p.equ_proofs) != 1 or p.equ_proofs[0].equ_type != ty:      # verifier.rs:25-26
            raise ValueError(f"{name}: exactly one EquProof of the equation's type per CProof")
        if len(e.a_consts) != n or len(e.b_consts) != m or len(e.gamma) != m or any(len(r) != n for r in e.gamma):
            raise ValueError(f"{name}: constants / Gamma do not match the number of variables")
    cat = lambda f: b"".join(f(e, p) for e, p in zip(equations, proofs))
    arrays = (cat(lambda e, p: b"".join(e.a_consts)), cat(lambda e, p: b"".join(e.b_consts)),
              cat(lambda e, p: _flat(e.gamma)), cat(lambda e, p: e.target), cat(lambda e, p: b"".join(p.xcoms.coms)),
              cat(lambda e, p: b"".join(p.ycoms.coms)), cat(lambda e, p: b"".join(p.equ_proofs[0].pi)),
              cat(lambda e, p: b"".join(p.equ_proofs[0].theta)))
    return ty, m, n, arrays


def verify_each_randomized(equations, proofs, crs: CRS, rho: bytes = None) -> List[bool]:
    """Per-proof verdicts of a batch of one type and shape at close to the randomised cost (opt-in, not in the reference):
    each proof's four ComT entries are folded with its own random weights into one pairing product and ONE final
    exponentiation (gs_verify_each_rand).  A bad proof is accepted with probability <= 2^-62 over `rho` (2*count + 1
    64-bit words, drawn from the OS CSPRNG when not given), each proof on its own, so a batch with some bad proofs still
    costs one randomised pass.  Inputs must be group members (deserialised values are), PPE targets members of GT."""
    ty, m, n, arrays = _batch_arrays(equations, proofs, "verify_each_randomized")
    ok = crs._use().verify_each_rand(ty, len(equations), m, n, *arrays, rho=rho)
    return [b == 1 for b in ok]


# ---------------------------------------------------------------- vector <-> matrix helpers (data_structures.rs:143-160)
def col_vec_to_vec(mat):
    """Collapse a 1 x n row or an n x 1 column into a list (:145-151)."""
    return list(mat[0]) if len(mat) == 1 else [row[0] for row in mat]


def vec_to_col_vec(vec):
    """Expand a list into an n x 1 column matrix (:154-160)."""
    return [[e] for e in vec]


# ---------------------------------------------------------------- Com1 / Com2 / ComT  (data_structures.rs)
class _ComGroup:
    """Add / Sub / Neg / Sum / Zero of a commitment group (impl_base_commit_groups! :162-255, ComT :391-479).
    Elements are C-ABI byte strings; lists are processed in one GPU pass."""
    kind = None
    size = 0

    @classmethod
    def _eng(cls, engine): return engine or default_engine()
    @classmethod
    def add(cls, a, b, engine=None): return cls._eng(engine).elementwise(cls.kind, "add", a, b)
    @classmethod
    def sub(cls, a, b, engine=None): return cls._eng(engine).elementwise(cls.kind, "sub", a, b)
    @classmethod
    def neg(cls, a, engine=None): return cls._eng(engine).elementwise(cls.kind, "neg", a)
    @classmethod
    def sum(cls, elems, engine=None): return cls._eng(engine).group_sum(cls.kind, b"".join(elems))

    @classmethod
    def batch_add(cls, xs, ys, engine=None):
        assert len(xs) == len(ys)
        return _split(cls._eng(engine).elementwise(cls.kind, "add", b"".join(xs), b"".join(ys)), cls.size)


class Com1(_ComGroup):
    kind, size = "com1", 192
    @staticmethod
    def zero(): return bytes(192)                                           # :257-266
    @staticmethod
    def as_col_vec(c): return [[c[:G1]], [c[G1:]]]                          # :301-303
    @staticmethod
    def as_vec(c): return [c[:G1], c[G1:]]                                  # :305-307
    @staticmethod
    def from_matrix(mat):                                                   # From<Matrix<G1Affine>> :283-290
        assert len(mat) == 2 and len(mat[0]) == 1 and len(mat[1]) == 1
        return mat[0][0] + mat[1][0]
    @staticmethod
    def linear_map(x): return G1_ZERO + x                                   # :310-312
    @staticmethod
    def batch_linear_map(xs): return [G1_ZERO + x for x in xs]
    @staticmethod
    def scalar_linear_map(x, key: CRS):                                     # :323-326  x * (u2 + (O, g1))
        return batch_commit_scalar_b1_norand(key, [x])[0]
    @staticmethod
    def batch_scalar_linear_map(xs, key: CRS): return batch_commit_scalar_b1_norand(key, xs)   # :328-334
    @staticmethod
    def scalar_mul(c, s, engine=None):                                      # :336-342
        return (engine or default_engine()).com1_matmul(1, 1, 1, s, c)


class Com2(_ComGroup):
    kind, size = "com2", 384
    @staticmethod
    def zero(): return bytes(384)                                           # :268-277
    @staticmethod
    def as_col_vec(c): return [[c[:G2]], [c[G2:]]]                          # :346-348
    @staticmethod
    def as_vec(c): return [c[:G2], c[G2:]]                                  # :350-352
    @staticmethod
    def from_matrix(mat):                                                   # From<Matrix<G2Affine>> :291-298
        assert len(mat) == 2 and len(mat[0]) == 1 and len(mat[1]) == 1
        return mat[0][0] + mat[1][0]
    @staticmethod
    def linear_map(y): return G2_ZERO + y                                   # :355-357
    @staticmethod
    def batch_linear_map(ys): return [G2_ZERO + y for y in ys]
    @staticmethod
    def scalar_linear_map(y, key: CRS):                                     # :368-371  y * (v2 + (O, g2))
        return batch_commit_scalar_b2_norand(key, [y])[0]
    @staticmethod
    def batch_scalar_linear_map(ys, key: CRS): return batch_commit_scalar_b2_norand(key, ys)   # :373-379
    @staticmethod
    def scalar_mul(c, s, engine=None):                                      # :381-387
        return (engine or default_engine()).com2_matmul(1, 1, 1, s, c)


def batch_commit_scalar_b1_norand(key: CRS, xs):
    """iota_1'(x) = x W1: a scalar commitment with zero randomness."""
    out = key._use().batch_commit_scalar_b1(b"".join(xs), bytes(FR * len(xs)))
    return _split(out, 192)


def batch_commit_scalar_b2_norand(key: CRS, ys):
    """iota_2'(y) = y W2: a scalar commitment with zero randomness."""
    out = key._use().batch_commit_scalar_b2(b"".join(ys), bytes(FR * len(ys)))
    return _split(out, 384)


class ComT(_ComGroup):
    kind, size = "comt", 2304
    @staticmethod
    def zero(engine=None): return (engine or default_engine()).group_sum("comt", b"")   # four GT identities :412-421
    @staticmethod
    def as_matrix(c): return [[c[0:576], c[576:1152]], [c[1152:1728], c[1728:2304]]]     # :1361-1377 row-major
    @staticmethod
    def from_matrix(mat):                                                   # From<Matrix<PairingOutput>> :467-474
        assert len(mat) == 2 and len(mat[0]) == 2 and len(mat[1]) == 2
        return mat[0][0] + mat[0][1] + mat[1][0] + mat[1][1]
    @staticmethod
    def pairing(x, y, engine=None):                                         # :484-491
        return (engine or default_engine()).comt_pairing(x, y)
    @staticmethod
    def pairing_sum(xs, ys, engine=None):                                   # :494-502
        if len(xs) != len(ys):
            raise AssertionError("pairing_sum: x_vec.len() != y_vec.len()")
        return (engine or default_engine()).comt_pairing_sum(b"".join(xs), b"".join(ys))
    @staticmethod
    def linear_map_PPE(z, key: CRS): return key._use().comt_linear_map(0, z)       # :509-516
    @staticmethod
    def linear_map_MSMEG1(z, key: CRS): return key._use().comt_linear_map(1, z)    # :519-524
    @staticmethod
    def linear_map_MSMEG2(z, key: CRS): return key._use().comt_linear_map(2, z)    # :527-532
    @staticmethod
    def linear_map_quad(z, key: CRS): return key._use().comt_linear_map(3, z)      # :535-540


# ---------------------------------------------------------------- Mat  (data_structures.rs:545-913)
def _dims(mat): return len(mat), (len(mat[0]) if mat else 0)


def _unflat(b, rows, cols, size):
    return [_split(b[i * cols * size:(i + 1) * cols * size], size) for i in range(rows)]


def mat_transpose(mat):
    """Mat::transpose (:630-643, :809-822): pure data movement, no arithmetic."""
    r, c = _dims(mat)
    return [[mat[i][j] for i in range(r)] for j in range(c)]


def fr_right_mul(a, rhs, engine=None):
    """Matrix<Fr>::right_mul :824-868 (self * rhs)."""
    (r, k), (k2, c) = _dims(a), _dims(rhs)
    if r == 0 or k == 0 or k2 == 0 or c == 0:
        return []
    assert k == k2
    out = (engine or default_engine()).fr_matmul(r, k, c, _flat(a), _flat(rhs))
    return _unflat(out, r, c, FR)


def fr_left_mul(a, lhs, engine=None):
    """Matrix<Fr>::left_mul :870-912 (lhs * self)."""
    return fr_right_mul(lhs, a, engine)


def fr_add(a, b, engine=None):
    """Matrix<Fr>::add :771-785 (asserts equal dimensions)."""
    assert _dims(a) == _dims(b)
    r, c = _dims(a)
    return _unflat((engine or default_engine()).elementwise("fr", "add", _flat(a), _flat(b)), r, c, FR)


def fr_neg(a, engine=None):
    """Matrix<Fr>::neg :787-794."""
    r, c = _dims(a)
    return _unflat((engine or default_engine()).elementwise("fr", "neg", _flat(a)), r, c, FR)


def fr_scalar_mul(a, s, engine=None):
    """Matrix<Fr>::scalar_mul :796-807."""
    r, c = _dims(a)
    return _unflat((engine or default_engine()).fr_scale(s, _flat(a)), r, c, FR)


def _com(which): return ("com1", 192) if which == 1 else ("com2", 384)


def com_add(a, b, which, engine=None):
    """Matrix<Com1|Com2>::add :590-603."""
    assert _dims(a) == _dims(b)
    kind, size = _com(which)
    r, c = _dims(a)
    return _unflat((engine or default_engine()).elementwise(kind, "add", _flat(a), _flat(b)), r, c, size)


def com_neg(a, which, engine=None):
    """Matrix<Com1|Com2>::neg :606-615."""
    kind, size = _com(which)
    r, c = _dims(a)
    return _unflat((engine or default_engine()).elementwise(kind, "neg", _flat(a)), r, c, size)


def com_scalar_mul(a, s, which, engine=None):
    """Matrix<Com1|Com2>::scalar_mul :617-628: every entry times the same scalar."""
    kind, size = _com(which)
    r, c = _dims(a)
    eng = engine or default_engine()
    fn = eng.com1_matmul if which == 1 else eng.com2_matmul
    return _unflat(fn(1, 1, r * c, s, _flat(a)), r, c, size)


def com_left_mul(mat, lhs, which, engine=None):
    """Matrix<Com1|Com2>::left_mul :696-742: out[i][j] = sum_k lhs[i][k] * mat[k][j]."""
    (r, k), (k2, c) = _dims(lhs), _dims(mat)
    if r == 0 or k == 0 or k2 == 0 or c == 0:
        return []
    assert k == k2
    eng = engine or default_engine()
    size = 192 if which == 1 else 384
    fn = eng.com1_matmul if which == 1 else eng.com2_matmul
    out = fn(r, k, c, _flat(lhs), _flat(mat))
    return _unflat(out, r, c, size)


def com_right_mul(mat, rhs, which, engine=None):
    """Matrix<Com1|Com2>::right_mul :645-694: out[i][j] = sum_k mat[i][k] * rhs[k][j]  (= (rhs^T * mat^T)^T)."""
    (r, k), (k2, c) = _dims(mat), _dims(rhs)
    if r == 0 or k == 0 or k2 == 0 or c == 0:
        return []
    assert k == k2
    return mat_transpose(com_left_mul(mat_transpose(mat), mat_transpose(rhs), which, engine))


# ---------------------------------------------------------------- canonical serialisation (ark-serialize layout)
# serialize_compressed of the reference's derived types: fields in declaration order, Vec<T> = u64-LE length then the
# items, Com1 / Com2 = two compressed points, Fr = 32 B LE, PairingOutput = 576 B LE, EquType = one byte
# (generator.rs:35-42, prover/commit.rs:18-28, prover/prove.rs:55-61, statement.rs:61-97).  The framing is host
# logic; every element conversion (compression, decompression + subgroup check, Montgomery <-> canonical) is one
# batched GPU call per element kind.
class SerializationError(ValueError):
    """ark_serialize::SerializationError::InvalidData."""


def _u64(n): return int(n).to_bytes(8, "little")


class _Reader:
    def __init__(self, b):
        self.b, self.o = b, 0

    def take(self, n):
        if self.o + n > len(self.b):
            raise SerializationError("unexpected end of input")
        out = self.b[self.o:self.o + n]
        self.o += n
        return out

    def u64(self): return int.from_bytes(self.take(8), "little")


def _ser_points(eng, kind, pts): return eng.serialize(kind, b"".join(pts)) if pts else b""


def _de(eng, kind, wire, what):
    out, ok = eng.deserialize(kind, wire)
    if ok != b"\x01" * len(ok):
        raise SerializationError(f"invalid {what} encoding at element {ok.index(0)}")
    return out


def _ser_matrix(eng, mat):
    flat = eng.serialize("fr", _flat(mat)) if mat and mat[0] else b""
    out, o = _u64(len(mat)), 0
    for row in mat:
        out += _u64(len(row)) + flat[o:o + 32 * len(row)]
        o += 32 * len(row)
    return out


def _de_matrix(eng, rd):
    rows = rd.u64()
    lens, wire = [], b""
    for _ in range(rows):
        k = rd.u64()
        lens.append(k)
        wire += rd.take(32 * k)
    vals = _split(_de(eng, "fr", wire, "Fr"), FR) if wire else []
    out, o = [], 0
    for k in lens:
        out.append(vals[o:o + k])
        o += k
    return out


def _com_points(coms, size): return [c[i * size:(i + 1) * size] for c in coms for i in range(2)]


def _ser_coms(eng, coms, which):
    kind, size = ("g1", G1) if which == 1 else ("g2", G2)
    return _u64(len(coms)) + _ser_points(eng, kind, _com_points(coms, size))


def _de_coms(eng, rd, which):
    kind, size, wsz = ("g1", G1, 48) if which == 1 else ("g2", G2, 96)
    n = rd.u64()
    pts = _de(eng, kind, rd.take(2 * n * wsz), "G1" if which == 1 else "G2") if n else b""
    return _split(pts, 2 * size)


def serialize_crs(crs: CRS) -> bytes:
    """CRS::serialize_compressed: 1,312 bytes (SURVEY.md §8a a11)."""
    eng = crs.engine or default_engine()
    return (_ser_coms(eng, crs.u, 1) + _ser_coms(eng, crs.v, 2) + eng.serialize("g1", crs.g1_gen) +
            eng.serialize("g2", crs.g2_gen) + eng.serialize("gt", crs.gt_gen))


def deserialize_crs(b: bytes, engine: Engine = None) -> CRS:
    eng = engine or default_engine()
    rd = _Reader(b)
    u, v = _de_coms(eng, rd, 1), _de_coms(eng, rd, 2)
    g1 = _de(eng, "g1", rd.take(48), "G1")
    g2 = _de(eng, "g2", rd.take(96), "G2")
    gt = _de(eng, "gt", rd.take(576), "GT")
    if len(u) != 2 or len(v) != 2:
        raise SerializationError("CRS keys must hold two commitments each")
    return CRS.from_bytes(b"".join(u) + b"".join(v) + g1 + g2 + gt, eng)


def serialize_commit(c: _Commit, engine: Engine = None) -> bytes:
    eng = engine or default_engine()
    return _ser_coms(eng, c.coms, 1 if isinstance(c, Commit1) else 2) + _ser_matrix(eng, c.rand)


def deserialize_commit(b: bytes, which: int, engine: Engine = None):
    eng = engine or default_engine()
    rd = _Reader(b)
    coms = _de_coms(eng, rd, which)
    return (Commit1 if which == 1 else Commit2)(coms, _de_matrix(eng, rd))


def serialize_equ_proof(p: EquProof, engine: Engine = None) -> bytes:
    eng = engine or default_engine()
    return _ser_coms(eng, p.pi, 2) + _ser_coms(eng, p.theta, 1) + bytes([p.equ_type]) + _ser_matrix(eng, p.rand)


def deserialize_equ_proof(b: bytes, engine: Engine = None) -> EquProof:
    eng = engine or default_engine()
    rd = _Reader(b)
    pi, theta = _de_coms(eng, rd, 2), _de_coms(eng, rd, 1)
    ty = rd.take(1)[0]
    if ty > 3:
        raise SerializationError("bad EquType byte")       # statement.rs:88-95
    return EquProof(pi, theta, ty, _de_matrix(eng, rd))


# equations (statement.rs:117-185): a_consts, b_consts, gamma, target in declaration order; constants and targets are
# G1 / G2 / Fr / PairingOutput depending on the equation type (the type itself is NOT on the wire: the caller
# names the struct it deserialises, as in Rust).
_A_KIND = {0: "g1", 1: "g1", 2: "fr", 3: "fr"}
_B_KIND = {0: "g2", 1: "fr", 2: "g2", 3: "fr"}
_T_KIND = {0: "gt", 1: "g1", 2: "g2", 3: "fr"}
_WIRE = {"g1": 48, "g2": 96, "fr": 32, "gt": 576}
_MEM = {"g1": G1, "g2": G2, "fr": FR, "gt": GT}


def _ser_vec(eng, kind, items):
    return _u64(len(items)) + (eng.serialize(kind, b"".join(items)) if items else b"")


def _de_vec(eng, rd, kind):
    n = rd.u64()
    return _split(_de(eng, kind, rd.take(n * _WIRE[kind]), kind), _MEM[kind]) if n else []


def serialize_equation(e: _Equation, engine: Engine = None) -> bytes:
    """PPE / MSMEG1 / MSMEG2 / QuadEqu ::serialize_compressed (statement.rs:117-185)."""
    eng, ty = engine or default_engine(), e.equ_type
    return (_ser_vec(eng, _A_KIND[ty], e.a_consts) + _ser_vec(eng, _B_KIND[ty], e.b_consts) +
            _ser_matrix(eng, e.gamma) + eng.serialize(_T_KIND[ty], e.target))


def deserialize_equation(b: bytes, equ_type: int, engine: Engine = None) -> _Equation:
    eng = engine or default_engine()
    rd = _Reader(b)
    a, bc = _de_vec(eng, rd, _A_KIND[equ_type]), _de_vec(eng, rd, _B_KIND[equ_type])
    gamma = _de_matrix(eng, rd)
    t = _de(eng, _T_KIND[equ_type], rd.take(_WIRE[_T_KIND[equ_type]]), "target")
    return (PPE, MSMEG1, MSMEG2, QuadEqu)[equ_type](a, bc, gamma, t)
