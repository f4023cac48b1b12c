"""ctypes binding of libgs_b200.so (include/gs_b200.h).  Bytes in, bytes out.

Element encodings are the C ABI's (= arkworks' in-memory Montgomery limbs, see the header):
Fr 32 B, G1 96 B, G2 192 B, Com1 192 B, Com2 384 B, GT 576 B, ComT 2304 B; the identity
point is all-zero bytes.  There is no CPU fallback: a missing library or GPU raises GsError.
"""
import ctypes
import os

FR, G1, G2, COM1, COM2, GT, COMT = 32, 96, 192, 192, 384, 576, 2304
CRS_BYTES = 2 * COM1 + 2 * COM2 + G1 + G2 + GT
PPE, MSMEG1, MSMEG2, QUAD = 0, 1, 2, 3

EXPORTED_SYMBOLS = [
    "gs_ctx_create", "gs_ctx_destroy", "gs_last_error", "gs_launch_count", "gs_stream",
    "gs_profile_enable", "gs_profile_read", "gs_diag_fpmul_rate",
    "gs_crs_generate", "gs_crs_load",
    "gs_batch_commit_g1", "gs_batch_commit_g2", "gs_batch_commit_scalar_b1", "gs_batch_commit_scalar_b2",
    "gs_prove", "gs_prove_batch", "gs_rerandomize", "gs_rerandomize_batch", "gs_extract", "gs_verify_batch", "gs_verify_batch_dev", "gs_verify_batch_rand", "gs_verify_batch_rand_dev",
    "gs_verify_each_rand", "gs_verify_each_rand_dev",
    "gs_verify_partial", "gs_verify_partial_dev", "gs_verify_finish", "gs_verify_finish_dev", "gs_verify_sharded",
    "gs_comt_pairing", "gs_comt_pairing_sum", "gs_comt_linear_map", "gs_pairing",
    "gs_com1_matmul", "gs_com2_matmul", "gs_fr_matmul",
    "gs_com1_add", "gs_com1_sub", "gs_com1_neg", "gs_com1_sum", "gs_com2_add", "gs_com2_sub", "gs_com2_neg", "gs_com2_sum",
    "gs_comt_add", "gs_comt_sub", "gs_comt_neg", "gs_comt_sum", "gs_fr_add", "gs_fr_sub", "gs_fr_neg", "gs_fr_scale",
    "gs_g1_compress", "gs_g1_decompress", "gs_g2_compress", "gs_g2_decompress",
    "gs_fr_to_bytes", "gs_fr_from_bytes", "gs_gt_to_bytes", "gs_gt_from_bytes",
    "gs_g1_serialize_uncompressed", "gs_g1_deserialize_uncompressed", "gs_g2_serialize_uncompressed", "gs_g2_deserialize_uncompressed",
]


# gs_allgather_fn: int (*)(void* user, const void* send_dev, void* recv_dev, size_t bytes_per_rank)
ALLGATHER_FN = ctypes.CFUNCTYPE(ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_size_t)


class GsError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"gs_b200 error {code}: {msg}")
        self.code = code


def lib_path():
    """The in-tree library; GS_B200_LIB points at an experiment build of the same sources (tools, never the tests)."""
    return os.environ.get("GS_B200_LIB") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "libgs_b200.so")


_lib = None


def load_library():
    """dlopen the in-tree library; fails loudly when it has not been built."""
    global _lib
    if _lib is None:
        path = lib_path()
        if not os.path.exists(path):
            raise GsError(-1, f"{path} not built -- run `python groth-sahai-rs_b200/build.py` (no CPU fallback exists)")
        lib = ctypes.CDLL(path)
        vp, sz, ci = ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int
        lib.gs_ctx_create.argtypes = [ci, ctypes.POINTER(vp)]
        lib.gs_ctx_destroy.argtypes = [vp]
        lib.gs_ctx_destroy.restype = None
        lib.gs_last_error.argtypes = [vp]
        lib.gs_last_error.restype = ctypes.c_char_p
        lib.gs_launch_count.argtypes = [vp]
        lib.gs_launch_count.restype = ctypes.c_uint64
        lib.gs_stream.argtypes = [vp]
        lib.gs_stream.restype = vp
        lib.gs_profile_enable.argtypes = [vp, ci]
        lib.gs_profile_read.argtypes = [vp, vp, sz]
        lib.gs_diag_fpmul_rate.argtypes = [vp, ctypes.POINTER(ctypes.c_double)]
        lib.gs_crs_generate.argtypes = [vp] * 8
        lib.gs_crs_load.argtypes = [vp, vp]
        for f in ("gs_batch_commit_g1", "gs_batch_commit_g2", "gs_batch_commit_scalar_b1", "gs_batch_commit_scalar_b2"):
            getattr(lib, f).argtypes = [vp, sz, vp, vp, vp]
        lib.gs_prove.argtypes = [vp, ci, sz, sz] + [vp] * 10
        lib.gs_prove_batch.argtypes = [vp, ci, sz, sz, sz] + [vp] * 8 + [ci, vp, vp]
        lib.gs_rerandomize.argtypes = [vp, ci, sz, sz] + [vp] * 14
        lib.gs_rerandomize_batch.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10 + [ci] + [vp] * 4
        lib.gs_extract.argtypes = [vp, sz, vp, vp, sz, vp, vp, vp, vp]
        lib.gs_verify_batch.argtypes = [vp, ci, sz, sz, sz] + [vp] * 9
        lib.gs_verify_batch_dev.argtypes = [vp, ci, sz, sz, sz] + [vp] * 9
        lib.gs_verify_batch_rand.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10
        lib.gs_verify_batch_rand_dev.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10
        lib.gs_verify_each_rand.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10
        lib.gs_verify_each_rand_dev.argtypes = [vp, ci, sz, sz, sz] + [vp] * 10
        lib.gs_verify_partial.argtypes = [vp, ci, sz, sz, sz] + [vp] * 8 + [ci, ci, vp]
        lib.gs_verify_partial_dev.argtypes = [vp, ci, sz, sz, sz] + [vp] * 8 + [ci, ci, vp]
        lib.gs_verify_finish.argtypes = [vp, ci, sz, ci, vp, vp, vp]
        lib.gs_verify_finish_dev.argtypes = [vp, ci, sz, ci, vp, vp, vp]
        lib.gs_verify_sharded.argtypes = [vp, ci, sz, sz, sz] + [vp] * 8 + [ci, ci, ALLGATHER_FN, vp, vp]
        lib.gs_comt_pairing.argtypes = [vp, sz, vp, vp, vp]
        lib.gs_comt_pairing_sum.argtypes = [vp, sz, vp, vp, vp]
        lib.gs_comt_linear_map.argtypes = [vp, ci, vp, vp]
        lib.gs_pairing.argtypes = [vp, sz, vp, vp, vp]
        for f in ("gs_com1_matmul", "gs_com2_matmul", "gs_fr_matmul"):
            getattr(lib, f).argtypes = [vp, sz, sz, sz, vp, vp, vp]
        for g in ("com1", "com2", "comt", "fr"):
            getattr(lib, f"gs_{g}_add").argtypes = [vp, sz, vp, vp, vp]
            getattr(lib, f"gs_{g}_sub").argtypes = [vp, sz, vp, vp, vp]
            getattr(lib, f"gs_{g}_neg").argtypes = [vp, sz, vp, vp]
        for g in ("com1", "com2", "comt"):
            getattr(lib, f"gs_{g}_sum").argtypes = [vp, sz, vp, vp]
        lib.gs_fr_scale.argtypes = [vp, sz, vp, vp, vp]
        for f in ("gs_g1_compress", "gs_g2_compress", "gs_fr_to_bytes", "gs_gt_to_bytes"):
            getattr(lib, f).argtypes = [vp, sz, vp, vp]
        for f in ("gs_g1_decompress", "gs_g2_decompress", "gs_g1_deserialize_uncompressed", "gs_g2_deserialize_uncompressed"):
            getattr(lib, f).argtypes = [vp, sz, vp, ci, vp, vp]
        for f in ("gs_g1_serialize_uncompressed", "gs_g2_serialize_uncompressed"):
            getattr(lib, f).argtypes = [vp, sz, vp, vp]
        for f in ("gs_fr_from_bytes", "gs_gt_from_bytes"):
            getattr(lib, f).argtypes = [vp, sz, vp, vp, vp]
        _lib = lib
    return _lib


def _buf(b):
    """bytes-like -> (keepalive, void*)"""
    if isinstance(b, bytes) and len(b):   # pass the bytes object's own buffer: no copy (a 1024 x 1024 Gamma is 32 MiB)
        return b, ctypes.cast(ctypes.c_char_p(b), ctypes.c_void_p)
    if isinstance(b, (bytes, bytearray, memoryview)):
        arr = (ctypes.c_char * len(b)).from_buffer_copy(bytes(b)) if len(b) else (ctypes.c_char * 1)()
        return arr, ctypes.cast(arr, ctypes.c_void_p)
    if hasattr(b, "ctypes"):  # numpy array (must be C-contiguous)
        return b, ctypes.c_void_p(b.ctypes.data)
    raise TypeError(f"unsupported buffer type {type(b)}")


def _a_size(ty): return G1 if ty in (PPE, MSMEG1) else FR
def _b_size(ty): return G2 if ty in (PPE, MSMEG2) else FR
def _t_size(ty): return {PPE: GT, MSMEG1: G1, MSMEG2: G2, QUAD: FR}[ty]
def _cx(ty): return 2 if ty in (PPE, MSMEG1) else 1
def _cy(ty): return 2 if ty in (PPE, MSMEG2) else 1


class Engine:
    """One GPU context (stream + device CRS + fixed-base tables + scratch)."""

    def __init__(self, device=0):
        self.lib = load_library()
        h = ctypes.c_void_p()
        rc = self.lib.gs_ctx_create(int(device), ctypes.byref(h))
        if rc != 0 or not h.value:
            raise GsError(rc, f"gs_ctx_create(device={device}) failed -- a CUDA device is required (no CPU fallback)")
        self.h = h
        self.device = device

    def close(self):
        if getattr(self, "h", None) is not None and self.h.value:
            self.lib.gs_ctx_destroy(self.h)
            self.h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _chk(self, rc):
        if rc != 0:
            raise GsError(rc, self.lib.gs_last_error(self.h).decode())

    @property
    def launch_count(self):
        return int(self.lib.gs_launch_count(self.h))

    @property
    def stream(self):
        return int(self.lib.gs_stream(self.h) or 0)

    # ---- measurement hooks
    def profile_enable(self, on=True):
        self._chk(self.lib.gs_profile_enable(self.h, 1 if on else 0))

    def profile_read(self):
        """{kernel name: (launches, total_ms)} since the last read (CUDA events on the engine's stream)."""
        buf = ctypes.create_string_buffer(1 << 16)
        n = self.lib.gs_profile_read(self.h, ctypes.cast(buf, ctypes.c_void_p), len(buf))
        if n < 0:
            raise GsError(-n, "gs_profile_read failed")
        out = {}
        for line in buf.value.decode().splitlines():
            name, cnt, ms = line.rsplit(" ", 2)
            out[name.strip("()")] = (int(cnt), float(ms))
        return out

    def fpmul_rate(self) -> float:
        r = ctypes.c_double()
        self._chk(self.lib.gs_diag_fpmul_rate(self.h, ctypes.byref(r)))
        return r.value

    # ---- CRS
    def crs_generate(self, p1, p2, a1, a2, t1, t2) -> bytes:
        out = ctypes.create_string_buffer(CRS_BYTES)
        ks = [_buf(x) for x in (p1, p2, a1, a2, t1, t2)]
        self._chk(self.lib.gs_crs_generate(self.h, *[k[1] for k in ks], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw

    def crs_load(self, crs: bytes):
        assert len(crs) == CRS_BYTES
        k = _buf(crs)
        self._chk(self.lib.gs_crs_load(self.h, k[1]))

    # ---- commitments
    def _commit(self, fn, n, a, b, out_size):
        out = ctypes.create_string_buffer(max(1, n * out_size))
        ka, kb = _buf(a), _buf(b)
        self._chk(fn(self.h, n, ka[1], kb[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * out_size]

    def batch_commit_g1(self, xvars: bytes, rand: bytes) -> bytes:
        n = len(xvars) // G1
        assert len(xvars) == n * G1 and len(rand) == 2 * n * FR
        return self._commit(self.lib.gs_batch_commit_g1, n, xvars, rand, COM1)

    def batch_commit_g2(self, yvars: bytes, rand: bytes) -> bytes:
        n = len(yvars) // G2
        assert len(yvars) == n * G2 and len(rand) == 2 * n * FR
        return self._commit(self.lib.gs_batch_commit_g2, n, yvars, rand, COM2)

    def batch_commit_scalar_b1(self, xs: bytes, rand: bytes) -> bytes:
        n = len(xs) // FR
        assert len(xs) == n * FR and len(rand) == n * FR
        return self._commit(self.lib.gs_batch_commit_scalar_b1, n, xs, rand, COM1)

    def batch_commit_scalar_b2(self, ys: bytes, rand: bytes) -> bytes:
        n = len(ys) // FR
        assert len(ys) == n * FR and len(rand) == n * FR
        return self._commit(self.lib.gs_batch_commit_scalar_b2, n, ys, rand, COM2)

    # ---- prove / verify
    def prove(self, ty, m, n, a_consts, b_consts, gamma, xvars, yvars, x_rand, y_rand, pf_rand):
        cx, cy = _cx(ty), _cy(ty)
        if m and n:
            assert len(a_consts) == n * _a_size(ty) and len(b_consts) == m * _b_size(ty)
            assert len(gamma) == m * n * FR and len(xvars) == m * _a_size(ty) and len(yvars) == n * _b_size(ty)
            assert len(x_rand) == m * cx * FR and len(y_rand) == n * cy * FR and len(pf_rand) == cx * cy * FR
        pi = ctypes.create_string_buffer(cx * COM2)
        th = ctypes.create_string_buffer(cy * COM1)
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, xvars, yvars, x_rand, y_rand, pf_rand)]
        self._chk(self.lib.gs_prove(self.h, ty, m, n, *[k[1] for k in ks], ctypes.cast(pi, ctypes.c_void_p),
                                    ctypes.cast(th, ctypes.c_void_p)))
        return pi.raw, th.raw

    def prove_batch(self, ty, count, m, n, a_consts, b_consts, gamma, xvars, yvars, x_rand, y_rand, pf_rand, shared_vars=False):
        """`count` independent proofs in one pass (gs_prove_batch); returns (pi bytes, theta bytes), proof-major."""
        cx, cy = _cx(ty), _cy(ty)
        reps = 1 if shared_vars else count
        if count and m and n:
            assert len(a_consts) == count * n * _a_size(ty) and len(b_consts) == count * m * _b_size(ty)
            assert len(gamma) == count * m * n * FR and len(pf_rand) == count * cx * cy * FR
            assert len(xvars) == reps * m * _a_size(ty) and len(yvars) == reps * n * _b_size(ty)
            assert len(x_rand) == reps * m * cx * FR and len(y_rand) == reps * n * cy * FR
        pi = ctypes.create_string_buffer(max(1, count * cx * COM2))
        th = ctypes.create_string_buffer(max(1, count * cy * COM1))
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, xvars, yvars, x_rand, y_rand, pf_rand)]
        self._chk(self.lib.gs_prove_batch(self.h, ty, count, m, n, *[k[1] for k in ks], 1 if shared_vars else 0,
                                          ctypes.cast(pi, ctypes.c_void_p), ctypes.cast(th, ctypes.c_void_p)))
        return pi.raw[: count * cx * COM2], th.raw[: count * cy * COM1]

    def rerandomize_batch(self, ty, count, m, n, a_consts, b_consts, gamma, xcoms, ycoms, pi, theta, x_rand, y_rand, pf_rand,
                          shared_coms=False):
        """`count` committed proofs rerandomised in one pass (gs_rerandomize_batch) with fresh R' = x_rand, S' = y_rand,
        T' = pf_rand; returns (xcoms, ycoms, pi, theta) bytes, proof-major.  With shared_coms the commitments and R', S'
        are one set for every equation, and so are the returned commitments."""
        cx, cy = _cx(ty), _cy(ty)
        reps = 1 if shared_coms else count
        if count and m and n:
            assert len(a_consts) == count * n * _a_size(ty) and len(b_consts) == count * m * _b_size(ty)
            assert len(gamma) == count * m * n * FR and len(pf_rand) == count * cx * cy * FR
            assert len(pi) == count * cx * COM2 and len(theta) == count * cy * COM1
            assert len(xcoms) == reps * m * COM1 and len(ycoms) == reps * n * COM2
            assert len(x_rand) == reps * m * cx * FR and len(y_rand) == reps * n * cy * FR
        outs = [ctypes.create_string_buffer(max(1, k)) for k in
                (reps * m * COM1, reps * n * COM2, count * cx * COM2, count * cy * COM1)]
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, xcoms, ycoms, pi, theta, x_rand, y_rand, pf_rand)]
        self._chk(self.lib.gs_rerandomize_batch(self.h, ty, count, m, n, *[k[1] for k in ks], 1 if shared_coms else 0,
                                                *[ctypes.cast(o, ctypes.c_void_p) for o in outs]))
        return (outs[0].raw[: reps * m * COM1], outs[1].raw[: reps * n * COM2], outs[2].raw[: count * cx * COM2],
                outs[3].raw[: count * cy * COM1])

    def rerandomize(self, ty, m, n, a_consts, b_consts, gamma, xcoms, ycoms, pi, theta, x_rand, y_rand, pf_rand):
        """One committed proof rerandomised (gs_rerandomize); returns (xcoms, ycoms, pi, theta) bytes."""
        cx, cy = _cx(ty), _cy(ty)
        if m and n:
            assert len(a_consts) == n * _a_size(ty) and len(b_consts) == m * _b_size(ty) and len(gamma) == m * n * FR
            assert len(xcoms) == m * COM1 and len(ycoms) == n * COM2 and len(pi) == cx * COM2 and len(theta) == cy * COM1
            assert len(x_rand) == m * cx * FR and len(y_rand) == n * cy * FR and len(pf_rand) == cx * cy * FR
        outs = [ctypes.create_string_buffer(max(1, k)) for k in (m * COM1, n * COM2, cx * COM2, cy * COM1)]
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, xcoms, ycoms, pi, theta, x_rand, y_rand, pf_rand)]
        self._chk(self.lib.gs_rerandomize(self.h, ty, m, n, *[k[1] for k in ks], *[ctypes.cast(o, ctypes.c_void_p) for o in outs]))
        return outs[0].raw[: m * COM1], outs[1].raw[: n * COM2], outs[2].raw[: cx * COM2], outs[3].raw[: cy * COM1]

    # ---- extraction with the binding key (gs_extract)
    def extract(self, xcoms: bytes = b"", xkey: bytes = None, ycoms: bytes = b"", ykey: bytes = None):
        """X_i = xcoms[i].1 - xkey xcoms[i].0 and Y_i = ycoms[i].1 - ykey ycoms[i].0 in one call; xkey = a1, ykey = a2 of
        crs_generate (Fr bytes).  Returns (G1 bytes, G2 bytes).  A key that does not match the loaded CRS raises GsError."""
        nx, ny = len(xcoms) // COM1, len(ycoms) // COM2
        assert len(xcoms) == nx * COM1 and len(ycoms) == ny * COM2
        assert (not nx or len(xkey) == FR) and (not ny or len(ykey) == FR)
        ox, oy = ctypes.create_string_buffer(max(1, nx * G1)), ctypes.create_string_buffer(max(1, ny * G2))
        ks = [_buf(x) if x else (None, ctypes.c_void_p(0)) for x in (xcoms, xkey, ycoms, ykey)]
        self._chk(self.lib.gs_extract(self.h, nx, ks[0][1], ks[1][1], ny, ks[2][1], ks[3][1], ctypes.cast(ox, ctypes.c_void_p),
                                      ctypes.cast(oy, ctypes.c_void_p)))
        return ox.raw[: nx * G1], oy.raw[: ny * G2]

    @staticmethod
    def _check_verify_sizes(ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta, gamma_rows=None):
        """The C side reads count * (shape) bytes from every buffer: a short one would be read past its end.  Gamma holds
        `gamma_rows` rows per problem (default m; gs_verify_sharded: this rank's rows only)."""
        cx, cy = _cx(ty), _cy(ty)
        gm = m if gamma_rows is None else gamma_rows
        want = [count * n * _a_size(ty), count * m * _b_size(ty), count * gm * n * FR, count * _t_size(ty),
                count * m * COM1, count * n * COM2, count * cx * COM2, count * cy * COM1]
        names = ["a_consts", "b_consts", "gamma", "target", "xcoms", "ycoms", "pi", "theta"]
        for nm, buf, w in zip(names, (a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta), want):
            have = buf.nbytes if hasattr(buf, "nbytes") else len(buf)
            if have != w:
                raise GsError(1, f"verify: {nm} is {have} bytes, expected {w} for type {ty}, count {count}, m {m}, n {n}")

    def verify_batch(self, ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta) -> bytes:
        if count and m and n:
            self._check_verify_sizes(ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)
        ok = ctypes.create_string_buffer(max(1, count))
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)]
        self._chk(self.lib.gs_verify_batch(self.h, ty, count, m, n, *[k[1] for k in ks], ctypes.cast(ok, ctypes.c_void_p)))
        return ok.raw[:count]

    def verify_batch_dev(self, ty, count, m, n, ptrs, out_ok_ptr):
        """All-device variant: `ptrs` = 8 device addresses (ints) in C-ABI order; asynchronous on self.stream."""
        self._chk(self.lib.gs_verify_batch_dev(self.h, ty, count, m, n, *[ctypes.c_void_p(int(p)) for p in ptrs],
                                               ctypes.c_void_p(int(out_ok_ptr))))

    def verify(self, ty, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta) -> bool:
        return self.verify_batch(ty, 1, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta) == b"\x01"

    # ---- randomised batch verification (gs_verify_batch_rand, SURVEY.md 8f.4): ONE verdict for the batch
    @staticmethod
    def _rho(count, rho):
        """2*count + 1 random 64-bit words; drawn from the OS CSPRNG unless the caller brings them (tests: a fixed seed)."""
        need = 8 * (2 * count + 1)
        if rho is None:
            import secrets
            rho = secrets.token_bytes(need)
        if len(rho) != need:
            raise GsError(1, f"verify_batch_rand: rho is {len(rho)} bytes, expected {need}")
        return rho

    def verify_batch_rand(self, ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta, rho=None) -> bool:
        """True iff every proof of the batch verifies (error <= 2^-62 over rho).  Not the reference's per-proof answer: on
        False, verify_batch says which ones failed."""
        if count and m and n:
            self._check_verify_sizes(ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)
        kr = _buf(self._rho(count, rho))
        ok = ctypes.create_string_buffer(1)
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)]
        self._chk(self.lib.gs_verify_batch_rand(self.h, ty, count, m, n, *[k[1] for k in ks], kr[1], ctypes.cast(ok, ctypes.c_void_p)))
        return ok.raw == b"\x01"

    def verify_batch_rand_dev(self, ty, count, m, n, ptrs, out_ok_ptr, rho=None):
        """All-device variant (rho stays on the host); asynchronous on self.stream, one verdict byte at out_ok_ptr."""
        kr = _buf(self._rho(count, rho))
        self._chk(self.lib.gs_verify_batch_rand_dev(self.h, ty, count, m, n, *[ctypes.c_void_p(int(p)) for p in ptrs], kr[1],
                                                    ctypes.c_void_p(int(out_ok_ptr))))

    # ---- randomised per-proof verification (gs_verify_each_rand): one verdict per proof, one final exponentiation each
    def verify_each_rand(self, ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta, rho=None) -> bytes:
        """count verdict bytes: 1 iff proof p verifies (a bad proof passes with probability <= 2^-62 over rho, each on its
        own).  Same weights and rho layout as verify_batch_rand; not bit-comparable with verify_batch."""
        if count and m and n:
            self._check_verify_sizes(ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)
        kr = _buf(self._rho(count, rho))
        ok = ctypes.create_string_buffer(max(1, count))
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)]
        self._chk(self.lib.gs_verify_each_rand(self.h, ty, count, m, n, *[k[1] for k in ks], kr[1], ctypes.cast(ok, ctypes.c_void_p)))
        return ok.raw[:count]

    def verify_each_rand_dev(self, ty, count, m, n, ptrs, out_ok_ptr, rho=None):
        """All-device variant (rho stays on the host); asynchronous on self.stream, count verdict bytes at out_ok_ptr."""
        kr = _buf(self._rho(count, rho))
        self._chk(self.lib.gs_verify_each_rand_dev(self.h, ty, count, m, n, *[ctypes.c_void_p(int(p)) for p in ptrs], kr[1],
                                                   ctypes.c_void_p(int(out_ok_ptr))))

    # ---- one statement sharded by slot over several GPUs (gs_verify_partial / gs_verify_finish)
    def verify_partial(self, ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta, rank, world) -> bytes:
        """This rank's un-exponentiated Miller products: count x 4 GT values (2304 B per statement)."""
        if count and m and n:
            self._check_verify_sizes(ty, count, m, n, a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)
        out = ctypes.create_string_buffer(max(1, count * COMT))
        ks = [_buf(x) for x in (a_consts, b_consts, gamma, target, xcoms, ycoms, pi, theta)]
        self._chk(self.lib.gs_verify_partial(self.h, ty, count, m, n, *[k[1] for k in ks], int(rank), int(world),
                                             ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: count * COMT]

    def verify_finish(self, ty, count, partials: bytes, target: bytes) -> bytes:
        """partials = the ranks' verify_partial outputs concatenated rank-major; returns count verdict bytes."""
        assert count and len(partials) % (count * COMT) == 0
        nparts = len(partials) // (count * COMT)
        ok = ctypes.create_string_buffer(max(1, count))
        kp, kt = _buf(partials), _buf(target)
        self._chk(self.lib.gs_verify_finish(self.h, ty, count, nparts, kp[1], kt[1], ctypes.cast(ok, ctypes.c_void_p)))
        return ok.raw[:count]

    def verify_sharded(self, ty, count, m, n, a_consts, b_consts, gamma_rows, target, xcoms, ycoms, pi, theta, rank, world,
                       allgather) -> bytes:
        """gs_verify_sharded: the statement MSM split by base, the Miller pairs by slot, two all-gathers through
        `allgather(send_ptr, recv_ptr, nbytes) -> None` (device pointers; shard.make_allgather builds one over
        torch.distributed).  gamma_rows = this rank's rows of Gamma only (shard.gamma_rows_of)."""
        self._check_verify_sizes(ty, count, m, n, a_consts, b_consts, gamma_rows, target, xcoms, ycoms, pi, theta,
                                 gamma_rows=len(range(rank, m, world)))
        err = []

        def cb(_user, send, recv, nbytes):
            try:
                allgather(int(send), int(recv), int(nbytes))
                return 0
            except Exception as ex:  # noqa: BLE001 -- must not unwind through the C frames
                err.append(ex)
                return 1

        fn = ALLGATHER_FN(cb)
        ok = ctypes.create_string_buffer(max(1, count))
        ks = [_buf(x) if len(x) else (None, ctypes.c_void_p(0)) for x in (a_consts, b_consts, gamma_rows, target, xcoms, ycoms, pi, theta)]
        rc = self.lib.gs_verify_sharded(self.h, ty, count, m, n, *[k[1] for k in ks], int(rank), int(world), fn, None,
                                        ctypes.cast(ok, ctypes.c_void_p))
        if err:
            raise err[0]
        self._chk(rc)
        return ok.raw[:count]

    # ---- ComT
    def comt_pairing(self, xs: bytes, ys: bytes) -> bytes:
        n = len(xs) // COM1
        assert len(xs) == n * COM1 and len(ys) == n * COM2
        out = ctypes.create_string_buffer(max(1, n * COMT))
        kx, ky = _buf(xs), _buf(ys)
        self._chk(self.lib.gs_comt_pairing(self.h, n, kx[1], ky[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * COMT]

    def comt_pairing_sum(self, xs: bytes, ys: bytes) -> bytes:
        k = len(xs) // COM1
        if len(xs) != k * COM1 or len(ys) != k * COM2:
            raise GsError(1, "pairing_sum: length mismatch")  # reference: assert_eq!(x_vec.len(), y_vec.len())
        out = ctypes.create_string_buffer(COMT)
        kx, ky = _buf(xs), _buf(ys)
        self._chk(self.lib.gs_comt_pairing_sum(self.h, k, kx[1], ky[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw

    def comt_linear_map(self, ty, target: bytes) -> bytes:
        assert len(target) == _t_size(ty)
        out = ctypes.create_string_buffer(COMT)
        kt = _buf(target)
        self._chk(self.lib.gs_comt_linear_map(self.h, ty, kt[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw

    def pairing(self, ps: bytes, qs: bytes) -> bytes:
        n = len(ps) // G1
        assert len(ps) == n * G1 and len(qs) == n * G2
        out = ctypes.create_string_buffer(max(1, n * GT))
        kp, kq = _buf(ps), _buf(qs)
        self._chk(self.lib.gs_pairing(self.h, n, kp[1], kq[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * GT]

    # ---- entry-wise group arithmetic: kind in ("com1", "com2", "comt", "fr"); element sizes from the ABI
    _ESIZE = {"com1": COM1, "com2": COM2, "comt": COMT, "fr": FR}

    def elementwise(self, kind, op, a: bytes, b: bytes = None) -> bytes:
        """op in ("add", "sub", "neg"): out[i] = a[i] op b[i] over len(a) / element-size elements."""
        es = self._ESIZE[kind]
        n = len(a) // es
        assert len(a) == n * es and (op == "neg" or len(b) == len(a))
        out = ctypes.create_string_buffer(max(1, n * es))
        ka = _buf(a)
        fn = getattr(self.lib, f"gs_{kind}_{op}")
        if op == "neg":
            self._chk(fn(self.h, n, ka[1], ctypes.cast(out, ctypes.c_void_p)))
        else:
            kb = _buf(b)
            self._chk(fn(self.h, n, ka[1], kb[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * es]

    def group_sum(self, kind, a: bytes) -> bytes:
        es = self._ESIZE[kind]
        n = len(a) // es
        assert len(a) == n * es and kind != "fr"
        out = ctypes.create_string_buffer(es)
        ka = _buf(a)
        self._chk(getattr(self.lib, f"gs_{kind}_sum")(self.h, n, ka[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw

    def fr_scale(self, s: bytes, a: bytes) -> bytes:
        n = len(a) // FR
        assert len(s) == FR and len(a) == n * FR
        out = ctypes.create_string_buffer(max(1, n * FR))
        ks, ka = _buf(s), _buf(a)
        self._chk(self.lib.gs_fr_scale(self.h, n, ks[1], ka[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * FR]

    # ---- wire formats: kind in ("g1", "g2") for points, ("fr", "gt") for canonical integers
    _WIRE = {"g1": (G1, 48), "g2": (G2, 96), "fr": (FR, 32), "gt": (GT, 576)}

    def serialize(self, kind, elems: bytes, compressed=True) -> bytes:
        """ABI elements -> wire bytes (compressed / uncompressed points, canonical little-endian integers)."""
        if not compressed and kind in ("g1", "g2"):
            return self._uncompressed(kind, elems)
        esz, wsz = self._WIRE[kind]
        n = len(elems) // esz
        assert len(elems) == n * esz
        out = ctypes.create_string_buffer(max(1, n * wsz))
        k = _buf(elems)
        fn = getattr(self.lib, f"gs_{kind}_compress" if kind in ("g1", "g2") else f"gs_{kind}_to_bytes")
        self._chk(fn(self.h, n, k[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * wsz]

    def _uncompressed(self, kind, elems):
        esz = self._WIRE[kind][0]
        n = len(elems) // esz
        assert len(elems) == n * esz
        out = ctypes.create_string_buffer(max(1, n * esz))
        k = _buf(elems)
        self._chk(getattr(self.lib, f"gs_{kind}_serialize_uncompressed")(self.h, n, k[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: n * esz]

    def deserialize(self, kind, wire: bytes, check_subgroup=True, compressed=True):
        """wire bytes -> (ABI elements, verdict bytes); invalid encodings give verdict 0 and a zeroed element."""
        if not compressed and kind in ("g1", "g2"):
            esz = self._WIRE[kind][0]
            n = len(wire) // esz
            assert len(wire) == n * esz
            out = ctypes.create_string_buffer(max(1, n * esz))
            ok = ctypes.create_string_buffer(max(1, n))
            k = _buf(wire)
            self._chk(getattr(self.lib, f"gs_{kind}_deserialize_uncompressed")(self.h, n, k[1], 1 if check_subgroup else 0,
                                                                               ctypes.cast(out, ctypes.c_void_p), ctypes.cast(ok, ctypes.c_void_p)))
            return out.raw[: n * esz], ok.raw[:n]
        esz, wsz = self._WIRE[kind]
        n = len(wire) // wsz
        assert len(wire) == n * wsz
        out = ctypes.create_string_buffer(max(1, n * esz))
        ok = ctypes.create_string_buffer(max(1, n))
        k = _buf(wire)
        if kind in ("g1", "g2"):
            self._chk(getattr(self.lib, f"gs_{kind}_decompress")(self.h, n, k[1], 1 if check_subgroup else 0,
                                                               ctypes.cast(out, ctypes.c_void_p), ctypes.cast(ok, ctypes.c_void_p)))
        else:
            self._chk(getattr(self.lib, f"gs_{kind}_from_bytes")(self.h, n, k[1], ctypes.cast(out, ctypes.c_void_p),
                                                               ctypes.cast(ok, ctypes.c_void_p)))
        return out.raw[: n * esz], ok.raw[:n]

    # ---- Mat
    def _matmul(self, fn, r, k, c, lhs, mat, esize_l, esize_m, esize_o):
        assert len(lhs) == r * k * esize_l and len(mat) == k * c * esize_m
        out = ctypes.create_string_buffer(max(1, r * c * esize_o))
        kl, km = _buf(lhs), _buf(mat)
        self._chk(fn(self.h, r, k, c, kl[1], km[1], ctypes.cast(out, ctypes.c_void_p)))
        return out.raw[: r * c * esize_o]

    def com1_matmul(self, r, k, c, lhs, mat): return self._matmul(self.lib.gs_com1_matmul, r, k, c, lhs, mat, FR, COM1, COM1)
    def com2_matmul(self, r, k, c, lhs, mat): return self._matmul(self.lib.gs_com2_matmul, r, k, c, lhs, mat, FR, COM2, COM2)
    def fr_matmul(self, r, k, c, a, b): return self._matmul(self.lib.gs_fr_matmul, r, k, c, a, b, FR, FR, FR)
