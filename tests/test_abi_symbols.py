"""CPU-side checks of the drop-in boundary: the C-ABI library builds (cross-compile, no GPU),
loads, and exports every symbol include/gs_b200.h declares.  No compute calls here."""
import ctypes
import os
import re
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def lib():
    sys.path.insert(0, ROOT)
    import __graft_entry__
    __graft_entry__.build_product()
    import groth_sahai_rs_b200 as gsb
    return gsb.load_library()


def header_symbols():
    src = open(os.path.join(ROOT, "include", "gs_b200.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(gs_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported(lib):
    syms = header_symbols()
    assert len(syms) >= 20
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/gs_b200.h but not exported"


def test_python_binding_covers_header(lib):
    import groth_sahai_rs_b200 as gsb
    assert sorted(gsb.EXPORTED_SYMBOLS) == header_symbols()


def test_no_cpu_fallback():
    """Without a CUDA device the product must fail loudly, never compute on the CPU.  Checked in a child process with every
    device hidden, so that it runs on a machine with a GPU as well."""
    code = ("import sys\nsys.path.insert(0, %r)\nimport groth_sahai_rs_b200 as gsb\n"
            "try:\n    gsb.Engine(0)\nexcept gsb.GsError:\n    sys.exit(0)\nsys.exit('Engine(0) did not raise GsError')") % ROOT
    r = subprocess.run([sys.executable, "-c", code], env=dict(os.environ, CUDA_VISIBLE_DEVICES=""),
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr


def test_product_does_not_import_oracle():
    pkg = os.path.join(ROOT, "groth-sahai-rs_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".inc", ".h")):
                txt = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in txt and "from oracle" not in txt and "oracle/" not in txt.replace("(the oracle", ""), f


def test_vector_matrix_helpers_are_pure_host_reshapes():
    """col_vec_to_vec / vec_to_col_vec (data_structures.rs:143-160), as_col_vec / as_vec (:301-307, :346-352) and the
    From<Matrix> impls (:283-298, :467-474) with their dimension asserts: no device work, so they are checked here."""
    import pytest
    from groth_sahai_rs_b200 import api
    a, b = bytes([1]) * 96, bytes([2]) * 96
    c = api.Com1.from_matrix([[a], [b]])
    assert c == a + b and api.Com1.as_vec(c) == [a, b] and api.Com1.as_col_vec(c) == [[a], [b]]
    q, r = bytes([3]) * 192, bytes([4]) * 192
    d = api.Com2.from_matrix(api.Com2.as_col_vec(q + r))
    assert d == q + r and api.Com2.as_vec(d) == [q, r]
    g = [bytes([i]) * 576 for i in range(4)]
    t = api.ComT.from_matrix([[g[0], g[1]], [g[2], g[3]]])
    assert api.ComT.as_matrix(t) == [[g[0], g[1]], [g[2], g[3]]]                 # row-major, :1361-1377
    assert api.col_vec_to_vec([[a], [b]]) == [a, b] and api.col_vec_to_vec([[a, b]]) == [a, b]
    assert api.vec_to_col_vec([a, b]) == [[a], [b]] and api.col_vec_to_vec(api.vec_to_col_vec([a])) == [a]
    for bad in ([[a]], [[a, b], [b]], [[a], [b], [a]]):
        with pytest.raises(AssertionError):
            api.Com1.from_matrix(bad)
    with pytest.raises(AssertionError):
        api.ComT.from_matrix([[g[0]], [g[1]]])


def test_rust_shim_binds_the_header():
    """rust/src/ffi.rs (the host shim a maintainer builds; this image has no rustc) declares every symbol of
    include/gs_b200.h that the reference's API needs -- everything except the measurement hooks and the `_dev` variants --
    and nothing the header does not have."""
    src = open(os.path.join(ROOT, "rust", "src", "ffi.rs")).read()
    rust = set(re.findall(r"pub fn (gs_[a-z0-9_]+)\s*\(", src))
    hdr = set(header_symbols())
    assert rust <= hdr, sorted(rust - hdr)
    skipped = {s for s in hdr if s.endswith("_dev")} | {"gs_stream", "gs_profile_enable", "gs_profile_read", "gs_diag_fpmul_rate"}
    assert hdr - rust <= skipped, sorted(hdr - rust - skipped)
    # one shim body per public function of the reference's API (SURVEY.md §8b)
    tree = "".join(open(os.path.join(ROOT, "rust", "src", f)).read() for f in
                   ("generator.rs", "verifier.rs", "data_structures.rs", "statement.rs", "prover/commit.rs", "prover/prove.rs"))
    for name in ("generate_crs", "batch_commit_G1", "batch_commit_G2", "batch_commit_scalar_to_B1", "batch_commit_scalar_to_B2",
                 "commit_G1", "commit_G2", "commit_scalar_to_B1", "commit_scalar_to_B2", "commit_and_prove", "fn prove<",
                 "fn verify(", "fn pairing(", "fn pairing_sum(", "linear_map_PPE", "linear_map_MSMEG1", "linear_map_MSMEG2",
                 "linear_map_quad", "scalar_linear_map", "batch_scalar_linear_map", "fn scalar_mul(", "fn left_mul(", "fn right_mul(",
                 "col_vec_to_vec", "vec_to_col_vec", "fn append("):
        assert name in tree, name
