"""Builds libgs_b200.so in-tree with nvcc for sm_100a (cross-compiles without a GPU).

One translation unit per kernel family, compiled in parallel (cicc and ptxas are single-threaded per
TU and the big-integer kernels are tens of thousands of instructions each), then linked.

    python groth-sahai-rs_b200/build.py [--force] [-v]
"""
import os
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
OBJ = os.path.join(HERE, "build")
OUT = os.path.join(HERE, "libgs_b200.so")
SOURCES = ["core.cu", "pairing.cu", "finalexp.cu", "verify.cu", "prover.cu", "prover_g1.cu", "prover_g2.cu", "groupops.cu", "serial.cu", "extract.cu"]
NVCC_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
              "-Xcompiler", "-fPIC"]


def _headers():
    hs = [os.path.join(CSRC, f) for f in os.listdir(CSRC) if f.endswith((".cuh", ".h", ".inc"))]
    hs.append(os.path.join(HERE, "..", "include", "gs_b200.h"))
    return hs


def _sources():
    return [s for s in SOURCES if os.path.exists(os.path.join(CSRC, s))]


def _stale(target, deps):
    if not os.path.exists(target):
        return True
    t = os.path.getmtime(target)
    return any(os.path.getmtime(d) > t for d in deps)


def build(force=False, verbose=False):
    """GS_EXTRA_NVCC_FLAGS (e.g. "-DGS_FP2_INLINE") and GS_LIB_OUT (output path) build experiment variants beside the product."""
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    extra = os.environ.get("GS_EXTRA_NVCC_FLAGS", "").split()
    global OBJ, OUT
    if os.environ.get("GS_LIB_OUT"):
        OUT = os.path.abspath(os.environ["GS_LIB_OUT"])
        OBJ = OUT + ".objs"
        force = True
    os.makedirs(OBJ, exist_ok=True)
    hdrs = _headers()
    jobs = []
    objs = []
    for src in _sources():
        obj = os.path.join(OBJ, src.replace(".cu", ".o"))
        objs.append(obj)
        if force or _stale(obj, hdrs + [os.path.join(CSRC, src)]):
            jobs.append([nvcc] + NVCC_FLAGS + extra + (["-Xptxas", "-v"] if verbose else []) + ["-c", "-o", obj, src])
    if jobs:
        def run(cmd):
            r = subprocess.run(cmd, cwd=CSRC, capture_output=True, text=True)
            return cmd, r
        with ThreadPoolExecutor(max_workers=min(len(jobs), os.cpu_count() or 4)) as ex:
            for cmd, r in ex.map(run, jobs):
                if verbose or r.returncode != 0:
                    sys.stderr.write(" ".join(cmd) + "\n" + r.stdout + r.stderr)
                if r.returncode != 0:
                    raise subprocess.CalledProcessError(r.returncode, cmd)
    if jobs or force or _stale(OUT, objs):
        subprocess.check_call([nvcc, "-shared", "-gencode", "arch=compute_100a,code=sm_100a", "-o", OUT] + objs, cwd=CSRC)
    return OUT


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose="-v" in sys.argv))
