#!/usr/bin/env python3
"""Extraction with the binding key (gs_extract) against batch_commit of the same shape: 2^20 G1 + 2^20 G2 commitments
(the C2 shape) by default.  Inputs are seeded (random Fr randomness; witnesses = a pool of distinct multiples of the CRS
generators, tiled).  Every call is a host-buffer call that ends in a device synchronise; the legs alternate within one
process.  Reported per leg:
  * end to end: the host call (copies in and out included), median over --reps;
  * resident: the kernels alone -- one profiled call of each leg (CUDA events around every launch, gs_profile_enable /
    gs_profile_read) and, for extraction, one unchunked launch per side at --resident-n elements (inputs already in HBM
    when the event pair starts, so the event time is the kernel's).
Card name and power limit are read in the same run.  Writes one JSON document.

    python tools/bench_extract.py [--n 1048576] [--reps 5] [--out extract.json]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

FR, G1, G2, COM1, COM2 = 32, 96, 192, 192, 384


def rand_fr(n, seed):
    """n field elements (Montgomery limbs below 2^254, so below the modulus)"""
    rs = np.random.RandomState(seed)
    a = rs.randint(0, 2 ** 63 - 1, size=(n, 4), dtype=np.int64).astype(np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a.tobytes()


def points(eng, gen, k, seed, g2side, pool=4096):
    """k points: a pool of distinct multiples of the generator, tiled"""
    p = min(k, pool)
    ks = rand_fr(p, seed)
    if g2side:
        out = np.frombuffer(eng.com2_matmul(p, 1, 1, ks, gen + gen), dtype=np.uint8).reshape(p, COM2)[:, :G2]
    else:
        out = np.frombuffer(eng.com1_matmul(p, 1, 1, ks, gen + gen), dtype=np.uint8).reshape(p, COM1)[:, :G1]
    return np.resize(out, (k, out.shape[1])).tobytes()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as ex:  # noqa: BLE001
        return {"gpu": "unknown", "error": str(ex)}


def profiled(eng, fn):
    eng.profile_enable(True)
    fn()
    prof = eng.profile_read()
    eng.profile_enable(False)
    return {k: {"launches": v[0], "ms": round(v[1], 4)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20, help="commitments per side")
    ap.add_argument("--resident-n", type=int, default=1 << 17, help="elements per side of the single-launch kernel timing")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import groth_sahai_rs_b200 as gsb
    from gsutil import make_crs, crs_bytes, fr_b, g1_b, g2_b
    crs, draws = make_crs(7)
    a1, a2 = fr_b(draws[2]), fr_b(draws[3])
    eng = gsb.Engine(0)
    eng.crs_load(crs_bytes(crs))
    g1, g2 = g1_b(crs.g1_gen), g2_b(crs.g2_gen)
    n = args.n
    X, Y = points(eng, g1, n, 21, False), points(eng, g2, n, 22, True)
    xr, yr = rand_fr(2 * n, 23), rand_fr(2 * n, 24)
    xc, yc = eng.batch_commit_g1(X, xr), eng.batch_commit_g2(Y, yr)

    def commit_leg():
        eng.batch_commit_g1(X, xr)
        eng.batch_commit_g2(Y, yr)

    def extract_leg():
        return eng.extract(xc, a1, yc, a2)

    commit_leg()
    got = extract_leg()  # warm-up (module load, key check)
    assert got == (X, Y), "extract(commit(X)) != X"
    tc, te = [], []
    for _ in range(args.reps):
        for leg, ts in ((commit_leg, tc), (extract_leg, te)):
            t0 = time.perf_counter()
            leg()
            ts.append(time.perf_counter() - t0)
    mc, me = statistics.median(tc), statistics.median(te)
    doc = {"card": card(), "n_per_side": n, "reps": args.reps,
           "end_to_end": {"batch_commit_ms": [round(t * 1e3, 3) for t in tc], "extract_ms": [round(t * 1e3, 3) for t in te],
                          "batch_commit_median_ms": round(mc * 1e3, 3), "extract_median_ms": round(me * 1e3, 3),
                          "batch_commit_per_s_per_side": round(n / mc, 1), "extract_per_s_per_side": round(n / me, 1),
                          "time_ratio_extract_over_commit": round(me / mc, 3)},
           "kernels_extract": profiled(eng, extract_leg), "kernels_commit": profiled(eng, commit_leg)}
    # resident: one unchunked k_extract launch per side (inputs uploaded before the event pair opens)
    rn = args.resident_n
    res = {}
    for side, coms, key in (("g1", xc[:rn * COM1], a1), ("g2", yc[:rn * COM2], a2)):
        ms = []
        for _ in range(args.reps):
            prof = profiled(eng, lambda: eng.extract(coms, key) if side == "g1" else eng.extract(ycoms=coms, ykey=key))
            ms.append(prof["k_extract<F>"]["ms"])
        med = statistics.median(ms)
        res[side] = {"n": rn, "kernel_ms": ms, "kernel_median_ms": med, "per_s": round(rn / (med * 1e-3), 1)}
    doc["resident_extract"] = res
    eng.close()
    text = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(json.dumps({"card": doc["card"], "end_to_end": doc["end_to_end"], "resident_extract": res}))


if __name__ == "__main__":
    main()
