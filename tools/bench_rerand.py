#!/usr/bin/env python3
"""Proof rerandomisation (gs_rerandomize_batch) against commit + prove of the same shape, from host buffers, on three
workloads: C5 (65,536 independent 4 x 4 PPE proofs), C4 (1,024 equations over one set of 64 x 64 commitments) and C3
(one 1024 x 1024 PPE, latency).  Inputs are seeded (random Fr; points = multiples of the CRS generators, a pool of
distinct points tiled over the batch).  The two legs alternate within one process, each call ends in a device
synchronise (the host-buffer entry points return after their copies back); after the timed reps one profiled call of
each leg gives the per-kernel CUDA-event times (gs_profile_enable / gs_profile_read).  Card name and power limit are read
in the same run.  Writes one JSON document.

    python tools/bench_rerand.py [--reps 5] [--out rerand.json]
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

FR, COM1, COM2 = 32, 192, 384


def rand_fr(n, seed):
    """n field elements (Montgomery limbs below 2^254, so below the modulus)"""
    rs = np.random.RandomState(seed)
    a = rs.randint(0, 2 ** 63 - 1, size=(n, 4), dtype=np.int64).astype(np.uint64)
    a[:, 3] &= np.uint64((1 << 62) - 1)
    return a.tobytes()


def points(eng, gen2, k, seed, g2side, pool=4096):
    """k points: a pool of distinct multiples of the generator, tiled"""
    p = min(k, pool)
    ks = rand_fr(p, seed)
    if g2side:
        out = np.frombuffer(eng.com2_matmul(p, 1, 1, ks, gen2 + gen2), dtype=np.uint8).reshape(p, 384)[:, :192]
    else:
        out = np.frombuffer(eng.com1_matmul(p, 1, 1, ks, gen2 + gen2), dtype=np.uint8).reshape(p, 192)[:, :96]
    return np.resize(out, (k, out.shape[1])).tobytes()


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "max_sm_clock": clk}
    except Exception as ex:  # noqa: BLE001
        return {"gpu": "unknown", "error": str(ex)}


def timed(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts


def workload(eng, g1, g2, count, m, n, shared, seed):
    """PPE inputs + a committed proof of each equation (made by the engine; the proofs need not verify to be timed)"""
    reps = 1 if shared else count
    w = dict(count=count, m=m, n=n, shared=shared)
    w["A"] = points(eng, g1, count * n, seed, False)
    w["B"] = points(eng, g2, count * m, seed + 1, True)
    w["G"] = rand_fr(count * m * n, seed + 2)
    w["X"] = points(eng, g1, reps * m, seed + 3, False)
    w["Y"] = points(eng, g2, reps * n, seed + 4, True)
    w["xr"], w["yr"] = rand_fr(reps * m * 2, seed + 5), rand_fr(reps * n * 2, seed + 6)
    w["Tr"] = rand_fr(count * 4, seed + 7)
    w["xr2"], w["yr2"] = rand_fr(reps * m * 2, seed + 8), rand_fr(reps * n * 2, seed + 9)
    w["Tr2"] = rand_fr(count * 4, seed + 10)
    commit_prove(eng, w)
    w["xc"], w["yc"], w["pi"], w["th"] = w.pop("out")
    return w


def commit_prove(eng, w):
    xc = eng.batch_commit_g1(w["X"], w["xr"])
    yc = eng.batch_commit_g2(w["Y"], w["yr"])
    if w["count"] == 1:
        pi, th = eng.prove(0, w["m"], w["n"], w["A"], w["B"], w["G"], w["X"], w["Y"], w["xr"], w["yr"], w["Tr"])
    else:
        pi, th = eng.prove_batch(0, w["count"], w["m"], w["n"], w["A"], w["B"], w["G"], w["X"], w["Y"], w["xr"], w["yr"],
                                 w["Tr"], shared_vars=w["shared"])
    w["out"] = (xc, yc, pi, th)


def rerandomize(eng, w):
    args = (w["A"], w["B"], w["G"], w["xc"], w["yc"], w["pi"], w["th"], w["xr2"], w["yr2"], w["Tr2"])
    if w["count"] == 1:
        return eng.rerandomize(0, w["m"], w["n"], *args)
    return eng.rerandomize_batch(0, w["count"], w["m"], w["n"], *args, shared_coms=w["shared"])


def profiled(eng, fn):
    eng.profile_enable(True)
    fn()
    prof = eng.profile_read()
    eng.profile_enable(False)
    return {k: {"launches": v[0], "ms": round(v[1], 4)} for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c5", type=int, default=65536)
    ap.add_argument("--c4", type=int, default=1024)
    ap.add_argument("--c3", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import groth_sahai_rs_b200 as gsb
    from gsutil import make_crs, crs_bytes, g1_b, g2_b
    crs, _ = make_crs(7)
    eng = gsb.Engine(0)
    eng.crs_load(crs_bytes(crs))
    g1, g2 = g1_b(crs.g1_gen), g2_b(crs.g2_gen)
    doc = {"card": card(), "reps": args.reps, "workloads": {}}
    shapes = {"C5": (args.c5, 4, 4, False), "C4": (args.c4, 64, 64, True), "C3": (1, args.c3, args.c3, False)}
    for name, (count, m, n, shared) in shapes.items():
        w = workload(eng, g1, g2, count, m, n, shared, seed=11)
        prove_leg, rr_leg = (lambda: commit_prove(eng, w)), (lambda: rerandomize(eng, w))
        prove_leg()
        rr_leg()  # warm-up (module load, fixed-base tables at the batch's window size)
        tp, tr = [], []
        for _ in range(args.reps):
            tp += timed(prove_leg, 1)
            tr += timed(rr_leg, 1)
        mp, mr = statistics.median(tp), statistics.median(tr)
        # variable-base products per equation: prove (m + n)(cx + cy); rerandomise (m + 2n) cx + (n + 2m) cy
        ops = ((m + 2 * n) * 2 + (n + 2 * m) * 2) / ((m + n) * 4)
        doc["workloads"][name] = {
            "count": count, "m": m, "n": n, "shared_commitments": shared,
            "commit_prove_ms": [round(t * 1e3, 3) for t in tp], "rerandomize_ms": [round(t * 1e3, 3) for t in tr],
            "commit_prove_median_ms": round(mp * 1e3, 3), "rerandomize_median_ms": round(mr * 1e3, 3),
            "commit_prove_per_s": round(count / mp, 1), "rerandomize_per_s": round(count / mr, 1),
            "time_ratio_rerandomize_over_commit_prove": round(mr / mp, 3),
            "msm_product_ratio_rerandomize_over_prove": round(ops, 3),
            "kernels_rerandomize": profiled(eng, rr_leg), "kernels_commit_prove": profiled(eng, prove_leg),
        }
        print(name, json.dumps({k: v for k, v in doc["workloads"][name].items() if not k.startswith("kernels")}), flush=True)
    eng.close()
    text = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
