#!/usr/bin/env python3
"""Rerandomisation of zero-knowledge PPE proofs (gs_zk_ppe_rerandomize_batch) against the zk prover and the plain
rerandomisation of the original PPE, from host buffers, under the hiding CRS of one set of draws:
  C5  65,536 independent 4 x 4 statements, K = 1, every point distinct (throughput)
  C1  one 4 x 4 statement, K = 1 (latency)
  K3  one 4 x 4 statement, K = 3 (latency; each target pair adds one x-variable to PPE' and one linear equation)
Legs, alternating within one process: zk rerandomise, zk prove of the same shape (gs_zk_ppe_prove_batch), and
gs_rerandomize_batch of the original m x n PPE (its own commit + prove made once beforehand).  Inputs are seeded (random
Fr; points = multiples of the CRS generators).  The proofs to rerandomise come from gs_zk_ppe_simulate_batch, so they
verify whatever the random target pairs are; every rerandomised statement is checked with gs_zk_ppe_verify_batch.  Every call
ends in a device synchronise.  After the timed legs, one profiled rerandomise per workload gives the time of
k_fixed_com_add (the linear equations' fixed-base sums) on its own, from CUDA events around each launch.  Card name and
power limit are read in the same run.  Writes one JSON document.

    python tools/bench_zk_rerand.py [--reps 5] [--out profiles/r12_zk_rerand.json]
"""
import argparse
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True

from bench_rerand import card, profiled, rand_fr, timed  # noqa: E402
from bench_zk import workload  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c5", type=int, default=65536)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import groth_sahai_rs_b200 as gsb
    from gsutil import make_crs, crs_bytes, fr_b, g1_b, g2_b
    from simulate_ref import hiding_crs
    crs, (_, _, _, _, t1, t2) = make_crs(7)
    hid = hiding_crs(crs)
    tkey = fr_b(t1) + fr_b(t2)
    eng = gsb.Engine(0)
    eng.crs_load(crs_bytes(hid))
    g1, g2 = g1_b(hid.g1_gen), g2_b(hid.g2_gen)
    doc = {"card": card(), "reps": args.reps, "crs": "hiding", "workloads": {}}
    for name, (count, m, n, K) in {"C5": (args.c5, 4, 4, 1), "C1": (1, 4, 4, 1), "K3": (1, 4, 4, 3)}.items():
        w = workload(eng, g1, g2, count, m, n, K, seed=17)
        stmt = (w["A"], w["B"], w["G"], w["P"], w["Q"])
        rnd = (w["xr"], w["yr"], w["Tr"], w["Lr"])
        fresh = (rand_fr(count * (m + K) * 2, 31), rand_fr(count * n * 2, 32), rand_fr(count * 4, 33), rand_fr(count * K * 2, 34))
        proof = eng.zk_ppe_simulate_batch(count, m, n, K, *stmt, *rnd, tkey)   # verifies for any target pairs
        xc, yc = eng.batch_commit_g1(w["X"], w["xr0"]), eng.batch_commit_g2(w["Y"], w["yr"])
        plain = (xc, yc, *eng.prove_batch(0, count, m, n, w["A"], w["B"], w["G"], w["X"], w["Y"], w["xr0"], w["yr"], w["Tr"]))
        res = {}

        def zk_rerandomize(): res["rr"] = eng.zk_ppe_rerandomize_batch(count, m, n, K, w["A"], w["B"], w["G"], w["Q"], *proof, *fresh)
        def zk_prove(): eng.zk_ppe_prove_batch(count, m, n, K, *stmt, w["X"], w["Y"], *rnd)
        def plain_rerandomize():
            eng.rerandomize_batch(0, count, m, n, w["A"], w["B"], w["G"], *plain, fresh[0][:count * m * 2 * 32], fresh[1], fresh[2])

        legs = {"zk_rerandomize": zk_rerandomize, "zk_prove": zk_prove, "plain_rerandomize": plain_rerandomize}
        for f in legs.values():   # warm-up (module load, fixed-base tables)
            f()
        ts = {k: [] for k in legs}
        reps = args.reps if count > 1 else 20 * args.reps
        for _ in range(reps):
            for k, f in legs.items():
                ts[k] += timed(f, 1)
        med = {k: statistics.median(v) for k, v in ts.items()}
        ok = eng.zk_ppe_verify_batch(count, m, n, K, *stmt, *res["rr"])
        prof = profiled(eng, zk_rerandomize)
        doc["workloads"][name] = {
            "count": count, "m": m, "n": n, "K": K,
            **{f"{k}_ms": [round(t * 1e3, 3) for t in v] for k, v in ts.items()},
            **{f"{k}_median_ms": round(v * 1e3, 3) for k, v in med.items()},
            **{f"{k}_per_s": round(count / v, 1) for k, v in med.items()},
            "ratio_zk_rerandomize_over_zk_prove": round(med["zk_rerandomize"] / med["zk_prove"], 3),
            "ratio_zk_rerandomize_over_plain_rerandomize": round(med["zk_rerandomize"] / med["plain_rerandomize"], 3),
            "k_fixed_com_add_ms": {k: v for k, v in prof.items() if "k_fixed_com_add" in k},
            "profiled_kernels_ms": prof,
            "rerandomised_all_verify": ok == b"\x01" * count,
        }
        print(name, json.dumps({k: v for k, v in doc["workloads"][name].items()
                                if not k.endswith("_ms") or k.endswith("median_ms") or k == "k_fixed_com_add_ms"}), flush=True)
    eng.close()
    text = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
