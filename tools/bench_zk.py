#!/usr/bin/env python3
"""Zero-knowledge proofs of PPEs with targets given as pairs (gs_zk_ppe_*_batch) against the plain PPE paths, from host
buffers, under the hiding CRS of one set of draws:
  C5  65,536 independent 4 x 4 statements, K = 1, every point distinct (throughput)
  C1  one 4 x 4 statement, K = 1 (latency)
  K3  one 4 x 4 statement, K = 3 (latency; each target pair adds one x-variable and one MSMEG1 proof)
Legs, alternating within one process: zk prove against commit + prove of the original PPE (gs_batch_commit_g1 / _g2 +
gs_prove_batch), zk simulate, and zk verify against gs_verify_batch of the original PPE.  Inputs are seeded (random Fr;
points = multiples of the CRS generators); the statements need not hold to be timed.  Every call ends in a device
synchronise (the host-buffer entry points return after their copies back).  The simulated proofs are checked with
gs_zk_ppe_verify_batch (they verify for any target pairs).  Card name and power limit are read in the same run.  Writes
one JSON document.

    python tools/bench_zk.py [--reps 5] [--out profiles/r08_zk.json]
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

from bench_rerand import card, points, rand_fr, timed  # noqa: E402


def workload(eng, g1, g2, count, m, n, K, seed):
    from gsutil import fp12_b, FP12_ONE
    w = dict(count=count, m=m, n=n, K=K)
    pt1 = lambda k, s: points(eng, g1, k, s, False, pool=k)
    pt2 = lambda k, s: points(eng, g2, k, s, True, pool=k)
    w["A"], w["B"], w["G"] = pt1(count * n, seed), pt2(count * m, seed + 1), rand_fr(count * m * n, seed + 2)
    w["P"], w["Q"] = pt1(count * K, seed + 3), pt2(count * K, seed + 4)
    w["X"], w["Y"] = pt1(count * m, seed + 5), pt2(count * n, seed + 6)
    w["xr"], w["yr"] = rand_fr(count * (m + K) * 2, seed + 7), rand_fr(count * n * 2, seed + 8)
    w["Tr"], w["Lr"] = rand_fr(count * 4, seed + 9), rand_fr(count * K * 2, seed + 10)
    w["xr0"] = rand_fr(count * m * 2, seed + 11)   # the plain PPE's R (m rows)
    w["T1"] = fp12_b(FP12_ONE) * count             # the plain PPE's target (its verdict is not the point)
    return w


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
        res = {}

        def plain_prove():
            xc, yc = eng.batch_commit_g1(w["X"], w["xr0"]), eng.batch_commit_g2(w["Y"], w["yr"])
            res["plain"] = (xc, yc, *eng.prove_batch(0, count, m, n, w["A"], w["B"], w["G"], w["X"], w["Y"], w["xr0"], w["yr"], w["Tr"]))

        def zk_prove(): res["zk"] = eng.zk_ppe_prove_batch(count, m, n, K, *stmt, w["X"], w["Y"], *rnd)
        def zk_simulate(): res["sim"] = eng.zk_ppe_simulate_batch(count, m, n, K, *stmt, *rnd, tkey)
        def plain_verify(): eng.verify_batch(0, count, m, n, w["A"], w["B"], w["G"], w["T1"], *res["plain"])
        def zk_verify(): res["ok"] = eng.zk_ppe_verify_batch(count, m, n, K, *stmt, *res["sim"])

        legs = {"plain_commit_prove": plain_prove, "zk_prove": zk_prove, "zk_simulate": zk_simulate,
                "plain_verify": plain_verify, "zk_verify": zk_verify}
        for f in legs.values():   # warm-up (module load, fixed-base tables, stored lines), in dependency order
            f()
        ts = {k: [] for k in legs}
        reps = args.reps if count > 1 else 20 * args.reps
        for _ in range(reps):
            for k, f in legs.items():
                ts[k] += timed(f, 1)
        med = {k: statistics.median(v) for k, v in ts.items()}
        doc["workloads"][name] = {
            "count": count, "m": m, "n": n, "K": K,
            **{f"{k}_ms": [round(t * 1e3, 3) for t in v] for k, v in ts.items()},
            **{f"{k}_median_ms": round(v * 1e3, 3) for k, v in med.items()},
            **{f"{k}_per_s": round(count / v, 1) for k, v in med.items()},
            "ratio_zk_prove_over_plain": round(med["zk_prove"] / med["plain_commit_prove"], 3),
            "ratio_zk_simulate_over_plain_prove": round(med["zk_simulate"] / med["plain_commit_prove"], 3),
            "ratio_zk_verify_over_plain": round(med["zk_verify"] / med["plain_verify"], 3),
            "simulated_all_verify": res["ok"] == b"\x01" * count,
        }
        print(name, json.dumps({k: v for k, v in doc["workloads"][name].items() if not k.endswith("_ms")}), flush=True)
    eng.close()
    text = json.dumps(doc, indent=1)
    if args.out:
        with open(args.out, "w") as f:
            f.write(text + "\n")
    else:
        print(text)


if __name__ == "__main__":
    main()
