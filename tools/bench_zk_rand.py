#!/usr/bin/env python3
"""Randomised per-statement verification of zero-knowledge PPE proofs (gs_zk_ppe_verify_each_rand) against the exact zk
verifier (gs_zk_ppe_verify_batch), from host buffers, under the hiding CRS of one set of draws:
  C5  65,536 independent 4 x 4 statements, K = 1, every point distinct, 1 % tampered (throughput)
  C1  one 4 x 4 statement, K = 1 (latency)
  K3  one 4 x 4 statement, K = 3 (latency)
The statements are bench_zk.py's (seeded random Fr; points = distinct multiples of the CRS generators; targets that need
not hold) with simulated proofs, which verify for any target pairs; in every 100th statement of C5 the two pi elements of
PPE' are exchanged.  The two legs alternate within one process, every call ends in a device synchronise (the host-buffer
entry points return after their copies back), and the medians are reported.  The two verdict bitmaps must be equal, and
equal to the tamper mask.  Card name and power limit are read in the same run.  Writes one JSON document.

    python tools/bench_zk_rand.py [--reps 5] [--out profiles/r11_zk_rand.json]
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

from bench_rerand import card, timed  # noqa: E402
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
    doc = {"card": card(), "reps": args.reps, "crs": "hiding", "tampered": "pi[0] <-> pi[1] of PPE' in every 100th statement",
           "workloads": {}}
    for name, (count, m, n, K) in {"C5": (args.c5, 4, 4, 1), "C1": (1, 4, 4, 1), "K3": (1, 4, 4, 3)}.items():
        w = workload(eng, g1, g2, count, m, n, K, seed=17)
        stmt = (w["A"], w["B"], w["G"], w["P"], w["Q"])
        sim = list(eng.zk_ppe_simulate_batch(count, m, n, K, *stmt, w["xr"], w["yr"], w["Tr"], w["Lr"], tkey))
        pi = bytearray(sim[2])
        bad = range(0, count, 100) if count > 1 else range(0)
        for i in bad:
            pi[i * 768:(i + 1) * 768] = pi[i * 768 + 384:(i + 1) * 768] + pi[i * 768:i * 768 + 384]
        sim[2] = bytes(pi)
        want = bytearray(b"\x01" * count)
        for i in bad:
            want[i] = 0
        res = {}

        def exact(): res["exact"] = eng.zk_ppe_verify_batch(count, m, n, K, *stmt, *sim)
        def each(): res["each"] = eng.zk_ppe_verify_each_rand(count, m, n, K, *stmt, *sim)

        legs = {"exact": exact, "each_rand": each}
        for f in legs.values():   # warm-up (module load, stored lines)
            f()
        ts = {k: [] for k in legs}
        reps = args.reps if count > 1 else 20 * args.reps
        for _ in range(reps):
            for k, f in legs.items():
                ts[k] += timed(f, 1)
        if res["each"] != res["exact"] or res["exact"] != bytes(want):
            raise SystemExit(f"{name}: verdicts differ (each_rand vs exact vs the tamper mask)")
        med = {k: statistics.median(v) for k, v in ts.items()}
        doc["workloads"][name] = {
            "count": count, "m": m, "n": n, "K": K, "tampered": len(bad),
            **{f"{k}_ms": [round(t * 1e3, 3) for t in v] for k, v in ts.items()},
            **{f"{k}_median_ms": round(v * 1e3, 3) for k, v in med.items()},
            **{f"{k}_per_s": round(count / v, 1) for k, v in med.items()},
            "speedup_each_rand_over_exact": round(med["exact"] / med["each_rand"], 3),
            "verdicts_equal": True,
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
