#!/usr/bin/env python3
"""Zero-knowledge simulation (gs_simulate_batch) against commit + prove of the same shape, from host buffers, under the
hiding CRS of one set of draws: C5 (65,536 independent 4 x 4 statements, PPE with target 1 and MSMEG1 with random
targets), C4 (1,024 PPE equations over one set of 64 x 64 commitments) and C3 (one 1024 x 1024 PPE, latency).  Inputs are
seeded (random Fr; points = multiples of the CRS generators, a pool of distinct points tiled over the batch).  The two legs
alternate within one process; every call ends in a device synchronise (the host-buffer entry points return after their
copies back).  After the timed reps, one profiled call of each leg gives the per-kernel CUDA-event times.  The first and
the last simulated proof of every workload are compared byte for byte with the C oracle's commit + prove of the augmented
equation, and every output is checked with gs_verify_batch.  Card name and power limit are read in the same run.  Writes
one JSON document.

    python tools/bench_simulate.py [--reps 5] [--out simulate.json]
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

from bench_rerand import card, points, profiled, rand_fr, timed  # noqa: E402

FR, G1, COM1, COM2 = 32, 96, 192, 384


def g1_neg(pts: bytes) -> bytes:
    """-P for affine G1 points in the ABI encoding (y -> p - y on the Montgomery limbs; the identity stays)"""
    from oracle.bls12_381 import P
    out = bytearray()
    for i in range(0, len(pts), G1):
        x, y = pts[i:i + 48], int.from_bytes(pts[i + 48:i + 96], "little")
        out += x + (((P - y) % P) if y else 0).to_bytes(48, "little")
    return bytes(out)


def workload(eng, g1, g2, ty, count, m, n, shared, seed):
    """inputs of one type (0: PPE, target 1; 1: MSMEG1, random targets) for both legs; the witnesses of commit + prove
    need not satisfy the statement to be timed"""
    from gsutil import fp12_b, FP12_ONE
    reps = 1 if shared else count
    cx, cy = 2, (2 if ty == 0 else 1)
    w = dict(ty=ty, count=count, m=m, n=n, shared=shared)
    w["A"] = points(eng, g1, count * n, seed, False)
    w["B"] = points(eng, g2, count * m, seed + 1, True) if ty == 0 else rand_fr(count * m, seed + 1)
    w["G"] = rand_fr(count * m * n, seed + 2)
    w["T"] = fp12_b(FP12_ONE) * count if ty == 0 else points(eng, g1, count, seed + 3, False)
    w["X"] = points(eng, g1, reps * m, seed + 4, False)
    w["Y"] = points(eng, g2, reps * n, seed + 5, True) if ty == 0 else rand_fr(reps * n, seed + 5)
    w["xr"], w["yr"] = rand_fr(reps * m * cx, seed + 6), rand_fr(reps * n * cy, seed + 7)
    w["Tr"] = rand_fr(count * cx * cy, seed + 8)
    return w


def commit_prove(eng, w):
    xc = eng.batch_commit_g1(w["X"], w["xr"])
    yc = eng.batch_commit_g2(w["Y"], w["yr"]) if w["ty"] == 0 else eng.batch_commit_scalar_b2(w["Y"], w["yr"])
    args = (w["A"], w["B"], w["G"], w["X"], w["Y"], w["xr"], w["yr"], w["Tr"])
    if w["count"] == 1:
        return xc, yc, *eng.prove(w["ty"], w["m"], w["n"], *args)
    return xc, yc, *eng.prove_batch(w["ty"], w["count"], w["m"], w["n"], *args, shared_vars=w["shared"])


def simulate(eng, w, tkey):
    args = (w["A"], w["B"], w["G"], w["T"], w["xr"], w["yr"], w["Tr"], tkey)
    if w["count"] == 1:
        return eng.simulate(w["ty"], w["m"], w["n"], *args)
    return eng.simulate_batch(w["ty"], w["count"], w["m"], w["n"], *args, shared_coms=w["shared"])


def oracle_check(w, out, crsb, t1, t2, i):
    """proof i of the simulated batch against the C oracle's commit + prove of its augmented equation"""
    from oracle import cbaseline as cb
    from gsutil import fr_b
    ty, m, n = w["ty"], w["m"], w["n"]
    cx, cy = 2, (2 if ty == 0 else 1)
    k = 0 if w["shared"] else i
    A, B = w["A"][i * n * G1:(i + 1) * n * G1], w["B"][i * m * cb.y_size(ty):(i + 1) * m * cb.y_size(ty)]
    G = w["G"][i * m * n * FR:(i + 1) * m * n * FR]
    xr, yr = w["xr"][k * m * cx * FR:(k + 1) * m * cx * FR], w["yr"][k * n * cy * FR:(k + 1) * n * cy * FR]
    nn = n
    if ty == 1:   # one more y-variable with randomness [t2], constant -T1, a zero column of Gamma
        A += g1_neg(w["T"][i * G1:(i + 1) * G1])
        G = b"".join(G[r * n * FR:(r + 1) * n * FR] + bytes(FR) for r in range(m))
        yr += fr_b(t2)
        nn += 1
    X, Y = bytes(m * G1), bytes(nn * cb.y_size(ty))
    nt = cb.host_cores()
    want = (cb.commit_x(ty, X, xr, crsb, nt)[:m * COM1], cb.commit_y(ty, Y, yr, crsb, nt)[:n * COM2],
            *cb.prove(ty, m, nn, A, B, G, X, Y, xr, yr, w["Tr"][i * cx * cy * FR:(i + 1) * cx * cy * FR], crsb, nt))
    xc, yc, pi, th = out
    got = (xc[k * m * COM1:(k + 1) * m * COM1], yc[k * n * COM2:(k + 1) * n * COM2], pi[i * cx * COM2:(i + 1) * cx * COM2],
           th[i * cy * COM1:(i + 1) * cy * COM1])
    return got == want


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--c5", type=int, default=65536)
    ap.add_argument("--c4", type=int, default=1024)
    ap.add_argument("--c3", type=int, default=1024)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import groth_sahai_rs_b200 as gsb
    from gsutil import make_crs, crs_bytes, fr_b, g1_b, g2_b
    from simulate_ref import hiding_crs
    crs, (_, _, _, _, t1, t2) = make_crs(7)
    hid = hiding_crs(crs)
    crsb, tkey = crs_bytes(hid), fr_b(t1) + fr_b(t2)
    eng = gsb.Engine(0)
    eng.crs_load(crsb)
    g1, g2 = g1_b(hid.g1_gen), g2_b(hid.g2_gen)
    doc = {"card": card(), "reps": args.reps, "crs": "hiding", "workloads": {}}
    shapes = {"C5_PPE": (0, args.c5, 4, 4, False), "C5_MSMEG1": (1, args.c5, 4, 4, False),
              "C4_PPE": (0, args.c4, 64, 64, True), "C3_PPE": (0, 1, args.c3, args.c3, False)}
    for name, (ty, count, m, n, shared) in shapes.items():
        w = workload(eng, g1, g2, ty, count, m, n, shared, seed=13)
        prove_leg, sim_leg = (lambda: commit_prove(eng, w)), (lambda: simulate(eng, w, tkey))
        prove_leg()
        out = sim_leg()  # warm-up (module load, fixed-base tables at the batch's window size)
        tp, ts = [], []
        for _ in range(args.reps):
            tp += timed(prove_leg, 1)
            ts += timed(sim_leg, 1)
        mp, msim = statistics.median(tp), statistics.median(ts)
        reps = count if shared else 1
        ok = eng.verify_batch(ty, count, m, n, w["A"], w["B"], w["G"], w["T"], out[0] * reps, out[1] * reps, out[2], out[3])
        doc["workloads"][name] = {
            "type": ty, "count": count, "m": m, "n": n, "shared_commitments": shared,
            "commit_prove_ms": [round(t * 1e3, 3) for t in tp], "simulate_ms": [round(t * 1e3, 3) for t in ts],
            "commit_prove_median_ms": round(mp * 1e3, 3), "simulate_median_ms": round(msim * 1e3, 3),
            "commit_prove_per_s": round(count / mp, 1), "simulate_per_s": round(count / msim, 1),
            "time_ratio_simulate_over_commit_prove": round(msim / mp, 3),
            "oracle_sample_equal": all(oracle_check(w, out, crsb, t1, t2, i) for i in sorted({0, count - 1})),
            "verify_batch_all_accept": ok == b"\x01" * count,
            "kernels_simulate": profiled(eng, sim_leg), "kernels_commit_prove": profiled(eng, prove_leg),
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
