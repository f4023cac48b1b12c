#!/usr/bin/env python3
"""Randomised per-proof verification (gs_verify_each_rand_dev) against the two ways the engine had to get per-proof
answers for a batch with bad proofs, on C5: 65,536 independent 4 x 4 PPE proofs, 1 % tampered (bench.py's workload:
build_workload, pi[0] <-> pi[1] swapped in every 100th proof), one GPU, inputs resident in HBM.

    exact   gs_verify_batch_dev (four ComT entries, four final exponentiations per proof)
    each    gs_verify_each_rand_dev (one folded pairing product and one final exponentiation per proof)
    today   api.verify_batch(randomized=True) on device buffers: gs_verify_batch_rand_dev, which rejects the batch, then the
            exact gs_verify_batch_dev

The three legs run in a fixed interleaved order (exact, each, today) for --runs rounds of --steps calls each; every
round is timed with CUDA events on the engine's stream.  Afterwards one profiled call of each of exact / each gives the
per-kernel CUDA-event times (gs_profile_enable / gs_profile_read), and the verdict bitmaps are compared with each other
and with the tamper mask.  The card's name, power limit and clocks are read in the same run; no device setting is
changed.  Writes one JSON document.

    python tools/bench_each_rand.py [--proofs 65536] [--runs 5] [--steps 2] [--out each_rand.json]
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


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power, clk, clk_max = [x.strip() for x in q.split(",")]
        return {"gpu": name, "power_limit": power, "sm_clock": clk, "max_sm_clock": clk_max}
    except Exception as ex:  # noqa: BLE001
        return {"gpu": "unknown", "error": str(ex)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proofs", type=int, default=65536)
    ap.add_argument("--distinct", type=int, default=0, help="distinct proved instances (0 = every proof distinct)")
    ap.add_argument("--runs", type=int, default=5)
    ap.add_argument("--steps", type=int, default=2, help="calls per leg and run")
    ap.add_argument("--out", default="")
    a = ap.parse_args()
    import numpy as np
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_each_rand.py needs a CUDA device: the product has no CPU fallback")
    import bench
    import groth_sahai_rs_b200 as gsb
    eng = gsb.Engine(0)
    P, m, n = a.proofs, bench.M_VARS, bench.N_VARS
    t0 = time.perf_counter()
    arrays, expected, _ = bench.build_workload(eng, a.distinct or P, P)
    build_s = time.perf_counter() - t0
    stream = torch.cuda.ExternalStream(eng.stream)
    dev = [torch.from_numpy(x).cuda() for x in arrays]
    ptrs = [t.data_ptr() for t in dev]
    ok_exact = torch.zeros(P, dtype=torch.uint8, device="cuda")
    ok_each = torch.zeros(P, dtype=torch.uint8, device="cuda")
    ok_today = torch.zeros(P, dtype=torch.uint8, device="cuda")
    ok1 = torch.zeros(4, dtype=torch.uint8, device="cuda")
    rho = np.random.default_rng(5).bytes(8 * (2 * P + 1))   # seeded weights: the same inputs on every run
    torch.cuda.synchronize()

    def exact():
        eng.verify_batch_dev(0, P, m, n, ptrs, ok_exact.data_ptr())

    def each():
        eng.verify_each_rand_dev(0, P, m, n, ptrs, ok_each.data_ptr(), rho=rho)

    def today():  # what api.verify_batch(randomized=True) does: the batch check, then (rejected) the exact path
        eng.verify_batch_rand_dev(0, P, m, n, ptrs, ok1.data_ptr(), rho=rho)
        stream.synchronize()
        if int(ok1[0].item()) == 1:
            ok_today.fill_(1)
            torch.cuda.synchronize()
        else:
            eng.verify_batch_dev(0, P, m, n, ptrs, ok_today.data_ptr())

    legs = {"exact": exact, "each": each, "today": today}

    def timed(fn, k):
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(k):
            fn()
        e1.record(stream)
        stream.synchronize()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / k

    info = card()
    for fn in legs.values():  # warm-up: module loads, pool growth, the CRS lines
        fn()
    torch.cuda.synchronize()
    times = {k: [] for k in legs}
    for _ in range(a.runs):
        for k, fn in legs.items():
            times[k].append(timed(fn, a.steps))
    info_after = card()
    v_exact, v_each, v_today = (x.cpu().numpy() for x in (ok_exact, ok_each, ok_today))
    prof = {}
    for k in ("exact", "each"):
        eng.profile_enable(True)
        legs[k]()
        torch.cuda.synchronize()
        p = eng.profile_read()
        eng.profile_enable(False)
        prof[k] = {name.split("<")[0]: [c, round(ms, 3)] for name, (c, ms) in sorted(p.items(), key=lambda kv: -kv[1][1])}
    med = {k: statistics.median(v) for k, v in times.items()}
    out = {
        "workload": "C5: independent 4x4 PPE proofs, 1 % tampered (pi[0] <-> pi[1]), resident in HBM, one GPU",
        "proofs": P, "distinct": a.distinct or P, "build_s": round(build_s, 1), "runs": a.runs, "steps_per_run": a.steps,
        "card": info, "card_after": info_after,
        "ms_per_call": {k: [round(x, 2) for x in v] for k, v in times.items()},
        "ms_median": {k: round(v, 2) for k, v in med.items()},
        "verifies_per_s_median": {k: round(P / (v / 1e3)) for k, v in med.items()},
        "each_over_exact": round(med["exact"] / med["each"], 3),
        "each_over_today": round(med["today"] / med["each"], 3),
        "verdicts": {
            "each_equals_exact": bool((v_each == v_exact).all()),
            "exact_equals_mask": bool((v_exact == expected).all()),
            "today_equals_exact": bool((v_today == v_exact).all()),
            "rejected": int((v_each == 0).sum()), "tampered": int((expected == 0).sum()),
        },
        "prof_ms": prof,
    }
    s = json.dumps(out, indent=1)
    print(s)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(s + "\n")
    eng.close()


if __name__ == "__main__":
    main()
