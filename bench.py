#!/usr/bin/env python3
"""bench.py -- headline benchmark of the Groth-Sahai hot path on B200.

Headline workload (BASELINE.json configs[4], the one `metric` = "pairings/sec and PPE verifies/sec" is quoted
on): batch verification of 65,536 independent 4x4 PPE proofs (m = n = 4 variables, dense random Gamma, every
instance distinct, 1 % tampered) SHARDED ACROSS THE N GPUS (strong scaling: `--proofs` is the whole job, every
rank verifies a contiguous block of proofs/N, verdict bytes are all-gathered over NCCL).  One step = one pass of
Verifiable::verify over the whole batch.  Witnesses, commitments and proofs come from this engine's own
commit / prove path (byte-checked against the reference-order CPU restatement in tests/test_gpu_bigparity.py);
inside the bench a sample of the batch -- honest and tampered -- is re-verified by the C oracle outside the timed
region (`parity_sample`).

The same line carries the other multi-GPU configs of BASELINE.json as sub-records, each with its own per-kernel
times and the thing that limits it:
  c5_weak         (N > 1)  65,536 proofs PER GPU, the trivially parallel case
  c3_sharded      one PPE with m = n = 1024 and a dense Gamma, verify split by slot over the N GPUs (configs[2])
  c4_by_equation  4 x 256 equations over shared 64-variable witness sets: commit split by variable, prove and
                  verify split by equation over the N GPUs (configs[3])

    python bench.py [--gpus N] [--steps K] [--warmup W] [--proofs P] [--skip c3,c4,weak] [--impl reference]
                    [--dump-outputs DIR]

--dump-outputs DIR writes what the timed C5 path returned in its last step as DIR/<name>.npy (float32): the per-proof
verdicts of gs_verify_batch_dev and the one verdict of gs_verify_batch_rand_dev.  Inputs are seeded, so two builds run
with the same arguments can be compared output for output.

Prints ONE JSON line (see the task contract): value = verifies/s with inputs resident in HBM, e2e = the same
through the C ABI with host buffers (H2D + D2H inside the timed region), roofline = integer-multiply roofline of
the dominant kernel (measured live with CUDA events), cpu_baseline = the oracle's C restatement of the reference
algorithm timed on the host cores.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True          # the tree may be read-only: leave no __pycache__ behind
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

M_VARS = N_VARS = 4
# ---- algorithmic work model (Fp Montgomery products "M"; 1 M = 600 IMAD-equivalents, SURVEY.md §8d) ----
IMAD_PER_M = 600
M_SQR12, M_LINE, M_014 = 36, 4, 39           # Fp12 squaring, line evaluation at P, sparse product (tower formulas)
M_G2_DBL, M_G2_ADD = 21, 37                  # one doubling / addition step of the projective G2 line walk
M_FE = 8300                                  # final exponentiation (easy ~750 + 5 exp-by-x + products)
M_G1_DBL, M_G1_MADD, M_FP_INV = 7, 11, 490
MILLER_WAVE = 2368                           # proofs per wave of k_miller4 (2 groups x 148 SMs x 32 accumulators / 4 entries)


def work_model(m, n):
    """Algorithmic M per verified 4x4-shaped PPE proof, per kernel: the best sequential (tower / Karatsuba)
    operation counts of SURVEY.md §8d for what each kernel computes -- NOT the instructions it executes
    (k_miller4's unit-coefficient lines need fewer products than the 39 M sparse product charged here, which is
    why its model fraction can exceed its pipe utilisation; `pipe_util` reports the executed instructions)."""
    cx = cy = 2
    pairs = 2 * (n + cx + cy) + 2 * (n + m + cx + cy)            # Miller pairs over the 4 ComT entries
    g2_points = 2 * n + m + 2 * cx                                 # G2 coordinates walked per proof (the CRS points
    fixed_pairs = 2 * 2 * cy                                       # v_1, v_2 have their lines stored at key load)
    return {
        "k_miller4": 4 * 62 * M_SQR12 + pairs * 68 * M_014,
        "k_g2_prepare4": g2_points * (63 * M_G2_DBL + 5 * M_G2_ADD) + (pairs - fixed_pairs) * 68 * M_LINE,
        "k_fixed_tiles": fixed_pairs * 68 * M_LINE,
        "k_final_exp3": 4 * M_FE,
        # Straus over the GLV halves, signed 4-bit windows: 32 windows x (4 shared doublings + one addition per
        # half-scalar, 15/16 non-zero)
        "k_vmsm_partial": 2 * n * (128 * M_G1_DBL + 32 * 2 * m * (15 / 16) * M_G1_MADD),
        "k_vmsm_tables": 2 * m * (M_G1_DBL + 6 * M_G1_MADD + 8 * 9),
        "k_vmsm_reduce": 2 * n * (M_G1_MADD + 9),
        "pairs": pairs,
    }


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region.  The sampler process is started before the
    warm-up (nvidia-smi needs ~0.5 s to come up, longer than a short timed region on 8 GPUs) and only the samples that
    arrive between begin() and end() are kept."""

    def __init__(self, index):
        self.index = index
        self.rows = []
        self.proc = None
        self.t0 = self.t1 = None

    def begin(self):
        self.t0 = time.time()

    def end(self):
        self.t1 = time.time()

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "200"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        t0, t1 = self.t0 or 0.0, self.t1 or float("inf")
        inside = [r for ts, r in self.rows if t0 <= ts <= t1 + 0.2]     # (a sample is printed up to one period after it is taken)
        note = None
        if not inside and self.rows:                                    # region shorter than one sampling period
            inside = [min(self.rows, key=lambda tr: abs(tr[0] - t1))[1]]
            note = "timed region shorter than the 200 ms sampling period: nearest sample"
        rows = inside
        sm = sorted(int(float(r[0])) for r in rows if r and r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in rows)]
        mx = [int(float(r[1])) for r in rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        out = {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
               "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": reasons}
        if note:
            out["note"] = note
        return out


# ---------------------------------------------------------------- synthetic workload (C5)
def build_workload(eng, distinct, proofs, seed=5):
    """`distinct` satisfied 4x4 PPE instances (all different: own witnesses, constants, Gamma, randomness), committed
    and proved by the engine in batched calls, tiled to `proofs` when distinct < proofs; 1 % tampered.
    Returns (list of 8 numpy uint8 arrays [proofs, bytes] in gs_verify_batch order, expected verdict array)."""
    import numpy as np
    from gsutil import SeededRng, make_crs, crs_bytes, fr_b, g1_b, g2_b
    from oracle.bls12_381 import R
    crs, _ = make_crs(seed)
    eng.crs_load(crs_bytes(crs))
    rng = SeededRng(seed + 1)
    m, n = M_VARS, N_VARS
    g1b, g2b = g1_b(crs.g1_gen), g2_b(crs.g2_gen)
    D = distinct
    sc = lambda k: [rng.fr() for _ in range(k)]
    xs, ys, a, b = sc(D * m), sc(D * n), sc(D * n), sc(D * m)
    gam = sc(D * m * n)
    frs = lambda ks: b"".join(fr_b(k) for k in ks)

    def g1_multiples(ks):   # k * g1 via the Mat kernel: (len x 1 Fr) * (1 x 1 Com1), in slabs the kernel accepts
        out = []
        for o in range(0, len(ks), 1 << 18):
            part = ks[o:o + (1 << 18)]
            r = eng.com1_matmul(len(part), 1, 1, frs(part), g1b + g1b)
            out.append(np.frombuffer(r, dtype=np.uint8).reshape(len(part), 192)[:, :96])
        return np.concatenate(out)

    def g2_multiples(ks):
        out = []
        for o in range(0, len(ks), 1 << 18):
            part = ks[o:o + (1 << 18)]
            r = eng.com2_matmul(len(part), 1, 1, frs(part), g2b + g2b)
            out.append(np.frombuffer(r, dtype=np.uint8).reshape(len(part), 384)[:, :192])
        return np.concatenate(out)

    X, Y, A, B = g1_multiples(xs), g2_multiples(ys), g1_multiples(a), g2_multiples(b)
    # target = gt^val with val the equation "in the exponent": e(val * g1, g2)
    vals = []
    for d in range(D):
        xd, yd = xs[d * m:(d + 1) * m], ys[d * n:(d + 1) * n]
        gd = gam[d * m * n:(d + 1) * m * n]
        v = sum(a[d * n + j] * yd[j] for j in range(n)) + sum(xd[i] * b[d * m + i] for i in range(m))
        v += sum(gd[i * n + j] * xd[i] * yd[j] for i in range(m) for j in range(n))
        vals.append(v % R)
    tg = eng.pairing(np.ascontiguousarray(g1_multiples(vals)).tobytes(), g2b * D)
    xr, yr, Tr = frs(sc(D * 2 * m)), frs(sc(D * 2 * n)), frs(sc(D * 4))
    Xb, Yb = np.ascontiguousarray(X).tobytes(), np.ascontiguousarray(Y).tobytes()
    Ab, Bb, Gb = np.ascontiguousarray(A).tobytes(), np.ascontiguousarray(B).tobytes(), frs(gam)
    xc = eng.batch_commit_g1(Xb, xr)                       # D*m variables in one call
    yc = eng.batch_commit_g2(Yb, yr)
    crs2, _ = make_crs(seed)
    eng.crs_load(crs_bytes(crs2))                          # (a big commit batch may have switched the fixed-base tables)
    pi, th = eng.prove_batch(0, D, m, n, Ab, Bb, Gb, Xb, Yb, xr, yr, Tr, shared_vars=False)
    rows = lambda bts, w: np.frombuffer(bts, dtype=np.uint8).reshape(D, w)
    base = [rows(Ab, n * 96), rows(Bb, m * 192), rows(Gb, m * n * 32), rows(tg, 576), rows(xc, m * 192), rows(yc, n * 384),
            rows(pi, 768), rows(th, 384)]
    if D == proofs:
        arrays = [np.array(bs) for bs in base]
    else:
        idx = (np.arange(proofs, dtype=np.int64) * 7919 + 13) % D
        arrays = [np.ascontiguousarray(bs[idx]) for bs in base]
    expected = np.ones(proofs, dtype=np.uint8)
    bad = np.arange(37, proofs, 100)                        # 1 % tampered: swap pi[0] <-> pi[1]
    pi_arr = arrays[6]
    tmp = pi_arr[bad, :384].copy()
    pi_arr[bad, :384] = pi_arr[bad, 384:]
    pi_arr[bad, 384:] = tmp
    expected[bad] = 0
    return arrays, expected, crs_bytes(crs)


def parity_sample(arrays, got, crsb, m, n):
    """A sample of the batch -- honest and tampered -- re-verified by the C restatement of the reference's
    PPE::verify (oracle/gs_oracle.c, reference evaluation order), OUTSIDE the timed region."""
    import numpy as np
    from oracle import cbaseline as cb
    P = len(got)
    idx = sorted(set([i for i in range(0, min(P, 12))] + [i for i in range(37, P, 100)][:4] + [P - 1]))
    sub = [np.ascontiguousarray(a[idx]).tobytes() for a in arrays]
    ref = cb.verify_batch(0, len(idx), m, n, sub, crsb, cb.host_cores())
    mine = bytes(int(got[i]) for i in idx)
    return {"checked": len(idx), "tampered_in_sample": sum(1 for x in ref if x == 0), "agree": ref == mine,
            "checker": "oracle/gs_oracle.c gsref_verify_batch (reference order: 20 final exps, Gamma*d on G2)"}


# ---------------------------------------------------------------- reference arm (CPU)
def run_reference(args):
    """The reference's algorithm on the host cores: oracle C port (oracle/_ref does not exist: no Rust
    toolchain here, SURVEY.md §8c), all host threads, a bounded sample of the same workload per step."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oracle import cbaseline
    res = cbaseline.time_ppe_verify(m=M_VARS, n=N_VARS, sample=args.ref_sample, steps=args.steps, warmup=args.warmup)
    line = {
        "metric": "ppe_verifies_per_sec", "value": res["verifies_per_sec"], "unit": "verifies/s", "impl": "reference",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u64-montgomery", "data": "synthetic",
        "config": {"workload": "C5: batch verification of independent 4x4 PPE proofs (BASELINE.json configs[4]), "
                               "Verifiable::verify, reference algorithm on the host cores",
                   "m": M_VARS, "n": N_VARS, "proofs_per_step": res["sample"],
                   "note": "throughput-normalised: each CPU step verifies a bounded sample of the same 4x4 shape "
                           "(the GPU arm's 65,536 would take minutes per step on the host)"},
        "pairings_per_sec": res["verifies_per_sec"] * res["pairings_per_verify"],
        "cpu_baseline": {"value": res["verifies_per_sec"], "unit": "verifies/s", "cores": res["cores"], "kind": res["kind"],
                         "sample": res["sample_desc"]},
        "e2e": {"value": res["verifies_per_sec"], "unit": "verifies/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line))


# ---------------------------------------------------------------- helpers shared by the GPU legs
class Ranks:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local = int(os.environ.get("LOCAL_RANK", "0"))
        self.dist = None
        self.dev = f"cuda:{self.local}"

    def init(self):
        torch = self.torch
        if not torch.cuda.is_available():
            raise SystemExit("bench.py needs a CUDA device: the product has no CPU fallback")
        torch.cuda.set_device(self.local)
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=torch.device("cuda", self.local))
            self.dist = dist

    def barrier(self, stream=None):
        if self.world > 1:
            self.dist.barrier()
        if stream is not None:
            stream.synchronize()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        if self.world == 1:
            return float(x)
        t = self.torch.tensor([float(x)], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def wall_ms(self, fn, steps, warmup=1):
        """Wall clock around `steps` synchronous calls, bracketed by barriers, max over ranks (e2e figures)."""
        for _ in range(warmup):
            fn()
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            fn()
        self.barrier()
        return self.max_over_ranks((time.perf_counter() - t0) * 1e3 / steps)


def profiled(eng, fn):
    eng.profile_enable(True)
    fn()
    prof = eng.profile_read()
    eng.profile_enable(False)
    return {k: [v[0], round(v[1], 3)] for k, v in prof.items()}


def top_kernels(prof, k=3):
    tot = sum(v[1] for v in prof.values()) or 1.0
    top = sorted(prof.items(), key=lambda kv: -kv[1][1])[:k]
    return ", ".join(f"{name} {ms:.1f} ms ({100 * ms / tot:.0f} %)" for name, (_, ms) in top)


# ---------------------------------------------------------------- C5 (headline and the weak-scaling companion)
def bench_c5(R_, eng, P, distinct, steps, warmup, full):
    """P proofs on THIS rank.  Returns a dict with value-leg ms, e2e ms and (full) the per-kernel / roofline data."""
    import numpy as np
    torch = R_.torch
    m, n = M_VARS, N_VARS
    t0 = time.perf_counter()
    arrays, expected, crsb = build_workload(eng, distinct or P, P, seed=5 + R_.rank)
    build_s = time.perf_counter() - t0
    stream = torch.cuda.ExternalStream(eng.stream, device=R_.local)
    host = [torch.from_numpy(a).pin_memory() for a in arrays]         # pinned host copies (e2e leg)
    dev = [h.to(R_.dev) for h in host]                                 # resident in HBM (value leg)
    ok_dev = torch.zeros(P, dtype=torch.uint8, device=R_.dev)
    gathered = [torch.zeros_like(ok_dev) for _ in range(R_.world)] if R_.world > 1 else None
    torch.cuda.synchronize()

    def step_dev():
        eng.verify_batch_dev(0, P, m, n, [t.data_ptr() for t in dev], ok_dev.data_ptr())
        if R_.world > 1:                                                # verdict bytes over NCCL (SURVEY.md §8e)
            torch.cuda.current_stream().wait_stream(stream)
            R_.dist.all_gather(gathered, ok_dev)

    def timed(fn, k):
        """K steps bracketed by barrier + synchronize; device time from CUDA events on the engine's stream."""
        R_.barrier(stream)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(k):
            fn()
        if R_.world > 1:
            stream.wait_stream(torch.cuda.current_stream())
        e1.record(stream)
        R_.barrier(stream)
        return R_.max_over_ranks(e0.elapsed_time(e1))

    sampler = ClockSampler(R_.local)
    sampler.start()
    for _ in range(max(1, warmup)):
        step_dev()
    R_.barrier(stream)
    got = ok_dev.cpu().numpy()
    if not (got == expected).all():
        sampler.stop()
        raise SystemExit(f"verdict mismatch on rank {R_.rank}: {(got != expected).sum()} wrong of {P}")
    out = {"build_s": round(build_s, 1), "distinct": distinct or P}
    l0 = eng.launch_count
    sampler.begin()
    ms_total = timed(step_dev, steps)
    sampler.end()
    out["verdicts"] = (torch.cat(gathered) if R_.world > 1 else ok_dev).cpu().numpy()    # the last timed step's answer
    out["launches"] = eng.launch_count - l0
    out["clocks"] = sampler.stop()
    out["ms_per_step"] = ms_total / steps
    if not full:
        return out
    out["parity_sample"] = parity_sample(arrays, got, crsb, m, n) if R_.rank == 0 else None
    # ---- per-kernel device time (CUDA events inside the library, same stream), one extra profiled step
    eng.profile_enable(True)
    step_dev()
    out["prof"] = {k.split("<")[0]: v for k, v in eng.profile_read().items()}      # k_g2_prepare4<4> -> k_g2_prepare4
    eng.profile_enable(False)
    # ---- e2e: the public C-ABI call with HOST buffers (pinned), H2D and D2H inside the timed region
    ok_host = torch.zeros(P, dtype=torch.uint8).pin_memory()
    lib, vp = eng.lib, ctypes.c_void_p

    def step_e2e():
        rc = lib.gs_verify_batch(eng.h, 0, P, m, n, *[vp(h.data_ptr()) for h in host], vp(ok_host.data_ptr()))
        if rc != 0:
            raise SystemExit(lib.gs_last_error(eng.h).decode())

    step_e2e()
    if not (ok_host.numpy() == expected).all():
        raise SystemExit("e2e verdict mismatch")
    out["e2e_ms"] = R_.wall_ms(step_e2e, steps, warmup=0)
    out["h2d_bytes"] = int(sum(a.nbytes for a in arrays))
    out["d2h_bytes"] = P
    # ---- opt-in randomised batch verification (gs_verify_batch_rand, SURVEY.md 8f.4): ONE verdict per call.  Timed on the
    # honest proofs of this shard (a batch with a bad proof is rejected and then goes through the exact path above).
    try:
        honest = torch.from_numpy(np.flatnonzero(expected == 1)).to(R_.dev)
        Ph = int(honest.numel())
        devh = [t.index_select(0, honest).contiguous() for t in dev]
        ok1 = torch.zeros(4, dtype=torch.uint8, device=R_.dev)
        rho = np.random.default_rng(5 + R_.rank).bytes(8 * (2 * P + 1))   # seeded weights: the same inputs on every run

        def step_rand():
            eng.verify_batch_rand_dev(0, Ph, m, n, [t.data_ptr() for t in devh], ok1.data_ptr(), rho=rho[:8 * (2 * Ph + 1)])

        eng.verify_batch_rand_dev(0, P, m, n, [t.data_ptr() for t in dev], ok1.data_ptr(), rho=rho)   # 1 % tampered
        R_.barrier(stream)
        rejects = int(ok1[0].item()) == 0
        step_rand()
        R_.barrier(stream)
        accepts = int(ok1[0].item()) == 1
        l0 = eng.launch_count
        ms_rand = timed(step_rand, steps) / steps
        verdict_rand = ok1[:1].cpu().numpy()
        launches = (eng.launch_count - l0) // steps
        eng.profile_enable(True)
        step_rand()
        prof_r = {k.split("<")[0]: v for k, v in eng.profile_read().items()}
        eng.profile_enable(False)
        # the same through the host-buffer entry point (H2D of the whole batch inside, one verdict byte back)
        hosth = [h[honest.cpu()].contiguous().pin_memory() for h in host]
        ok1h = torch.zeros(4, dtype=torch.uint8).pin_memory()
        rho_buf = (ctypes.c_char * (8 * (2 * Ph + 1))).from_buffer_copy(rho[:8 * (2 * Ph + 1)])

        def step_rand_e2e():
            rc = lib.gs_verify_batch_rand(eng.h, 0, Ph, m, n, *[vp(h.data_ptr()) for h in hosth], ctypes.cast(rho_buf, vp), vp(ok1h.data_ptr()))
            if rc != 0:
                raise SystemExit(lib.gs_last_error(eng.h).decode())

        step_rand_e2e()
        accepts = accepts and int(ok1h[0]) == 1
        e2e_rand = R_.wall_ms(step_rand_e2e, steps, warmup=0)
        out["rand"] = {"proofs": Ph, "ms_per_step": ms_rand, "e2e_ms": e2e_rand, "accepts_honest_batch": accepts,
                       "rejects_batch_with_tampered": rejects, "launches_per_step": int(launches), "prof": prof_r,
                       "verdict": verdict_rand}
        del devh, hosth
    except Exception as ex:  # noqa: BLE001 -- the opt-in leg must not take the headline down
        out["rand"] = {"error": f"{type(ex).__name__}: {ex}"}
    return out


# ---------------------------------------------------------------- C3: one large statement split by slot
def bench_c3_sharded(R_, eng, size, steps):
    from gsutil import SeededRng, make_crs, crs_bytes, fr_b
    from workloads import instance
    torch = R_.torch
    crs, _ = make_crs(3)
    eng.crs_load(crs_bytes(crs))
    eng._crs = crs
    rng = SeededRng(3)
    m = n = size
    t0 = time.perf_counter()
    A, B, G, T, X, Y = instance(eng, 0, m, n, rng)
    xr = b"".join(fr_b(rng.fr()) for _ in range(2 * m))
    yr = b"".join(fr_b(rng.fr()) for _ in range(2 * n))
    Tr = b"".join(fr_b(rng.fr()) for _ in range(4))
    build_s = time.perf_counter() - t0
    xc, yc = eng.batch_commit_g1(X, xr), eng.batch_commit_g2(Y, yr)
    pi, th = eng.prove(0, m, n, A, B, G, X, Y, xr, yr, Tr)
    arrs = [A, B, G, T, xc, yc, pi, th]
    g = bytearray(G)
    g[32 * (5 * n + 7)] ^= 1
    bad = list(arrs)
    bad[2] = bytes(g)

    import groth_sahai_rs_b200 as gsb
    sh = gsb.shard

    # every rank HOLDS the rows of Gamma it owns (rows i = rank mod N: 1 / N of the statement) -- sliced outside the timed region
    rows_of = {id(arrs): sh.gamma_rows_of(arrs[2], 1, m, n, R_.rank, R_.world), id(bad): sh.gamma_rows_of(bad[2], 1, m, n, R_.rank, R_.world)}
    ag = sh.make_allgather(R_.dev)

    def sharded_verify(a):          # MSM split by base, Miller pairs by slot, two all-gathers over NCCL (gs_verify_sharded)
        return eng.verify_sharded(0, 1, m, n, a[0], a[1], rows_of[id(a)], a[3], a[4], a[5], a[6], a[7], R_.rank, R_.world, ag)

    def slot_verify(a):             # the round-1 path: everything split by slot, every rank uploads the whole statement
        mine = eng.verify_partial(0, 1, m, n, *a, R_.rank, R_.world)
        if R_.world == 1:
            return eng.verify_finish(0, 1, mine, a[3])
        t = torch.frombuffer(bytearray(mine), dtype=torch.uint8).to(R_.dev)
        parts = [torch.empty_like(t) for _ in range(R_.world)]
        R_.dist.all_gather(parts, t)
        return eng.verify_finish(0, 1, torch.cat(parts).cpu().numpy().tobytes(), a[3])

    assert sharded_verify(arrs) == b"\x01", "honest statement rejected"
    assert sharded_verify(bad) == b"\x00", "tampered Gamma accepted"
    assert slot_verify(arrs) == b"\x01" and slot_verify(bad) == b"\x00"
    ms = R_.wall_ms(lambda: sharded_verify(arrs), steps)
    ms_slot = R_.wall_ms(lambda: slot_verify(arrs), steps)
    prof = profiled(eng, lambda: sharded_verify(arrs))
    ms_prove = R_.wall_ms(lambda: eng.prove(0, m, n, A, B, G, X, Y, xr, yr, Tr), steps)
    prof_p = profiled(eng, lambda: eng.prove(0, m, n, A, B, G, X, Y, xr, yr, Tr))
    cpu_prove = None
    if R_.rank == 0 and R_.world == 1 and m <= 1024:     # the reference-order CPU prover on the same statement (outside any timing)
        try:
            from oracle import cbaseline as cb
            t0 = time.perf_counter()
            p_, t_ = cb.prove(0, m, n, A, B, G, X, Y, xr, yr, Tr, crs_bytes(crs), cb.host_cores())
            cpu_prove = {"prove_ms": round((time.perf_counter() - t0) * 1e3, 1), "cores": cb.host_cores(), "kind": "port",
                         "proof_bytes_equal_gpu": bool(p_ == pi and t_ == th),
                         "note": "C restatement, scalar multiplications of each left_mul spread over host threads "
                                 "(the reference itself runs <= 2 Rayon tasks in prove)"}
        except Exception as ex:  # noqa: BLE001
            cpu_prove = {"error": str(ex)}
    pairs = 4 * n + 2 * m + 16
    h2d = sum(len(a) for a in arrs) - len(G) + len(G) // R_.world
    return {"workload": f"C3: one PPE, m=n={m}, dense Gamma (BASELINE.json configs[2]); gs_verify_sharded x{R_.world}: statement MSM "
                        "split by base (every rank uploads its rows of Gamma only), all_gather of the partial sums "
                        f"({2 * n * 96} B per rank), Miller pairs split by slot, all_gather of 2,304 B, final exponentiation on every rank",
            "scaling": "strong", "n_gpus": R_.world, "verify_ms": round(ms, 3), "verifies_per_sec": round(1e3 / ms, 2),
            "verify_ms_split_by_slot_only": round(ms_slot, 3),
            "miller_pairs_per_verify": pairs, "pairings_per_sec": round(pairs / (ms * 1e-3), 1),
            "prove_ms_one_gpu": round(ms_prove, 3), "cpu_prove": cpu_prove, "h2d_bytes_per_rank": h2d, "instance_build_s": round(build_s, 1),
            "rank0_verify_kernels": prof, "rank0_prove_kernels": prof_p,
            "limiter": f"per-rank latency floors (one dependent chain each), not NCCL: {top_kernels(prof, 4)}; "
                       f"H2D per rank {h2d >> 20} MiB",
            "parity": "honest -> 1, one flipped Gamma bit -> 0 (sharded path); proof bytes == reference-order CPU proof at "
                      "this size in tests/test_gpu_bigparity.py::test_1024x1024_ppe"}


# ---------------------------------------------------------------- C4: a multi-equation statement split by equation
def bench_c4_by_equation(R_, eng, E, steps):
    import groth_sahai_rs_b200 as gsb
    from gsutil import SeededRng, make_crs, crs_bytes
    from workloads import instance_many
    sh = gsb.shard
    crs, _ = make_crs(4)
    crsb = crs_bytes(crs)
    eng.crs_load(crsb)
    eng._crs = crs
    m = n = 64
    rank, world, dev = R_.rank, R_.world, R_.dev
    names = ["PPE", "MSMEG1", "MSMEG2", "QuadEqu"]
    per_type = {}
    tot_commit = tot_prove = tot_verify = 0.0
    t_build0 = time.perf_counter()
    data = [instance_many(eng, ty, m, n, E, SeededRng(40 + ty)) for ty in range(4)]     # same seeded statement on every rank
    build_s = time.perf_counter() - t_build0
    for ty in range(4):
        A, B, G, T, X, Y, xr, yr, Tr = data[ty]
        gx, gy = ty in (0, 1), ty in (0, 2)
        xs, ys, cx, cy = (96 if gx else 32), (192 if gy else 32), (2 if gx else 1), (2 if gy else 1)
        ts = (576, 96, 192, 32)[ty]
        cat = b"".join
        Aall, Ball, Gall, Tall, Trall = cat(A), cat(B), cat(G), cat(T), cat(Tr)
        com_x = lambda a, k: (eng.batch_commit_g1 if gx else eng.batch_commit_scalar_b1)(a[0], a[1])
        com_y = lambda a, k: (eng.batch_commit_g2 if gy else eng.batch_commit_scalar_b2)(a[0], a[1])

        def commit():
            xc = sh.commit_sharded(com_x, [X, xr], [xs, cx * 32], m, 192, rank, world, device=dev)
            yc = sh.commit_sharded(com_y, [Y, yr], [ys, cy * 32], n, 384, rank, world, device=dev)
            return xc, yc

        def prove():
            return sh.prove_equations_sharded(
                lambda a, k: eng.prove_batch(ty, k, m, n, a[0], a[1], a[2], X, Y, xr, yr, a[3], shared_vars=True),
                [Aall, Ball, Gall, Trall], [n * xs, m * ys, m * n * 32, cx * cy * 32], E, cx * 384, cy * 192, rank, world,
                device=dev)

        xc, yc = commit()
        pi, th = prove()

        def verify(tg=Tall):
            return sh.verify_equations_sharded(
                lambda a, k: eng.verify_batch(ty, k, m, n, a[0], a[1], a[2], a[3], xc * k, yc * k, a[4], a[5]),
                [Aall, Ball, Gall, tg, pi, th], [n * xs, m * ys, m * n * 32, ts, cx * 384, cy * 192], E, rank, world,
                device=dev)

        def verify_by_base(tg=Tall):   # ONE call for the type's E equations: shared-base tables split by base over the ranks
            return sh.verify_statement_base_sharded(eng, ty, E, m, n, [Aall, Ball, Gall, tg, xc * E, yc * E, pi, th], rank, world, dev)

        ok = bytes(verify().cpu().tolist())
        assert ok == b"\x01" * E, f"C4 type {ty}: {ok.count(1)} of {E} verified"
        assert verify_by_base() == b"\x01" * E, f"C4 type {ty}: base-sharded verification disagrees"
        tb = bytearray(Tall)
        tb[3 * ts:4 * ts], tb[(E - 1) * ts:E * ts] = tb[(E - 1) * ts:E * ts], tb[3 * ts:4 * ts]   # swap two targets
        okb = bytes(verify(bytes(tb)).cpu().tolist())
        exp = bytearray(b"\x01" * E)
        exp[3] = exp[E - 1] = 0
        assert okb == bytes(exp), f"C4 type {ty}: tamper mask wrong"
        assert verify_by_base(bytes(tb)) == bytes(exp), f"C4 type {ty}: base-sharded tamper mask wrong"
        parity = None
        if rank == 0:      # two equations' proofs against the reference-order CPU prover (outside the timed region)
            from oracle import cbaseline as cb
            for e in (0, E - 1):
                p_, t_ = cb.prove(ty, m, n, A[e], B[e], G[e], X, Y, xr, yr, Tr[e], crsb, cb.host_cores())
                assert p_ == pi[e * cx * 384:(e + 1) * cx * 384] and t_ == th[e * cy * 192:(e + 1) * cy * 192], \
                    f"C4 type {ty} equation {e}: proof differs from the reference-order CPU proof"
            parity = "equations 0 and E-1: proof bytes == oracle/gs_oracle.c gsref_prove"
        t_c = R_.wall_ms(commit, steps)
        t_p = R_.wall_ms(prove, steps)
        t_v_eq = R_.wall_ms(verify, steps)
        t_v_base = R_.wall_ms(verify_by_base, steps)
        by_base = t_v_base < t_v_eq
        t_v = min(t_v_eq, t_v_base)
        prof_p = profiled(eng, prove)
        prof_v = profiled(eng, verify_by_base if by_base else verify)
        per_type[names[ty]] = {"commit_ms": round(t_c, 3), "prove_ms": round(t_p, 3), "verify_ms": round(t_v, 3),
                               "verify_split": "MSM by base + pairs by slot (gs_verify_sharded)" if by_base else "by equation (gs_verify_batch per rank)",
                               "verify_ms_by_equation": round(t_v_eq, 3), "verify_ms_by_base": round(t_v_base, 3),
                               "proved_per_sec": round(E / (t_p * 1e-3), 1), "verified_per_sec": round(E / (t_v * 1e-3), 1),
                               "rank0_prove_kernels": prof_p, "rank0_verify_kernels": prof_v, "parity": parity,
                               "limiter": f"prove: {top_kernels(prof_p, 2)}; verify: {top_kernels(prof_v, 2)}"}
        tot_commit += t_c
        tot_prove += t_p
        tot_verify += t_v
    return {"workload": f"C4: mixed statement, {E} each of PPE/MSMEG1/MSMEG2/QuadEqu over shared variable sets m=n=m'=n'=64 "
                        f"(BASELINE.json configs[3]); commit split by variable, prove and verify split by equation x{world}",
            "scaling": "strong", "n_gpus": world, "equations": 4 * E, "commit_ms": round(tot_commit, 3),
            "prove_ms": round(tot_prove, 3), "verify_ms": round(tot_verify, 3),
            "proved_per_sec": round(4 * E / (tot_prove * 1e-3), 1), "verified_per_sec": round(4 * E / (tot_verify * 1e-3), 1),
            "commit_prove_verify_per_sec": round(4 * E / ((tot_commit + tot_prove + tot_verify) * 1e-3), 1),
            "collectives": "all_gather of commitments (64 x 192 / 384 B), of proofs (<= 1,152 B per equation), of verdict bytes",
            "instance_build_s": round(build_s, 1), "per_type": per_type,
            "limiter": "per-rank fixed costs that do not shrink with the rank's share of the equations: the shared-base window "
                       "tables (built on every rank) and the G2 line walk of the shared y-commitments"}


def cpu_baseline_record(m, n):
    """The C restatement of the reference on the host cores: verify on all cores (bounded sample), plus the latency of one
    prove and one verify on one core (the reference's `prove` parallelises over <= 2 Rayon tasks)."""
    from oracle import cbaseline as cb
    r = cb.time_ppe_verify(m=m, n=n, sample=0, steps=1, warmup=0)
    rec = {"value": r["verifies_per_sec"], "unit": "verifies/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample_desc"],
           "single_core_verify_ms": round(r["single_core_verify_ms"], 2)}
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from bigcase import Case
        from gsutil import make_crs
        t0 = time.perf_counter()
        c = Case(0, m, n, make_crs(5)[0], seed=77, prove=False)
        t0 = time.perf_counter()
        cb.prove(0, m, n, c.A, c.B, c.G, c.X, c.Y, c.xr, c.yr, c.Tr, c.crsb, 1)
        rec["single_core_prove_ms"] = round((time.perf_counter() - t0) * 1e3, 2)
        t0 = time.perf_counter()
        cb.commit_x(0, c.X, c.xr, c.crsb)
        cb.commit_y(0, c.Y, c.yr, c.crsb)
        rec["single_core_commit_ms"] = round((time.perf_counter() - t0) * 1e3, 2)
    except Exception as ex:  # noqa: BLE001
        rec["prove_note"] = f"unavailable: {ex}"
    return rec


DUMP_BYTES = 64 << 20


def positive_int(s):
    v = int(s)
    if v < 1:
        raise argparse.ArgumentTypeError(f"{s} is not a positive integer")
    return v


def dump_outputs(d, arrays):
    """Each array as float32 d/<name>.npy, all of them within DUMP_BYTES: an array over its share is replaced by a fixed,
    seeded sample of its elements, and d/<name>_index.npy (float64) holds the positions sampled."""
    import numpy as np
    share = DUMP_BYTES // len(arrays) - 4096                  # (room for the .npy headers)
    for name, a in arrays.items():
        a = np.asarray(a, dtype=np.float32).ravel()
        if a.nbytes > share:
            idx = np.sort(np.random.default_rng(0).choice(a.size, share // 12, replace=False))
            np.save(os.path.join(d, f"{name}_index.npy"), idx.astype(np.float64))
            a = a[idx]
        np.save(os.path.join(d, f"{name}.npy"), a)


# ---------------------------------------------------------------- GPU arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=3, help="timed steps of every leg")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--proofs", type=int, default=65536, help="proofs per step in TOTAL (sharded over the GPUs)")
    ap.add_argument("--distinct", type=int, default=0, help="distinct proved instances per rank (0 = every proof distinct)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--ref-sample", type=int, default=0, help="proofs per CPU step (0 = auto, ~10-30 s)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--skip", default="", help="comma list of sub-records to skip: weak,c3,c4")
    ap.add_argument("--c3-size", type=int, default=1024)
    ap.add_argument("--c4-eqs", type=int, default=256)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's C5 outputs as DIR/<name>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs dumps the GPU path; it does not apply to --impl reference")
        return run_reference(args)
    if args.dump_outputs:
        os.makedirs(args.dump_outputs, exist_ok=True)       # fail before the run, not after it

    import groth_sahai_rs_b200 as gsb
    R_ = Ranks()
    R_.init()
    rank, world = R_.rank, R_.world
    skip = set(s for s in args.skip.split(",") if s)
    eng = gsb.Engine(R_.local)
    m, n = M_VARS, N_VARS
    lo, hi = gsb.shard.shard_range(args.proofs, rank, world)
    P = hi - lo
    if P * world != args.proofs:
        raise SystemExit("--proofs must be a multiple of the number of GPUs")
    c5 = bench_c5(R_, eng, P, args.distinct, args.steps, args.warmup, full=True)
    ms_per_step = c5["ms_per_step"]
    value = args.proofs / (ms_per_step * 1e-3)
    e2e_value = args.proofs / (c5["e2e_ms"] * 1e-3)

    wm = work_model(m, n)
    peak_m = eng.fpmul_rate()                       # measured Fp products/s (register-only chain) on this GPU
    peak_imad = peak_m * IMAD_PER_M
    prof = c5["prof"]
    step_ms_prof = sum(v[1] for v in prof.values())
    pipe = {}
    ipath = os.path.join(ROOT, "profiles", "imad_counts.json")     # executed IMAD.WIDE per proof from the committed ncu source pages
    if os.path.exists(ipath):
        pipe = json.load(open(ipath))
    n_sm = R_.torch.cuda.get_device_properties(R_.local).multi_processor_count
    sm_mhz = c5["clocks"].get("sm_mhz") or c5["clocks"].get("sm_max_mhz")
    pipe_peak = n_sm * sm_mhz * 1e6 if sm_mhz else None
    kern = {}
    for name, (cnt, ms) in prof.items():
        w = wm.get(name)
        kern[name] = {"launches": cnt, "ms": round(ms, 3), "share": round(ms / step_ms_prof, 4)}
        if w:
            kern[name]["frac_of_imad_peak"] = round(w * P / (ms * 1e-3) / peak_m, 4)
        ex = pipe.get("imad_wide_warp_per_proof", {}).get(name)
        if ex and pipe_peak:     # executed warp-level IMAD.WIDE / s against the pipe's rate: 1 warp instruction / clk / SM
            kern[name]["pipe_util"] = round(ex * P / (ms * 1e-3) / pipe_peak, 4)
    dom = max(prof.items(), key=lambda kv: kv[1][1])[0]
    dom_cnt, dom_ms = prof[dom]
    dom_achieved = wm[dom] * P * IMAD_PER_M / (dom_ms * 1e-3) if dom in wm else None
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")    # per-launch DRAM bytes from the committed ncu capture
    traffic_capture = None
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        traffic_capture = tj.get(dom)
        if traffic_capture:     # the capture ran 16,384 proofs per launch; scale linearly to THIS run's proofs per launch
            traffic = int(traffic_capture * (P / dom_cnt) / tj.get("proofs_per_launch", 16384))
    hbm = None
    try:                                                        # HBM view of the same kernel (north star: report GB/s for the
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))      # point-load phases): ncu DRAM bytes per launch,
        if traffic:                                             # (already scaled to this run's proofs per launch)
            gbs = traffic / (dom_ms / dom_cnt * 1e-3) / 1e9
            hbm = {"achieved_gbs": round(gbs, 1), "peak_gbs": peaks.get("hbm_gbs"), "frac": round(gbs / peaks["hbm_gbs"], 4),
                   "peak_source": "MEASURED_PEAKS.json (driver-measured copy bandwidth)"}
    except Exception:  # noqa: BLE001
        hbm = None
    whole = round(sum(wm[k] for k in wm if k != "pairs") * P / (ms_per_step * 1e-3) / peak_m, 4)
    roofline = {
        "bound": "imad", "kernel": dom, "achieved": dom_achieved and round(dom_achieved / 1e12, 3),
        "peak": round(peak_imad / 1e12, 3), "unit": "TIMAD/s", "frac": dom_achieved and round(dom_achieved / peak_imad, 4),
        "whole_step_frac": whole, "pipe_util": kern.get(dom, {}).get("pipe_util"),
        "frac_note": "frac = SURVEY.md §8d model work / time / measured peak; the model charges the 39 M tower formula per line "
                     "where the kernel's unit-coefficient lines need fewer products, so frac can exceed 1 -- pipe_util (executed "
                     "IMAD.WIDE from the committed ncu source page / the pipe's measured rate) and whole_step_frac are the "
                     "figures to lead with",
        "traffic": traffic, "traffic_source": "profiles/traffic.json (ncu --set full at 16,384 proofs per launch: %s B) scaled to this run's "
                                              "proofs per launch" % traffic_capture, "hbm": hbm,
        "peak_source": "measured live: register-only Fp Montgomery chain (gs_diag_fpmul_rate) x 600 IMAD/M; "
                       "MEASURED_PEAKS.json has no integer-pipe figure",
        "kernels": kern,
    }
    waves = -(-P // MILLER_WAVE)
    limiter = (f"integer-multiply issue rate ({top_kernels(prof)}); strong scaling: {P} proofs per GPU = {P / MILLER_WAVE:.2f} waves of "
               f"k_miller4 ({MILLER_WAVE} proofs per wave) -> wave quantisation {P / MILLER_WAVE / waves:.3f}; no collective on the "
               f"data path ({P} verdict bytes all-gathered)")

    extras = {}

    def sub(name, fn):
        try:
            extras[name] = fn()
        except Exception as ex:  # noqa: BLE001 -- a sub-record must never take the headline down
            import traceback
            extras[name] = {"error": f"{type(ex).__name__}: {ex}", "trace": traceback.format_exc()[-600:]}
            if world > 1:
                raise

    if world > 1 and "weak" not in skip:
        def weak():
            w = bench_c5(R_, eng, args.proofs, 4096, args.steps, 1, full=False)
            return {"workload": f"C5 weak: {args.proofs} proofs PER GPU (the round-1 headline)", "scaling": "weak", "n_gpus": world,
                    "value": round(world * args.proofs / (w["ms_per_step"] * 1e-3), 1), "unit": "verifies/s",
                    "ms_per_step": round(w["ms_per_step"], 3), "distinct_instances_per_gpu": 4096,
                    "limiter": "none: independent proofs, verdict bytes all-gathered"}
        sub("c5_weak", weak)
    if "c3" not in skip:
        sub("c3_sharded", lambda: bench_c3_sharded(R_, eng, args.c3_size, args.steps))
    if "c4" not in skip:
        sub("c4_by_equation", lambda: bench_c4_by_equation(R_, eng, args.c4_eqs, args.steps))

    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        try:
            cpu = cpu_baseline_record(m, n)
        except Exception as ex:  # noqa: BLE001
            cpu = {"value": None, "unit": "verifies/s", "cores": 0, "kind": "port", "sample": f"unavailable: {ex}"}

    if rank == 0:
        line = {
            "metric": "ppe_verifies_per_sec", "value": round(value, 1), "unit": "verifies/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms_per_step, 3), "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "u32x12-montgomery", "data": "synthetic",
            "config": {"workload": "C5: batch verification of 65,536 independent 4x4 PPE proofs sharded across the GPUs "
                                   "(BASELINE.json configs[4])",
                       "m": m, "n": n, "proofs_total": args.proofs, "proofs_per_gpu": P, "distinct_instances_per_gpu": c5["distinct"],
                       "tampered": "1%", "l2": "inputs+line scratch (GBs) exceed the 126 MB L2; no flush needed",
                       "parallelism": f"proof-sharded x{world} (contiguous blocks), verdict all_gather",
                       "workload_build_s": c5["build_s"]},
            "pairings_per_sec": round(value * wm["pairs"], 1),
            "miller_pairs_per_verify": wm["pairs"], "final_exps_per_verify": 4,
            "e2e": {"value": round(e2e_value, 1), "unit": "verifies/s", "ms_per_step": round(c5["e2e_ms"], 3),
                    "h2d_bytes_per_step": c5["h2d_bytes"] * world, "d2h_bytes_per_step": c5["d2h_bytes"] * world},
            "gpu_launches": int(c5["launches"]), "roofline": roofline, "clocks": c5["clocks"], "limiter": limiter,
            "parity_sample": c5["parity_sample"],
        }
        rnd = c5.get("rand")
        if rnd and "error" not in rnd:
            line["c5_randomised"] = {
                "workload": "the honest proofs of the same C5 batch through gs_verify_batch_rand (opt-in, SURVEY.md 8f.4): the four "
                            "ComT entries of all proofs folded into one pairing product with 64-bit random weights, ONE final "
                            "exponentiation and ONE verdict per call; not bit-comparable with the reference's per-proof booleans "
                            "(a rejected batch goes through the exact path)",
                "value": round(world * rnd["proofs"] / (rnd["ms_per_step"] * 1e-3), 1), "unit": "verifies/s",
                "proofs_per_gpu": rnd["proofs"], "ms_per_step": round(rnd["ms_per_step"], 3),
                "e2e": {"value": round(world * rnd["proofs"] / (rnd["e2e_ms"] * 1e-3), 1), "unit": "verifies/s",
                        "ms_per_step": round(rnd["e2e_ms"], 3)},
                "speedup_vs_exact": round((rnd["proofs"] / rnd["ms_per_step"]) / (P / ms_per_step), 3),
                "accepts_honest_batch": rnd["accepts_honest_batch"], "rejects_batch_with_tampered": rnd["rejects_batch_with_tampered"],
                "launches_per_step": rnd["launches_per_step"],
                "kernels_ms": {k: round(v[1], 3) for k, v in sorted(rnd["prof"].items(), key=lambda kv: -kv[1][1])},
            }
        elif rnd:
            line["c5_randomised"] = rnd
        line.update(extras)
        if cpu is not None:
            line["cpu_baseline"] = cpu
        if args.dump_outputs:
            outs = {"c5_verdicts": c5["verdicts"]}
            if rnd and "verdict" in rnd:
                outs["c5_randomised_verdict"] = rnd["verdict"]
            dump_outputs(args.dump_outputs, outs)
        print(json.dumps(line))
    if world > 1:
        R_.dist.destroy_process_group()


if __name__ == "__main__":
    main()
