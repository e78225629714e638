#!/usr/bin/env python
"""Headline benchmark: STARK proofs per second (and ms per proof) for the reference's proving path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl zkb200|reference] [--dump-outputs DIR]

A step is `--inflight` (default 4) complete proofs per GPU (`Prover::prove`, /root/reference src/main.rs:228), each of its own
seeded synthetic trace, kept in flight on separate contexts; `prove_ms` is the latency of one proof proved alone.
`value` times it with the trace already resident in HBM, `e2e` through the C ABI with pinned HOST columns
(H2D of the trace and D2H of the proof inside the timed region).  Multi-GPU runs one independent proof stream
per rank (weak scaling, no collective on the data path).  `--impl reference` times the CPU oracle — the
restatement of the reference's Winterfell CPU prover (the Rust original cannot be built in this image) —
on all host cores, on the same workload.  Prints exactly one JSON line (rank 0)."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# stdout carries exactly one JSON line.  Libraries write to file descriptor 1 behind Python's back (NCCL prints its version
# banner there), so fd 1 is pointed at stderr for the whole run and the JSON line goes to the saved original stdout.
_REAL_STDOUT = None


def capture_stdout():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (air, n, w, blowup, description)
    "training_2p16": ("training", 1 << 16, 240, 16, "training AIR (src/training), 2^16-row x 240-col trace, blowup 16 (LDE 2^20 rows)"),
    "training_8192": ("training", 8192, 240, 16, "training AIR, 8192-row trace (bs=50, the CLI maximum), blowup 16"),
    "training_2p18": ("training", 1 << 18, 240, 16, "training-shaped AIR, 2^18-row x 240-col trace, blowup 16"),
    "training_2p20": ("training", 1 << 20, 240, 16, "training-shaped AIR, 2^20-row x 240-col trace, blowup 16 (LDE 60 GiB)"),
    "mimc_2p14": ("mimc", 1 << 14, 64, 8, "MiMC chains, 2^14 steps x 64 columns, blowup 8"),
    "mimc_2p20": ("mimc", 1 << 20, 64, 8, "MiMC chains, 2^20 steps x 64 columns, blowup 8 (LDE 8 GiB)"),
    "mimc_2p22": ("mimc", 1 << 22, 64, 8, "MiMC chains, 2^22 steps x 64 columns, blowup 8 (LDE 32 GiB)"),
    "aggregation_16": ("aggregation", 32, 120, 16, "FedAvg aggregation AIR over 16 updates, 32 x 120 trace"),
}


def algorithmic_bytes(n, w, beta, ce, c, folding=16, rem_domain=128):
    """SURVEY §8(d): compulsory HBM traffic per proof, stage by stage."""
    s, N = 16, n * beta
    b = {
        "interp": 2 * w * n * s,
        "lde": w * n * s + w * N * s,
        "leaf": w * N * s + 32 * N,
        "merkle": 96 * N,
        "ceval": w * (ce * n) * s + ce * n * s,
        "comp": 2 * ce * n * s + c * n * s + c * N * s + (c * N * s + 32 * N) + 96 * N,
        "ood": (w + c) * n * s,
        "deep": (w + c) * n * s + n * s + (n * s + N * s),
    }
    fri, m = 0, N
    while m > rem_domain:
        fri += m * s + (m // folding) * s + 32 * m // folding + 96 * m // folding
        m //= folding
    b["fri"] = fri
    b["total"] = sum(b.values())
    return b


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device, self.samples, self.proc = device, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.device), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "25"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        rows = [r for t, r in self.samples if t0 <= t <= t1 and len(r) >= 7] or [r for _, r in self.samples if len(r) >= 7]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        try:
            sm = [float(r[0]) for r in rows]
            reasons = []
            for idx, name in ((3, "hw_slowdown"), (4, "hw_thermal_slowdown"), (5, "sw_thermal_slowdown"), (6, "sw_power_cap")):
                if any(r[idx].lower().startswith("active") for r in rows):
                    reasons.append(name)
            return {"sm_mhz": statistics.median(sm), "sm_max_mhz": float(rows[0][1]), "power_w_max": max(float(r[2]) for r in rows),
                    "samples": len(rows), "reasons": reasons}
        except ValueError:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unparsed"]}


def build_workload(name, seed):
    """Returns (air description, trace array (w, n, 2) uint64 or None when generated on the device, extra)."""
    import zk_stark_project_b200 as Z
    from zk_stark_project_b200 import synthetic as S
    kind, n, w, beta, _ = WORKLOADS[name]
    opts = Z.ProofOptions(40, beta, 21, Z.FieldExtension.NONE, 16, 7)  # src/main.rs:98-107 (MiMC: blowup 8 per BASELINE.json)
    if kind == "training":
        data = S.random_felts(w * n, seed).reshape(w, n, 2)
        return S.synthetic_training_air(n, opts, data), data, opts
    if kind == "aggregation":
        import random
        from zk_stark_project_b200 import field as F
        rng = random.Random(seed)
        mk = lambda sig: F.f64_to_signed_felt(rng.gauss(0, sig), 1e6)[0]
        gw = [[mk(1e4) for _ in range(9)] for _ in range(6)]
        gb = [mk(1e4) for _ in range(6)]
        reps = [rng.randrange(2**64) for _ in range(16)]
        lw = [[[Z.f64_to_felt(r / 1e6)] * 9 for _ in range(6)] for r in reps]
        lb = [[Z.f64_to_felt(r / 1e6)] * 6 for r in reps]
        p = Z.GlobalUpdateProver(opts, gw, gb, lw, lb, Z.f64_to_felt(16.0), seed=seed)
        tr = p.build_trace()
        return p.describe(tr), np.ascontiguousarray(tr.data), opts
    # mimc: the chain trace is produced by the caller-side generator (device kernel for the product, oracle for the reference)
    return None, None, opts


def mimc_air(opts, w, n, first, last):
    import zk_stark_project_b200 as Z
    pub = Z.MimcInputs(first, last)
    return Z.MimcAir(w, n, pub, opts).describe()


DUMP_LIMIT = 64 << 20


def dump_outputs(path, results):
    """--dump-outputs: what the timed path returned in its last step, one row per proof of that step.  `proof.npy` holds the
    proof bytes (float32, one byte per element) and `transcript_<field>.npy` the Fiat-Shamir transcript returned with each proof
    (float64; every field is an integer below 2^53).  The proofs are deterministic (the smallest proof-of-work nonce), so two
    builds run with the same arguments must write the same arrays.  Rows beyond 64 MB in all are left out."""
    import ctypes
    row_bytes = 4 * len(results[0][0]) + 8 * ctypes.sizeof(results[0][1])  # a transcript has fewer fields than bytes
    results = results[:max(1, DUMP_LIMIT // row_bytes)]
    arrays = {"proof": np.stack([np.frombuffer(p, dtype=np.uint8) for p, _ in results]).astype(np.float32)}
    for name, _ in results[0][1]._fields_:
        if not name.startswith("_"):
            vals = [getattr(ts, name) for _, ts in results]
            arrays["transcript_" + name] = np.array([np.ctypeslib.as_array(v) if hasattr(v, "_length_") else v for v in vals], dtype=np.float64)
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(path, name + ".npy"), a)


def run_reference(args, rank, world):
    """CPU arm: the oracle prover (restatement of Winterfell's CPU prover) on all host cores."""
    if rank != 0:
        return
    from oracle import pyoracle as O
    import zk_stark_project_b200 as Z
    cores = os.cpu_count() or 1
    O.set_threads(cores)
    kind, n, w, beta, desc = WORKLOADS[args.workload]
    air, data, opts = build_workload(args.workload, 0x5EED0000)
    if kind == "mimc":
        rc = Z.get_round_constants()
        raw = O.mimc_trace([j + 1 for j in range(w)], n, rc)
        data = np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2)
        get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
        air = mimc_air(opts, w, n, [get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)])
    tb = data.tobytes()
    for _ in range(args.warmup):
        O.prove(air, tb)
    t0 = time.time()
    for _ in range(args.steps):
        proof, ts, _ = O.prove(air, tb)
    dt = (time.time() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, [(proof, ts)])
    val = 1.0 / dt
    line = {
        "impl": "reference", "metric": "stark_proofs_per_sec", "value": val, "unit": "proofs/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u128 mod p (f128 field), u32 BLAKE3", "data": "synthetic",
        "config": {"workload": f"{args.workload}: {desc}", "options": OPTIONS_TEXT, "l2": l2_text(n, w, beta)},
        "cpu_baseline": {"value": val, "unit": "proofs/s", "cores": cores, "kind": "port",
                         "sample": f"{args.steps} full proofs of the workload (C++ restatement of Winterfell 0.12's CPU prover, std::thread on all host cores, "
                                   "portable scalar BLAKE3 - upstream uses the SIMD blake3 crate; the Rust reference itself cannot be built in this image: "
                                   "no cargo/rustc)"},
        "e2e": {"value": val, "unit": "proofs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_mimc_helpers(args):
    """GPU counterpart of the reference's criterion bench for its MiMC helpers (benches/bench_mimc.rs:17-57): `mimc_cipher`
    (64 rounds of x <- (x + rc + z)^7, src/helper.rs:213-220) and `mimc_hash_matrix` over the bench's 6 x 9 weights + 6 biases
    (60 chained ciphers, src/helper.rs:222-233).  criterion times ONE call; a GPU needs a batch, so every case is one
    zkb_mimc_cipher_batch / zkb_mimc_hash_matrix_batch call through the C ABI with host buffers (copies inside the timed
    region).  cpu_baseline is the restatement's single-call latency on one host core."""
    import ctypes as C
    import numpy as np
    import zk_stark_project_b200 as Z
    from zk_stark_project_b200 import lib as L
    from zk_stark_project_b200 import synthetic as S

    def felts(vals):
        a = np.zeros((len(vals), 2), dtype=np.uint64)
        for i, v in enumerate(vals):
            a[i, 0], a[i, 1] = int(v) & 0xFFFFFFFFFFFFFFFF, int(v) >> 64
        return a

    def timed(fn):
        for _ in range(max(args.warmup, 1)):
            fn()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        return (time.perf_counter() - t0) / args.steps

    ctx = L.Context(0)
    lib = ctx.lib
    p = lambda a: a.ctypes.data_as(C.POINTER(C.c_uint8))
    rc = Z.get_round_constants()
    rc_arr = felts(rc)
    x0, r0 = 0x1234567890ABCDEF, 0x0FEDCBA987654321  # u64-sized inputs as in benches/bench_mimc.rs:22-25
    assert L.mimc_cipher_batch(ctx, [x0], [r0], [0])[0] == Z.mimc_cipher(x0, r0, 0)
    cpu = None
    if not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "oracle"))
        import pyoracle as O
        assert O.mimc_cipher(x0, r0, 0) == Z.mimc_cipher(x0, r0, 0)
        k = 20000
        t0 = time.perf_counter()
        for _ in range(k):
            O.mimc_cipher(x0, r0, 0)
        us = (time.perf_counter() - t0) / k * 1e6
        cpu = {"value": 1e6 / us, "unit": "ciphers/s", "cores": 1, "kind": "port",
               "sample": "%d single mimc_cipher calls through ctypes (call overhead included): %.2f us per call; "
                         "mimc_hash_matrix = 60 chained ciphers = %.0f us" % (k, us, 60 * us)}
    cases = []
    head = None
    for log_b in (0, 10, 16, 20, 22):
        b = 1 << log_b
        xs, rcs = S.random_felts(b, 7 + log_b), S.random_felts(b, 70 + log_b)
        xs[:, 1] = 0
        rcs[:, 1] = 0
        zs = np.zeros((b, 2), dtype=np.uint64)
        out = np.empty((b, 2), dtype=np.uint64)
        dt = timed(lambda: ctx.check(lib.zkb_mimc_cipher_batch(ctx.handle, p(xs), p(rcs), p(zs), C.c_uint64(b), p(out))))
        cases.append({"bench": "mimc_cipher", "batch": b, "call_ms": dt * 1e3, "ns_per_cipher": dt / b * 1e9, "ciphers_per_s": b / dt,
                      "field_muls_per_s": b * 256 / dt})
        if log_b == 20:
            head = (b, dt)
    ac, fe_n = 6, 9
    w_one, b_one = felts([Z.f64_to_felt(42.0)] * (ac * fe_n)), felts([Z.f64_to_felt(1.0)] * ac)  # benches/bench_mimc.rs:41-42
    want = Z.mimc_hash_matrix([[Z.f64_to_felt(42.0)] * fe_n] * ac, [Z.f64_to_felt(1.0)] * ac, rc)
    for log_b in (0, 10, 16, 18):
        b = 1 << log_b
        ws, bs = np.tile(w_one, (b, 1)), np.tile(b_one, (b, 1))
        out = np.empty((b, 2), dtype=np.uint64)
        dt = timed(lambda: ctx.check(lib.zkb_mimc_hash_matrix_batch(ctx.handle, p(ws), p(bs), C.c_uint32(ac), C.c_uint32(fe_n), p(rc_arr),
                                                                     C.c_uint32(len(rc)), C.c_uint64(b), p(out))))
        assert (int(out[b - 1, 0]) | (int(out[b - 1, 1]) << 64)) == want, "mimc_hash_matrix mismatch"
        cases.append({"bench": "mimc_hash_matrix", "batch": b, "call_ms": dt * 1e3, "us_per_hash": dt / b * 1e6, "hashes_per_s": b / dt})
    b, dt = head
    emit({"metric": "mimc_ciphers_per_sec", "value": b / dt, "unit": "ciphers/s", "n_gpus": 1, "steps": args.steps, "warmup": args.warmup,
          "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u128 mod p (f128 field)",
          "data": "synthetic", "config": {"workload": "mimc_helpers: batched mimc_cipher (headline: 2^20 per call) and mimc_hash_matrix 6x9+6",
                                          "reference": "benches/bench_mimc.rs:17-57"},
          "e2e": {"value": b / dt, "unit": "ciphers/s", "h2d_bytes_per_step": 48 * b, "d2h_bytes_per_step": 16 * b},
          "gpu_launches": ctx.launches(), "cases": cases, "cpu_baseline": cpu})


# dram__bytes_read.sum + dram__bytes_write.sum over the K1+K2 launches of ONE proof (transpose, interpolation passes, LDE passes),
# from an `ncu --set full` capture of that workload; None = not captured (never extrapolated).  Two passes through HBM per
# 2^16-point transform (a shared-memory tile holds 2^8 rows x 16 columns) make this 2.8x the algorithmic bytes.
NCU_TRAFFIC = {
    # interpolation passes 0.457 + 0.458 GB, LDE passes 4.259 + 8.031 GB (k_ntt_pass<true> x 4; the 0.5 GB transpose is not included)
    "training_2p16": (13.204e9, "profiles/r2_ncu_ntt_hash_training_2p16.txt (ncu --set full, dram__bytes_read.sum + dram__bytes_write.sum of the four K1+K2 launches)"),
}
OPTIONS_TEXT = "40 queries, grinding 21, FRI folding 16, remainder degree <= 7"


def l2_text(n, w, beta):
    return "inputs larger than L2 (trace %d MiB, LDE %d MiB)" % ((w * n * 16) >> 20, (w * n * 16 * beta) >> 20)


def counter_felts(w, n, seed, col0=0, cols=None):
    """Counter-based synthetic trace (so that a rank can build just its own columns): cell (j, i) = splitmix64 of a per-cell
    counter, hi word < 2^63 (canonical).  Returns a (cols, n, 2) uint64 array for columns [col0, col0 + cols)."""
    cols = w if cols is None else cols
    out = np.empty((cols, n, 2), dtype=np.uint64)

    def mix(x):
        x = x + np.uint64(0x9E3779B97F4A7C15)
        x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
        x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
        return x ^ (x >> np.uint64(31))
    idx = np.arange(n, dtype=np.uint64)
    with np.errstate(over="ignore"):
        for j in range(cols):
            base = np.uint64((seed * 0x100000001B3 + (col0 + j) * 2 * n) & 0xFFFFFFFFFFFFFFFF)
            out[j, :, 0] = mix(base + idx)
            out[j, :, 1] = mix(base + np.uint64(n) + idx) >> np.uint64(1)
    return out


def training_air_from_rows(n, w, opts, first, last):
    """Training AIR description from the boundary rows only (what get_pub_inputs reads, src/training/prover.rs:245-246)."""
    data = np.zeros((w, 2, 2), dtype=np.uint64)
    for j in range(w):
        data[j, 0, 0], data[j, 0, 1] = first[j] & 0xFFFFFFFFFFFFFFFF, first[j] >> 64
        data[j, 1, 0], data[j, 1, 1] = last[j] & 0xFFFFFFFFFFFFFFFF, last[j] >> 64
    from zk_stark_project_b200 import synthetic as S

    class _View:  # rows 0 and n-1 of the trace, addressed like the full array
        shape = (w, n, 2)

        def __getitem__(self, key):
            c, r, q = key
            return data[c, 0 if r == 0 else 1, q]
    return S.synthetic_training_air(n, opts, _View())


def roofline_of(workload, n, w_local, beta, lde_ms, alg_lde, peak, peak_src, sharded=False):
    achieved = alg_lde / (lde_ms * 1e-3) / 1e9
    traffic = NCU_TRAFFIC.get(workload) if not sharded else None
    bf = w_local * (n // 2) * (n.bit_length() - 1) * (beta + 1)
    return {
        "roofline": {"bound": "hbm", "kernel": "k_ntt_pass (K1 interpolation + K2 coset LDE)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic[0] if traffic else None,
                     "traffic_source": traffic[1] if traffic else "no ncu --set full capture of this workload",
                     "peak_source": peak_src, "algorithmic_bytes_per_proof": alg_lde, "kernel_ms_per_proof": lde_ms,
                     "note": "bound by integer issue, not HBM: a radix-2 f128 butterfly is ~69 SASS integer instructions per 32 bytes moved "
                             "(profiles/r2_mul_variants.txt, profiles/r2_sass_hist_hot_kernels.txt); ncu (profiles/r2_ncu_ntt_hash_training_2p16.txt): "
                             "issue slots 53-54% busy, ALU pipe 63%, FMA-heavy pipe 54%, DRAM 12-21% of peak"},
        # what actually bounds K1/K2: integer issue.  Peak = register-resident radix-2 f128 butterflies/s of the shipped twiddle multiplier
        # (four pre-shifted copies) on this pool's B200, best occupancy / ILP setting (tools/mul_variants.cu variant F; no memory traffic at all)
        "compute_roofline": {"unit": "G butterflies/s", "peak": 270.5, "achieved": bf / (lde_ms * 1e-3) / 1e9,
                             "frac": bf / (lde_ms * 1e-3) / 1e9 / 270.5, "source": "tools/mul_variants.cu variant F (251-270 G/s depending on ILP), profiles/r2_mul_variants.txt",
                             # against the MACHINE rather than against the multiplier's own ceiling: instruction issue.  Both integer pipes take one
                             # warp-instruction every two cycles per sub-partition, a balanced two-source mix issues 0.95/clk (profiles/r1_int_pipe_peaks.txt);
                             # ncu on the shipped LDE passes: 0.53-0.54 (profiles/r2_ncu_ntt_hash_training_2p16.txt) - carry-chained multi-limb code
                             # sits at 62-67 % of its binding pipe whatever the mix, so the lever left is the instruction count (69.4 per butterfly)
                             "issue_slots": {"unit": "warp-instr/clk/SMSP", "achieved_ncu": 0.535, "peak_measured_balanced_mix": 0.95, "frac": 0.56,
                                             "instr_per_butterfly": 69.4}},
    }


def pin_to_gpu_numa_node(device):
    """Multi-rank runs: bind this process (and with it the first-touch placement of its pinned trace buffers) to the CPUs NVML
    reports as local to its GPU, so that the end-to-end arm's H2D copies do not cross the socket interconnect.  Host plumbing
    only; returns the CPU count it was pinned to, or None when NVML / affinity is unavailable."""
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(device)
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (os.cpu_count() + 63) // 64)
        cpus = {64 * i + b for i, wd in enumerate(words) for b in range(64) if (wd >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="training_2p16", choices=sorted(WORKLOADS) + ["mimc_helpers"])
    ap.add_argument("--impl", default="zkb200", choices=["zkb200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the oracle timing at N=1")
    ap.add_argument("--no-headline", action="store_true", help="N=1: skip the 2^20-row-trace proofs (MiMC 64 x 2^20, training shape 240 x 2^20)")
    ap.add_argument("--no-sharded", action="store_true", help="N>1: skip the column-sharded single proof after the replica arm")
    ap.add_argument("--inflight", type=int, default=0,
                    help="independent proofs in flight per GPU in the throughput arms (one zkb_ctx + CUDA stream + host thread each; 0 = 4, or 2 on hosts with few cores); "
                         "single-proof latency is always measured too and reported as prove_ms")
    ap.add_argument("--sharded", action="store_true",
                    help="make the column-sharded proof of --workload the MAIN arm (ONE proof per step across all ranks, strong scaling) "
                         "instead of one independent proof stream per rank")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the proofs of the last step of the throughput arm (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.workload == "mimc_helpers":
        ap.error("--dump-outputs covers the proof workloads")
    capture_stdout()

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.workload == "mimc_helpers":  # benches/bench_mimc.rs counterpart: helper kernels, not a proof
        if rank == 0:
            run_mimc_helpers(args)
        return
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import zk_stark_project_b200 as Z
    from zk_stark_project_b200 import lib as L

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the zkb200 proving path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    numa = pin_to_gpu_numa_node(local_rank) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_ranks(*vals):
        if world == 1:
            return [float(v) for v in vals]
        t = torch.tensor(list(vals), device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return [float(x) for x in t]

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s (B200_PROFILING.md)"

    kind, n, w, beta, desc = WORKLOADS[args.workload]
    sharded = args.sharded and world > 1
    if args.sharded and kind == "aggregation":
        raise SystemExit("--sharded: the aggregation AIR couples columns i and i+60 and cannot be column-sharded")
    ctx = L.Context(local_rank)  # default stream: the same stream torch.cuda.Event records on
    mg_ready = False

    def ensure_mg():
        nonlocal mg_ready
        if not mg_ready:
            from zk_stark_project_b200 import multi_gpu as M
            M.init_sharded(ctx, rank, world, dist)
            mg_ready = True

    seed_rank = 0 if sharded else rank  # a sharded proof is ONE trace shared by all ranks
    air, data, opts = build_workload(args.workload, 0x5EED0000 + seed_rank)
    if kind == "mimc":
        rc = Z.get_round_constants()
        raw = ctx.mimc_trace([j + 1 + 1000 * seed_rank for j in range(w)], n, rc)  # device-side chain generator (SURVEY §8f)
        data = np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2)
        get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
        air = mimc_air(opts, w, n, [get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)])
    w_local = w // world if sharded else w
    if sharded:
        ensure_mg()
        data = data[rank * w_local:(rank + 1) * w_local]  # (every rank built the same seeded trace; it keeps its columns)
    nbytes = w_local * n * 16
    pinned = L.PinnedBuffer(nbytes)
    pinned.view()[:] = np.ascontiguousarray(data).reshape(-1).view(np.uint8)
    d_trace = ctx.upload_trace(pinned.ptr, w_local, n)
    air_dict, air = air, ctx.prepare(air)  # marshal the AIR description once, outside the timed regions
    prove_device = (lambda: ctx.mg_prove_device(air, d_trace)) if sharded else (lambda: ctx.prove_device(air, d_trace))

    ce = 8 if kind == "mimc" else 2
    c = 6 if kind == "mimc" else 1
    alg = algorithmic_bytes(n, w, beta, ce, c)

    # ---- contexts: one per in-flight proof, each on its own stream with its own device buffers --------------------------------
    # default: four proofs in flight per GPU; two when the host has fewer than 4 cores per rank.  A lane's host thread enqueues a whole
    # proof (the Fiat-Shamir channel runs on the device) and then sleeps on a blocking CUDA event, so lanes do not need a spinning
    # core each any more (round 1 had to drop to two lanes on the 32-core 8-GPU box)
    if args.inflight <= 0:
        args.inflight = 4 if (os.cpu_count() or 1) >= 4 * world else 2
    inflight = 1 if sharded else max(1, args.inflight)
    if 2.4 * n * beta * w_local * 16 * inflight > 100e9:  # LDE + NTT scratch + polys per lane must fit the 180 GB of HBM
        inflight = 1
    lanes = [(ctx, d_trace, pinned)]
    streams = []
    for _ in range(inflight - 1):
        st = torch.cuda.Stream(device=local_rank)
        streams.append(st)
        c2 = L.Context(local_rank, stream=st.cuda_stream)
        p2 = L.PinnedBuffer(nbytes)
        p2.view()[:] = pinned.view()
        lanes.append((c2, c2.upload_trace(p2.ptr, w_local, n), p2))

    def run_lanes(fn_of_lane, count):
        """`count` steps; every step proves one trace per lane concurrently (ctypes calls release the GIL)."""
        out = [None] * len(lanes)

        def work(i):
            for _ in range(count):
                out[i] = fn_of_lane(lanes[i])
        if len(lanes) == 1:
            work(0)
        else:
            th = [threading.Thread(target=work, args=(i,)) for i in range(len(lanes))]
            for t_ in th:
                t_.start()
            for t_ in th:
                t_.join()
        return out

    dev_fn = (lambda ln: ln[0].mg_prove_device(air, ln[1])) if sharded else (lambda ln: ln[0].prove_device(air, ln[1]))
    host_fn = (lambda ln: ln[0].mg_prove_host(air, ln[2].ptr, world)) if sharded else (lambda ln: ln[0].prove_host(air, ln[2].ptr))

    # ---- single-proof latency (one proof in flight), device-resident: `prove_ms` + per-stage times -------------------------------
    for _ in range(args.warmup):
        prove_device()
    stage_acc = {}
    barrier()
    l0 = ctx.launches()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record()
    for _ in range(args.steps):
        proof, ts = prove_device()
        for k_, v_ in ctx.stage_times().items():
            stage_acc[k_] = stage_acc.get(k_, 0.0) + v_
    g1.record()
    barrier()
    launches_per_proof = (ctx.launches() - l0) // args.steps
    ms_latency = g0.elapsed_time(g1)
    # ---- device-resident throughput arm (`value`): `inflight` proofs per GPU per step ------------------------------------------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    time.sleep(0.3)
    run_lanes(dev_fn, args.warmup)   # after the sampler's start-up pause: the timed region begins with clocks and lanes warm
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t_wall0 = time.time()
    e0.record()
    res = run_lanes(dev_fn, args.steps)
    e1.record()
    barrier()
    t_wall1 = time.time()
    launches = launches_per_proof * args.steps * inflight
    ms = e0.elapsed_time(e1)
    assert all(r[0] == proof for r in res), "in-flight proofs differ from the single-stream proof"
    last_step = res
    # ---- end-to-end arm: host columns in pinned memory through zkb_prove, same concurrency ----------------------------------------
    run_lanes(host_fn, min(args.warmup, 2))
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    res = run_lanes(host_fn, args.steps)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    sampler.stop()
    assert all(r[0] == proof for r in res), "e2e proof differs from the device-resident proof"

    ms, ms_e2e, ms_latency = max_ranks(ms, ms_e2e, ms_latency)
    if world > 1:
        lt = torch.tensor([launches], device="cuda", dtype=torch.int64)
        dist.all_reduce(lt, op=dist.ReduceOp.SUM)
        launches = int(lt[0])
    stages = {k_: v_ / args.steps for k_, v_ in stage_acc.items()}
    main_proof_len = len(proof)
    tb_main = bytes(pinned.view()) if (world == 1 and not args.no_cpu_baseline) else None

    # release the lanes: the next sections need the memory
    for c2, _, p2 in lanes[1:]:
        c2.close()
        p2.free()
    lanes = lanes[:1]
    pinned.free()

    def single_proof_case(name, steps, warm):
        """One proof at a time of workload `name` on this rank's context: device-resident latency, end-to-end latency from pinned
        host columns, stage times, roofline of the LDE stage.  Used for the 2^20-row-trace headline (N = 1)."""
        k2, n2, w2, b2, d2 = WORKLOADS[name]
        o2 = Z.ProofOptions(40, b2, 21, Z.FieldExtension.NONE, 16, 7)
        nb = w2 * n2 * 16
        pin = L.PinnedBuffer(nb)
        if k2 == "mimc":
            dptr = ctx.mimc_trace([j + 1 for j in range(w2)], n2, Z.get_round_constants(), device=True)
            pin.view()[:] = np.frombuffer(ctx.download(dptr, nb), dtype=np.uint8)
            arr = pin.view().view(np.uint64).reshape(w2, n2, 2)
            gv = lambda cc, r: int(arr[cc, r, 0]) | (int(arr[cc, r, 1]) << 64)
            a2 = mimc_air(o2, w2, n2, [gv(j, 0) for j in range(w2)], [gv(j, n2 - 1) for j in range(w2)])
        else:
            arr = pin.view().view(np.uint64).reshape(w2, n2, 2)
            arr[:] = counter_felts(w2, n2, 0x5EED2000)
            gv = lambda cc, r: int(arr[cc, r, 0]) | (int(arr[cc, r, 1]) << 64)
            a2 = training_air_from_rows(n2, w2, o2, [gv(j, 0) for j in range(w2)], [gv(j, n2 - 1) for j in range(w2)])
            dptr = ctx.upload_trace(pin.ptr, w2, n2)
        a2 = ctx.prepare(a2)
        for _ in range(warm):
            pr, _ = ctx.prove_device(a2, dptr)
        acc = {}
        torch.cuda.synchronize()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for _ in range(steps):
            pr2, _ = ctx.prove_device(a2, dptr)
            for k_, v_ in ctx.stage_times().items():
                acc[k_] = acc.get(k_, 0.0) + v_ / steps
        h1.record()
        torch.cuda.synchronize()
        assert pr2 == pr
        dev_ms = h0.elapsed_time(h1) / steps
        ctx.prove_host(a2, pin.ptr)
        h0.record()
        for _ in range(steps):
            pr3, _ = ctx.prove_host(a2, pin.ptr)
        h1.record()
        torch.cuda.synchronize()
        assert pr3 == pr, "e2e proof differs from the device-resident proof"
        e2e_ms = h0.elapsed_time(h1) / steps
        pin.free()
        ce2, c2_ = (8, 6) if k2 == "mimc" else (2, 1)
        al = algorithmic_bytes(n2, w2, b2, ce2, c2_)
        rec = {"workload": f"{name}: {d2}", "prove_ms": dev_ms, "e2e_ms": e2e_ms, "h2d_bytes": nb, "d2h_bytes": len(pr), "proof_bytes": len(pr),
               "steps": steps, "algorithmic_bytes": al["total"], "t_hbm_ms": al["total"] / peak / 1e6, "proof_roofline_frac": (al["total"] / peak / 1e6) / dev_ms,
               "stages_ms": {k_: round(v_, 3) for k_, v_ in acc.items() if v_ > 0 and k_ not in ("total", "h2d")}}
        rec.update(roofline_of(name, n2, w2, b2, max(acc.get("lde", 0.0), 1e-6), al["lde"] + al["interp"], peak, peak_src))
        return rec

    def sharded_case(name, steps, warm):
        """ONE proof of workload `name`, column-sharded over all ranks (zkb_mg_prove_device: NVLink all-to-all + all-gathers), timed
        as the max over ranks and compared byte for byte on rank 0 with the single-GPU proof (zkb_prove_device) of the same trace."""
        ensure_mg()
        k2, n2, w2, b2, d2 = WORKLOADS[name]
        o2 = Z.ProofOptions(40, b2, 21, Z.FieldExtension.NONE, 16, 7)
        wl = w2 // world
        if k2 == "mimc":
            # every rank runs the (deterministic) chain generator for all columns; its own columns are a contiguous slice
            dfull = ctx.mimc_trace([j + 1 for j in range(w2)], n2, Z.get_round_constants(), device=True)
            edge = lambda r: [int.from_bytes(ctx.download(dfull + (j * n2 + r) * 16, 16), "little") for j in range(w2)]
            a2 = mimc_air(o2, w2, n2, edge(0), edge(n2 - 1))
            dloc = dfull + rank * wl * n2 * 16
            pin = None
        else:
            # counter-based trace: a rank builds only its columns; rank 0 also builds the whole trace for the single-GPU proof
            mine = counter_felts(w2, n2, 0x5EED2000, rank * wl, wl)
            rows = torch.tensor(np.stack([mine[:, 0, :], mine[:, n2 - 1, :]]).astype(np.int64), device="cuda")
            allrows = [torch.empty_like(rows) for _ in range(world)]
            dist.all_gather(allrows, rows)
            fl = np.concatenate([t.cpu().numpy().astype(np.uint64) for t in allrows], axis=1)   # (2, w, 2)
            val = lambda r, j: int(fl[r, j, 0]) | (int(fl[r, j, 1]) << 64)
            a2 = training_air_from_rows(n2, w2, o2, [val(0, j) for j in range(w2)], [val(1, j) for j in range(w2)])
            pin = L.PinnedBuffer(wl * n2 * 16)
            pin.view()[:] = mine.reshape(-1).view(np.uint8)
            dloc = ctx.upload_trace(pin.ptr, wl, n2)
            dfull = None
        a2 = ctx.prepare(a2)
        for _ in range(warm):
            pr, _ = ctx.mg_prove_device(a2, dloc)
        acc = {}
        barrier()
        h0, h1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        h0.record()
        for _ in range(steps):
            pr, _ = ctx.mg_prove_device(a2, dloc)
            for k_, v_ in ctx.stage_times().items():
                acc[k_] = acc.get(k_, 0.0) + v_ / steps
        h1.record()
        barrier()
        sh_ms = h0.elapsed_time(h1) / steps
        (sh_ms,) = max_ranks(sh_ms)
        import hashlib
        digs = [None] * world
        dist.all_gather_object(digs, hashlib.sha256(pr).hexdigest())
        same_on_all = len(set(digs)) == 1
        rec = None
        single_ms, parity = None, None
        if rank == 0:
            if k2 != "mimc":
                if pin is not None:
                    pin.free()
                full = L.PinnedBuffer(w2 * n2 * 16)
                full.view().view(np.uint64).reshape(w2, n2, 2)[:] = counter_felts(w2, n2, 0x5EED2000)
                dfull = ctx.upload_trace(full.ptr, w2, n2)
                full.free()
            ref, _ = ctx.prove_device(a2, dfull)
            torch.cuda.synchronize()
            h0.record()
            for _ in range(max(1, steps - 1)):
                ref, _ = ctx.prove_device(a2, dfull)
            h1.record()
            torch.cuda.synchronize()
            single_ms = h0.elapsed_time(h1) / max(1, steps - 1)
            parity = bool(ref == pr and same_on_all)
            rec = {"workload": f"{name}: {d2}", "n_gpus": world, "prove_ms": sh_ms, "single_gpu_ms": single_ms, "speedup": single_ms / sh_ms,
                   "parity": parity, "parity_checked_against": "zkb_prove_device proof of the same trace on rank 0 (byte comparison); all ranks returned the same bytes: %s" % same_on_all,
                   "xchg_exposed_ms": round(acc.get("interpolate", 0.0), 4), "proof_bytes": len(pr), "steps": steps,
                   "stages_ms": {k_: round(v_, 3) for k_, v_ in acc.items() if v_ > 0 and k_ not in ("total", "h2d", "interpolate")}}
        barrier()
        return rec

    headline, sharded_recs = None, None
    if world == 1 and not args.no_headline and not sharded:
        headline = {"mimc": single_proof_case("mimc_2p20", 3, 1), "training": single_proof_case("training_2p20", 3, 1)}
    if world > 1 and not args.no_sharded and not sharded:
        sharded_recs = [sharded_case("mimc_2p20", 3, 1)]
        if world >= 4:
            sharded_recs.append(sharded_case("training_2p20", 2, 1))

    proofs_per_step = 1 if sharded else world * inflight
    if rank == 0:
        # interpolation (K1) and the coset LDE (K2) are interleaved per column group inside the library and timed together
        alg["lde"] += alg["interp"]
        if sharded:  # this rank transforms w/G columns
            alg["lde"] //= world
        lde_ms = max(stages.get("lde", 0.0), 1e-6)
        # per-stage achieved bandwidth against the same peak, for the profile notes
        per_stage = {}
        for st, key in (("lde", "lde"), ("leaf_hash", "leaf"), ("merkle", "merkle"), ("constraints", "ceval"),
                        ("composition", "comp"), ("ood", "ood"), ("deep", "deep"), ("fri", "fri")):
            t_ms = stages.get(st, 0.0)
            per_stage[st] = {"ms": round(t_ms, 4), "alg_GB": round(alg[key] / 1e9, 4),
                             "GBps": round(alg[key] / (t_ms * 1e-3) / 1e9, 1) if t_ms > 0 else None}
        per_stage["grind"] = {"ms": round(stages.get("grind", 0.0), 4)}
        per_stage["queries"] = {"ms": round(stages.get("queries", 0.0), 4)}
        if sharded:  # the part of the NVLink all-to-all that the LDE did not hide (carried in the `interpolate` slot)
            per_stage["xchg_exposed"] = {"ms": round(stages.get("interpolate", 0.0), 4)}
        line = {
            "metric": "stark_proofs_per_sec", "value": proofs_per_step * args.steps / (ms * 1e-3), "unit": "proofs/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong" if sharded else "weak",
            "vs_baseline": None, "dtype": "u128 mod p (f128 field, 4x u32 limbs), u32 BLAKE3", "data": "synthetic",
            "config": {"workload": f"{args.workload}: {desc}", "options": OPTIONS_TEXT, "l2": l2_text(n, w, beta)},
            "run": {"proofs_per_gpu_per_step": inflight, "proof_bytes": main_proof_len, "host_cpus_per_rank": numa or (os.cpu_count() or 1),
                    "parallelism": (f"one proof column-sharded over {world} GPUs: NCCL all-to-all (NVLink transpose) + all-gathers" if sharded
                                    else f"{world} independent proof stream(s), one per GPU, no data-path collective")},
            "prove_ms": ms_latency / args.steps,
            "proof_roofline": {"algorithmic_bytes": alg["total"], "t_hbm_ms": alg["total"] / peak / 1e6,
                               "frac": (alg["total"] / peak / 1e6) / (ms_latency / args.steps)},
            "stages": per_stage,
            "e2e": {"value": proofs_per_step * args.steps / (ms_e2e * 1e-3), "unit": "proofs/s", "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": nbytes * (world if sharded else world * inflight),
                    "d2h_bytes_per_step": main_proof_len * (1 if sharded else world * inflight)},
            "gpu_launches": launches,
            "clocks": sampler.summary(t_wall0, t_wall1),
        }
        line.update(roofline_of(args.workload, n, w_local, beta, lde_ms, alg["lde"], peak, peak_src, sharded))
        # ncu --set full of the shipped k_hash_lde_rows (profiles/r2_ncu_hash_deep_training_2p16_final.txt)
        line["compute_roofline"]["leaf_hash_pipes_pct"] = {"alu": 87.7, "fma_heavy": 65.4, "issue_slots": 82.4}
        if headline:
            # BASELINE.json `metric`, first half: prove time of a 2^20-ROW TRACE on one B200, measured in this same run
            line["headline_2p20"] = headline
        if sharded_recs:
            # BASELINE.json configs[4]: one large proof column-sharded over the ranks, checked against the single-GPU proof
            line["sharded"] = sharded_recs[0]
            if len(sharded_recs) > 1:
                line["sharded_training_2p20"] = sharded_recs[1]
        if world == 1 and not args.no_cpu_baseline:
            from oracle import pyoracle as O
            cores = os.cpu_count() or 1
            O.set_threads(cores)
            t0 = time.time()
            ref, ts_ref, secs = O.prove(air_dict, tb_main)
            dt = time.time() - t0
            line["cpu_baseline"] = {"value": 1.0 / dt, "unit": "proofs/s", "ms_per_proof": dt * 1e3, "cores": cores, "kind": "port",
                                    "sample": "1 full proof of the same workload (C++ restatement of Winterfell's CPU prover: std::thread over columns / rows on "
                                              "all host cores, portable scalar BLAKE3 - upstream uses the SIMD blake3 crate; not Winterfell itself)",
                                    "proof_identical_to_gpu": ref == proof}
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, last_step)
        emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
