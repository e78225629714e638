#!/usr/bin/env python
"""Batch verification on the GPU (zkb_verify_batch) against the CPU verifier, with the reference options (40 queries, blowup 16,
grinding 21, folding 16, remainder degree <= 7).

    python tools/verify_sweep.py [--reps 5] [--out profiles/r7_verify_sweep.json]

Workloads: aggregation over 16 updates (32 x 120), training bs = 1 (128 x 240), bs = 50 (8192 x 240), 2^16 x 240 (BASELINE.json
configs[1]) and MiMC 64 x 2^14.  Per workload four proofs are made on the GPU and cycled into batches of 1, 16 and 256.  Per
(workload, batch) the script reports:
  - gpu_ms: median host wall time of the whole zkb_verify_batch call (it ends in a stream synchronisation), and per proof; the
    AIR descriptions are marshalled once, outside the timed call, on both sides;
  - h2d_bytes: what one call copies host to device (zkb_h2d_bytes delta: the staging buffer with the proofs' sections, alignment
    padding, per-proof AIR tables and Merkle nodes, plus the Merkle / evaluation plan), next to the proofs' own bytes;
  - launches: kernel launches of one call (zkb_kernel_launches delta);
  - cpu_1core_ms: the oracle's verifier (orc_verify, scalar BLAKE3) over the batch on one host thread;
  - cpu_all_ms: the same with one host thread per core over the proofs (ctypes releases the GIL), with the core count.
With ZKB_HOST_PROFILE=1 in the environment the library prints every call's host and device phases on stderr.
The GPU name and power limit are read in the same run."""
import argparse
import concurrent.futures as cf
import ctypes as C
import json
import os
import statistics
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

from fri_folding_sweep import gpu_info  # noqa: E402

BATCHES = (1, 16, 256)


def workloads(oracle):
    import zk_stark_project_b200 as Z
    from tests import common as T
    ref = Z.ProofOptions.reference()

    def prover(p):
        tr = p.build_trace()
        return p.describe(tr), np.ascontiguousarray(tr.data)

    def synthetic(w, n, seed):
        data = T.random_felts(w * n, seed).reshape(w, n, 2)
        return T.synthetic_training_air(n, ref, data), np.ascontiguousarray(data)

    def mimc(w, n):
        p = T.mimc_prover(w, n, ref)
        raw = oracle.mimc_trace(p.seeds, n, p.rc)
        tr = Z.TraceTable(np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2))
        return p.describe(tr), np.ascontiguousarray(tr.data)

    return {
        "aggregation 16 updates (32 x 120)": [prover(T.aggregation_prover(16, ref, seed=0x5EED0300 + k)) for k in range(4)],
        "training bs=1 (128 x 240)": [prover(T.training_prover(1, ref, seed=0x5EED0400 + k)) for k in range(4)],
        "training bs=50 (8192 x 240)": [synthetic(240, 8192, 0x5EED0500 + k) for k in range(4)],
        "training 2^16 x 240": [synthetic(240, 1 << 16, 0x5EED0600 + k) for k in range(4)],
        "mimc 64 x 2^14": [mimc(64, 1 << 14)] * 4,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r7_verify_sweep.json"))
    args = ap.parse_args()
    from zk_stark_project_b200 import lib as L
    from oracle import pyoracle as O
    O.build()
    O.set_threads(1)
    info = gpu_info()
    cores = os.cpu_count() or 1
    ctx = L.Context(0)
    rows = []
    for name, cases in workloads(O).items():
        made = []
        for k, (air, data) in enumerate(cases):
            proof, _ = ctx.prove_host(air, data.ctypes.data, 0)
            made.append((air, proof))
        descs = [(L.Context.prepare(a), O.make_desc(a), p) for a, p in made]

        def cpu_verify(k):
            _, d, p = descs[k % len(descs)]
            ts, err = O.Transcript(), C.create_string_buffer(512)
            assert O.lib().orc_verify(C.byref(d), p, C.c_uint64(len(p)), C.byref(ts), err, C.c_uint64(512)) == 0, err.value

        for b in BATCHES:
            airs = [descs[i % len(descs)][0] for i in range(b)]
            proofs = [made[i % len(made)][1] for i in range(b)]
            verdicts, _ = ctx.verify_batch(airs, proofs)   # warm-up: buffers, module load
            assert verdicts == [0] * b, verdicts
            times, launches, h2d = [], None, None
            for _ in range(args.reps):
                l0, b0 = ctx.launches(), ctx.h2d_bytes()
                t0 = time.perf_counter()
                ctx.verify_batch(airs, proofs)
                times.append((time.perf_counter() - t0) * 1e3)
                launches, h2d = ctx.launches() - l0, ctx.h2d_bytes() - b0
            gpu_ms = statistics.median(times)
            t0 = time.perf_counter()
            for k in range(b):
                cpu_verify(k)
            cpu1 = (time.perf_counter() - t0) * 1e3
            with cf.ThreadPoolExecutor(cores) as ex:
                t0 = time.perf_counter()
                list(ex.map(cpu_verify, range(b)))
                cpu_all = (time.perf_counter() - t0) * 1e3
            row = dict(workload=name, batch=b, proof_bytes=len(proofs[0]), gpu_ms=round(gpu_ms, 3), gpu_ms_per_proof=round(gpu_ms / b, 4),
                       gpu_ms_all_reps=[round(t, 3) for t in times], proof_bytes_total=sum(len(p) for p in proofs), h2d_bytes=h2d, launches=launches,
                       cpu_1core_ms=round(cpu1, 3), cpu_all_cores_ms=round(cpu_all, 3), cpu_cores=cores)
            rows.append(row)
            print(json.dumps(row), flush=True)
    out = dict(gpu=info, options="reference (40 queries, blowup 16, grinding 21, folding 16, remainder degree 7)", rows=rows)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps(info))


if __name__ == "__main__":
    main()
