#!/usr/bin/env python
"""Cost of the FRI folding factor: for F in {2, 4, 8, 16}, single-proof latency of three workloads with the reference options
(40 queries, grinding 21, remainder degree <= 7) except the folding factor.

    python tools/fri_folding_sweep.py [--proofs 10] [--warmup 3] [--out profiles/rN_fri_folding_sweep.json]

Workloads: BASELINE.json configs[1] (training AIR 240 x 2^16, blowup 16), MiMC 64 x 2^20 (blowup 8) and the aggregation AIR over
16 updates (blowup 16).  Every proof is device-resident (zkb_prove_device, the trace uploaded once) and one proof is in flight at a
time.  Per (workload, F) the script reports the median wall time of `--proofs` warm proofs (the call returns after the device
finished and the proof is assembled), the median FRI stage time (zkb_last_stage_times().fri, CUDA events), the kernel launches per
proof (zkb_kernel_launches delta), the FRI layer count and the proof size.  The GPU name and power limit are read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

FACTORS = (2, 4, 8, 16)


def gpu_info():
    import torch
    out = {"torch_device_name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in q.split(",")]
        out.update(name=name, power_limit=power, max_sm_clock=clock)
    except Exception as e:  # the numbers stay usable, but say that the power limit is unknown
        out.update(power_limit=f"not read ({e})")
    return out


def workloads(ctx, folding):
    """(name, AIR description, column-major (w, n, 2) host trace) for each workload at folding factor `folding`."""
    import zk_stark_project_b200 as Z
    from zk_stark_project_b200 import synthetic as S
    opts = lambda beta: Z.ProofOptions(40, beta, 21, Z.FieldExtension.NONE, folding, 7)
    n, w = 1 << 16, 240
    data = S.random_felts(w * n, 0x5EED0002).reshape(w, n, 2)
    yield "training_2p16_x240_b16", S.synthetic_training_air(n, opts(16), data), data
    n, w = 1 << 20, 64
    data = np.frombuffer(ctx.mimc_trace([j + 1 for j in range(w)], n, Z.get_round_constants()), dtype=np.uint64).reshape(w, n, 2)
    get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
    air = Z.MimcAir(w, n, Z.MimcInputs([get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)]), opts(8)).describe()
    yield "mimc_2p20_x64_b8", air, data
    from tests import common as T
    p = T.aggregation_prover(16, opts(16))
    tr = p.build_trace()
    yield "aggregation_16_updates", p.describe(tr), np.ascontiguousarray(tr.data)


def measure(ctx, air, data, proofs, warmup):
    from zk_stark_project_b200 import lib as L
    w, n = data.shape[0], data.shape[1]
    pin = L.PinnedBuffer(w * n * 16)
    pin.view()[:] = np.ascontiguousarray(data).reshape(-1).view(np.uint8)
    d_trace = ctx.upload_trace(pin.ptr, w, n)
    desc = ctx.prepare(air)
    for _ in range(warmup):
        ctx.prove_device(desc, d_trace)
    wall, fri, first = [], [], None
    l0 = ctx.launches()
    for _ in range(proofs):
        t0 = time.perf_counter()
        proof, ts = ctx.prove_device(desc, d_trace)
        wall.append((time.perf_counter() - t0) * 1e3)
        fri.append(ctx.stage_times()["fri"])
        first = first or proof
        if proof != first:
            raise RuntimeError("proofs of the same trace differ")
    launches = (ctx.launches() - l0) / proofs
    pin.free()
    fri = [t for t in fri if t > 0]
    return {"prove_ms_median": statistics.median(wall), "prove_ms_min": min(wall), "fri_ms_median": statistics.median(fri) if fri else None,
            "launches_per_proof": launches, "fri_layers": int(ts.n_fri_layers), "proof_bytes": len(first)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--proofs", type=int, default=10, help="timed proofs per (workload, folding factor); at least 10")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", help="write the results as JSON here")
    ap.add_argument("--eager", action="store_true", help="ZKB_GRAPH=0: no CUDA-graph replay of small proofs, so that the aggregation "
                    "proofs record their stage times too (a replayed proof records none: its fri_ms is reported as null)")
    args = ap.parse_args()
    if args.proofs < 10:
        ap.error("--proofs must be at least 10")
    if args.eager:
        os.environ["ZKB_GRAPH"] = "0"
    import torch
    from zk_stark_project_b200 import lib as L
    if not torch.cuda.is_available():
        raise SystemExit("fri_folding_sweep.py needs a CUDA device")
    ctx = L.Context(0)
    result = {"gpu": gpu_info(), "options": "40 queries, grinding 21, remainder degree <= 7, FRI folding F", "proofs": args.proofs,
              "warmup": args.warmup, "graph_replay": not args.eager, "rows": []}
    for folding in FACTORS:
        for name, air, data in workloads(ctx, folding):
            row = dict(workload=name, folding=folding, **measure(ctx, air, data, args.proofs, args.warmup))
            result["rows"].append(row)
            print(json.dumps(row), flush=True)
    g = result["gpu"]
    print(f"\n{g.get('name', g['torch_device_name'])}, power limit {g.get('power_limit')}")
    print(f"{'workload':26s} {'F':>3s} {'layers':>6s} {'prove ms':>9s} {'FRI ms':>8s} {'launches':>8s} {'proof B':>8s}")
    for r in result["rows"]:
        print(f"{r['workload']:26s} {r['folding']:3d} {r['fri_layers']:6d} {r['prove_ms_median']:9.3f} {r['fri_ms_median'] or float('nan'):8.3f} "
              f"{r['launches_per_proof']:8.0f} {r['proof_bytes']:8d}")
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(result, f, indent=1)
    ctx.close()


if __name__ == "__main__":
    main()
