"""torchrun worker: column-sharded proofs across the GPUs of one node must equal the single-GPU proof byte for byte.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port P tests/mg_worker.py [cases]

cases: a JSON list of [kind, w, n, blowup] or [kind, w, n, blowup, folding] with kind "mimc" or "training"; FRI folding 16 when
omitted.

torch.distributed (gloo) is only the control plane here (NCCL id broadcast, result gathering); the data-path collectives
run inside libzkb200.so on its own NCCL communicator."""
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import zk_stark_project_b200 as Z  # noqa: E402
from zk_stark_project_b200 import lib as L  # noqa: E402
from tests import common as T  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    dist.init_process_group("gloo")
    ndev = torch.cuda.device_count()
    if ndev < world:
        # more ranks than GPUs (the sharded path tested on one GPU): NCCL refuses two ranks of one host on one device, so each
        # rank presents its own host id and the ranks exchange data over NCCL's socket transport
        os.environ["NCCL_HOSTID"] = f"zkb-mg-worker-rank-{rank}"
    ctx = L.Context(local % ndev)
    ids = [L.mg_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    ctx.mg_init(rank, world, ids[0])
    cases = json.loads(sys.argv[1]) if len(sys.argv) > 1 else [["mimc", 64, 4096, 8], ["mimc", 16, 256, 8], ["training", 128, 1024, 16],
                                                                ["training", 240, 512, 16], ["mimc", 24, 256, 8], ["mimc", 64, 1 << 16, 8]]
    results = []
    for case in cases:
        kind, w, n, blowup, folding = (case + [16])[:5]
        opts = T.options(blowup, 40, 16, folding)
        if kind == "mimc":
            rc = Z.get_round_constants()
            raw = ctx.mimc_trace([j + 1 for j in range(w)], n, rc)
            data = np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2).copy()
            get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
            air = Z.MimcAir(w, n, Z.MimcInputs([get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)]), opts).describe()
        else:
            air, data = T.training_case(w, n, opts, 99)
        prepared = ctx.prepare(air)
        t0 = time.time()
        single, ts1 = ctx.prove_host(prepared, data.ctypes.data)
        t1 = time.time()
        wl = w // world
        mine = np.ascontiguousarray(data[rank * wl:(rank + 1) * wl])
        dist.barrier()
        t2 = time.time()
        sharded, ts2 = ctx.mg_prove_host(prepared, mine.ctypes.data, world)
        t3 = time.time()
        ok = sharded == single
        results.append(dict(case=case, ok=ok, roots_equal=bytes(ts1.trace_root) == bytes(ts2.trace_root), z_equal=bytes(ts1.z) == bytes(ts2.z),
                            fri_layers=int(ts2.n_fri_layers), single_ms=(t1 - t0) * 1e3, sharded_ms=(t3 - t2) * 1e3, proof_len=len(sharded)))
    gathered = [None] * world
    dist.all_gather_object(gathered, results)
    if rank == 0:
        print(json.dumps(gathered))
        bad = [r for rr in gathered for r in rr if not r["ok"]]
        if bad:
            print("MISMATCH", bad)
            sys.exit(1)
        print("mg ok")
    dist.destroy_process_group()


if __name__ == "__main__":
    main()
