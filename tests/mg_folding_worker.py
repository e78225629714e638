"""torchrun worker: column-sharded proofs at a chosen FRI folding factor must equal the single-GPU proof byte for byte.

  python -m torch.distributed.run --nnodes=1 --nproc-per-node G --master-addr 127.0.0.1 --master-port P tests/mg_folding_worker.py \
      '[["mimc", w, n, blowup, folding], ["training", w, n, blowup, folding], ...]'

As in tests/mg_worker.py, torch.distributed (gloo) is only the control plane; the data-path collectives run inside libzkb200.so."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

import zk_stark_project_b200 as Z  # noqa: E402
from zk_stark_project_b200 import lib as L  # noqa: E402
from zk_stark_project_b200 import synthetic as S  # noqa: E402


def main():
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ.get("LOCAL_RANK", "0"))
    dist.init_process_group("gloo")
    ndev = torch.cuda.device_count()
    if ndev < world:
        # more ranks than GPUs: each rank presents its own host id so that NCCL uses its socket transport between them
        os.environ["NCCL_HOSTID"] = f"zkb-mg-folding-worker-rank-{rank}"
    ctx = L.Context(local % ndev)
    ids = [L.mg_unique_id() if rank == 0 else None]
    dist.broadcast_object_list(ids, src=0)
    ctx.mg_init(rank, world, ids[0])
    results = []
    for kind, w, n, blowup, folding in json.loads(sys.argv[1]):
        opts = Z.ProofOptions(40, blowup, 16, Z.FieldExtension.NONE, folding, 7)
        if kind == "mimc":
            raw = ctx.mimc_trace([j + 1 for j in range(w)], n, Z.get_round_constants())
            data = np.frombuffer(raw, dtype=np.uint64).reshape(w, n, 2).copy()
            get = lambda c, r: int(data[c, r, 0]) | (int(data[c, r, 1]) << 64)
            air = Z.MimcAir(w, n, Z.MimcInputs([get(j, 0) for j in range(w)], [get(j, n - 1) for j in range(w)]), opts).describe()
        else:
            data = S.random_felts(w * n, 99).reshape(w, n, 2)
            air = S.synthetic_training_air(n, opts, data)
        prepared = ctx.prepare(air)
        single, ts1 = ctx.prove_host(prepared, data.ctypes.data)
        wl = w // world
        mine = np.ascontiguousarray(data[rank * wl:(rank + 1) * wl])
        dist.barrier()
        sharded, ts2 = ctx.mg_prove_host(prepared, mine.ctypes.data, world)
        results.append(dict(case=[kind, w, n, blowup, folding], ok=sharded == single, fri_layers=int(ts2.n_fri_layers), proof_len=len(sharded)))
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
