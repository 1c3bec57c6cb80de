"""Multi-GPU parity (run on the GPU box):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29511 tests/multi_gpu_check.py
Every rank builds the same graph and weights, runs the propagation once unpartitioned and once
row-partitioned, and requires the two to be BIT-identical for all four layer families, ragged and even blocks,
peer stores / NCCL, both GCN transform kernels, row-major and column-blocked schedules; then checks
user-sharded catalog top-k.  The body lives in deep_cbrs_amar_renaissance_b200/selfcheck.py because bench.py runs
the same check before timing whenever WORLD_SIZE > 1 (its JSON line carries "partition_parity")."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from deep_cbrs_amar_renaissance_b200.selfcheck import partition_parity  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res = partition_parity(log=lambda m: print(m, flush=True))
    if rank == 0:
        print(json.dumps({"partition_parity": res, "world_size": dist.get_world_size()}), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if not res["bit_identical"]:
        raise SystemExit("partitioned result differs: %s" % res["failures"])


if __name__ == "__main__":
    main()
