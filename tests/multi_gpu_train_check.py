"""Multi-GPU training parity (run on a box with at least two GPUs):
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1 --master-port 29512 tests/multi_gpu_train_check.py
Every rank builds the same graph, weights and batches and runs three optimiser steps once unpartitioned and once
row-partitioned; losses, every weight (the embedding table included) and the Adam moments must be BIT-identical for
GCN, RGCN, LightGCN, GraphSage, GAT and the hybrid GCN, under peer stores and the NCCL all-gather, even and
edge-balanced cuts, row-major and column-blocked schedules.  The body is selfcheck.training_parity."""
import json
import os
import sys

import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from deep_cbrs_amar_renaissance_b200.selfcheck import training_parity  # noqa: E402


def main():
    rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    res = training_parity(log=lambda m: print(m, flush=True))
    if rank == 0:
        print(json.dumps({"training_parity": res, "world_size": dist.get_world_size()}), flush=True)
    dist.barrier()
    dist.destroy_process_group()
    if not res["bit_identical"]:
        raise SystemExit("partitioned training differs: %s" % res["failures"])


if __name__ == "__main__":
    main()
