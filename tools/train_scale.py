#!/usr/bin/env python
"""One optimiser step of BasicGCN (3 x 128, concatenation, BasicRS [48,48]/[64,64]) on a scaled synthetic graph: shows the
explicit backward kernels beyond MovieLens size.  Prints one JSON line (ms per step, loss trajectory on a fixed batch,
the sparse kernels' time per step from device events, the GPU name and power limit).

    python tools/train_scale.py [c5-tenth|c5-hundredth|c5-fifth]
    torchrun --nproc_per_node N tools/train_scale.py [scale] --gpus N    # row-partitioned step on N GPUs (rank 0 prints)"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from deep_cbrs_amar_renaissance_b200 import ops  # noqa: E402
from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph  # noqa: E402
from deep_cbrs_amar_renaissance_b200.keras_like import set_seed  # noqa: E402
from deep_cbrs_amar_renaissance_b200.models import basic  # noqa: E402


def _gpu_info(index):
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", str(index)],
                       capture_output=True, text=True)
    return q.stdout.strip() if q.returncode == 0 else "unavailable: " + q.stderr.strip()


def _sparse_ms(model, ud, idv, y, steps=3):
    """the sparse kernels' device time per step (CUDA events around every SpMM launch), in a pass of its own"""
    ops.PROFILE_ON, ops.PROFILE[:] = True, []
    try:
        for _ in range(steps):
            model.train_on_batch((ud, idv), y)
        torch.cuda.synchronize()
        return sum(e0.elapsed_time(e1) for kind, e0, e1, _ in ops.PROFILE if kind == "spmm") / steps
    finally:
        ops.PROFILE_ON, ops.PROFILE[:] = False, []


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("scale", nargs="?", default="c5-tenth")
    ap.add_argument("--gpus", type=int, default=1, help="ranks of the row partition (run under torchrun with as many)")
    args = ap.parse_args()
    scale = args.scale
    n_users, n_items, n_edges = {"c5-tenth": (1_000_000, 100_000, 100_000_000), "c5-hundredth": (100_000, 10_000, 10_000_000),
                                 "c5-fifth": (2_000_000, 200_000, 200_000_000)}[scale]
    batch = 65536
    rank, local = 0, 0
    if args.gpus > 1:
        import torch.distributed as dist
        if int(os.environ.get("WORLD_SIZE", "1")) != args.gpus:
            raise SystemExit("--gpus %d needs torchrun --nproc_per_node %d" % (args.gpus, args.gpus))
        rank, local = int(os.environ["RANK"]), int(os.environ["LOCAL_RANK"])
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    row, col = ops.synth_bipartite(n_users, n_items, n_edges, 42, dev)
    graph = DeviceGraph(row, col, None, n_users + n_items)
    del row, col
    set_seed(42)
    model = basic.BasicGCN(graph, n_hiddens=[128] * 3, embedding_dim=128, dense_units=[48, 48], clf_units=[64, 64],
                           final_node="concatenation", l2_regularizer=1e-6)
    nnz = graph.norm.nnz
    part = None
    if args.gpus > 1:
        from deep_cbrs_amar_renaissance_b200.distributed import RowPartition
        part = RowPartition([n_users, n_items], balance_rowptr=graph.norm.rowptr,
                            balance_min_len=graph.norm.blocking[1]).attach(model.gnn.gnn_layers)
    graph.release_coo()
    model.compile(loss="binary_crossentropy", optimizer={"learning_rate": 1e-3})
    rng = np.random.RandomState(0)
    u = rng.randint(0, n_users, size=batch)
    i = rng.randint(0, n_items, size=batch) + n_users
    y = ((u + i) % 2).astype(np.int64)  # a learnable parity rule
    ud, idv = torch.from_numpy(u).to(dev), torch.from_numpy(i).to(dev)
    losses = []
    for _ in range(3):
        loss, _ = model.train_on_batch((ud, idv), y)
        losses.append(float(loss.item()))
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    steps = 10
    ops.LAUNCHES = 0
    e0.record()
    for _ in range(steps):
        loss, correct = model.train_on_batch((ud, idv), y)
    e1.record()
    torch.cuda.synchronize()
    losses.append(float(loss.item()))
    ms = e0.elapsed_time(e1) / steps
    launches = ops.LAUNCHES / steps
    sparse = _sparse_ms(model, ud, idv, y)
    rank_sparse = [sparse]
    if part is not None:
        import torch.distributed as dist
        rank_sparse = [None] * args.gpus
        dist.all_gather_object(rank_sparse, sparse)
    if rank == 0:
        # forward + backward each run 3 sparse passes over nnz edges
        print(json.dumps({"model": "BasicGCN 3x128", "scale": scale, "gpus": args.gpus, "gpu": _gpu_info(local),
                          "nodes": n_users + n_items, "nnz_a_hat": nnz, "batch": batch, "train_step_ms": ms,
                          "rank_sparse_ms_per_step": rank_sparse, "launches_per_step": launches,
                          "edges_per_s_fwd_plus_bwd": 6 * nnz / (ms * 1e-3), "loss_first_3": losses[:3],
                          "loss_after_13": losses[-1], "accuracy_last": float(correct.item()) / batch}), flush=True)
    if part is not None:
        part.close()
        dist.destroy_process_group()
    assert np.isfinite(losses).all() and losses[-1] < losses[0]


if __name__ == "__main__":
    main()
