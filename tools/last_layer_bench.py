#!/usr/bin/env python
"""The last GCN layer of the per-batch call on one GPU at config-5 scale: the full sparse product over every row against
the product over the rows a 65,536-pair batch scores (graph.CsrSubset), and the cost of building that subset.

Same graph, batch and width as bench.py (seed 42 generator, ids from RandomState(1234)).  Prints one JSON line: the
card and its power limit, ms per launch (CUDA events, mean and min of the repeats after a warm-up) for fp32 and bf16
operands, the subset build's ms (host clock around it: it ends in a device-to-host copy of its counts), and the edges
and rows each launch processes.  It also checks that the subset launch writes the needed rows with the full launch's
bits."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from bench import DIM, PAIR_BATCH, SCALES  # noqa: E402
from deep_cbrs_amar_renaissance_b200 import ops  # noqa: E402
from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph  # noqa: E402


def events(fn, reps):
    fn()
    torch.cuda.synchronize()
    ms = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    return {"mean": float(np.mean(ms)), "min": float(np.min(ms)), "reps": reps}


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        return q
    except Exception as e:  # the timing stands without it; the line says why the card is not named
        return "unavailable: %s" % e


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", default="c5", choices=sorted(SCALES))
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    n_users, n_items, n_edges = SCALES[args.scale]
    n = n_users + n_items
    row, col = ops.synth_bipartite(n_users, n_items, n_edges, 42, dev, scatter_items=True)
    graph = DeviceGraph(row, col, None, n)
    del row, col
    csr = graph.norm
    graph.release_coo()
    rng = np.random.RandomState(1234)
    u = torch.from_numpy(rng.randint(0, n_users, size=PAIR_BATCH)).to(dev)
    i = torch.from_numpy(rng.randint(0, n_items, size=PAIR_BATCH) + n_users).to(dev)
    ids = torch.cat([u, i])

    gen = torch.Generator(dev).manual_seed(0)
    z = torch.randn(n, DIM, device=dev, generator=gen) * 0.05
    bias = torch.randn(DIM, device=dev, generator=gen) * 0.01
    out_full = torch.empty(n, DIM, device=dev)
    out_sub = torch.zeros(n, DIM, device=dev)

    build = []
    for _ in range(args.reps + 1):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sub = csr.row_subset(ids)
        torch.cuda.synchronize()
        build.append((time.perf_counter() - t0) * 1e3)
    build = build[1:]

    res = {"card": card(), "scale": args.scale, "pairs": PAIR_BATCH, "d": DIM,
           "full": {"edges": csr.nnz, "rows": csr.n_rows, "chunks": csr.chunks["n_chunks"], "heavy_rows": csr.chunks["n_heavy"]},
           "subset": {"edges": sub.nnz, "rows": sub.n_needed, "chunks": sub.chunks["n_chunks"],
                      "heavy_rows": sub.chunks["n_heavy"], "edge_share": sub.nnz / csr.nnz},
           "subset_build_ms": {"mean": float(np.mean(build)), "min": float(np.min(build)), "reps": args.reps}}
    for name, x in (("fp32", z), ("bf16", z.to(torch.bfloat16))):
        res["full"][name + "_ms"] = events(lambda: ops.spmm(csr, x, out_full, bias=bias, relu=True), args.reps)
        res["subset"][name + "_ms"] = events(lambda: ops.spmm(sub, x, out_sub, bias=bias, relu=True), args.reps)
        need = torch.unique(ids)
        res["subset"][name + "_rows_bit_identical"] = bool(torch.equal(out_full[need], out_sub[need]))
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
