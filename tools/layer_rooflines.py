#!/usr/bin/env python
"""Per-kernel throughput of every propagation layer family at scale (run under gpurun; writes one JSON line per
layer): GCN, LightGCN, GraphSage(mean), GAT on the scaled synthetic bipartite graph, D = 128, fp32, plus the device
graph build.  `achieved` = SURVEY 8d algorithmic bytes / CUDA-event time, against MEASURED_PEAKS.json."""
import json
import os
import sys
import time

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)
from deep_cbrs_amar_renaissance_b200 import _lib as L  # noqa: E402
from deep_cbrs_amar_renaissance_b200 import ops  # noqa: E402
from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph  # noqa: E402


def timeit(fn, n=5, warm=2):
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(n):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / n


def main():
    scale = sys.argv[1] if len(sys.argv) > 1 else "c5-tenth"
    n_users, n_items, n_edges = {"c5": (10_000_000, 1_000_000, 1_000_000_000), "c5-tenth": (1_000_000, 100_000, 100_000_000),
                                 "c5-fifth": (2_000_000, 200_000, 200_000_000)}[scale]
    d = 128
    peak = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))["hbm_gbs"]
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(0)
    n = n_users + n_items
    t0 = time.perf_counter()
    row, col = ops.synth_bipartite(n_users, n_items, n_edges, 42, dev)
    torch.cuda.synchronize()
    t_gen = time.perf_counter() - t0
    g = DeviceGraph(row, col, None, n)
    t0 = time.perf_counter()
    norm = g.norm
    torch.cuda.synchronize()
    t_norm = time.perf_counter() - t0
    t0 = time.perf_counter()
    raw = g.raw
    torch.cuda.synchronize()
    t_raw = time.perf_counter() - t0
    print(json.dumps({"op": "graph build", "scale": scale, "coo_entries": 2 * n_edges, "synth_s": t_gen, "norm_view_s": t_norm,
                      "raw_view_s": t_raw, "entries_per_s_norm": 2 * n_edges / t_norm}), flush=True)
    g.release_coo()
    del row, col
    x = torch.randn(n, d, device=dev) * 0.05
    w = torch.randn(d, d, device=dev) * 0.05
    w2 = torch.randn(2 * d, d, device=dev) * 0.05
    bias = torch.zeros(d, device=dev)
    a_s, a_n = torch.randn(d, device=dev) * 0.05, torch.randn(d, device=dev) * 0.05
    out = torch.empty(n, d, device=dev)
    s = 4

    def report(op, ms, nnz, alg_bytes, extra=None):
        line = {"op": op, "scale": scale, "d": d, "nnz": nnz, "ms": ms, "edges_per_s": nnz / (ms * 1e-3),
                "algorithmic_bytes": alg_bytes, "achieved_GBps": alg_bytes / (ms * 1e-3) / 1e9, "peak_GBps": peak,
                "frac": alg_bytes / (ms * 1e-3) / 1e9 / peak}
        line.update(extra or {})
        print(json.dumps(line), flush=True)

    # GCN / LightGCN sparse step: nnz*(4+4+D*s) + N*(D*s+8)
    ms = timeit(lambda: ops.spmm(norm, x, out, bias=bias, relu=True))
    report("GCN/LightGCN SpMM (A_hat, weighted)", ms, norm.nnz, norm.nnz * (8 + d * s) + n * (d * s + 8))
    # GraphSage mean aggregate: nnz*(4+F*s) + N*(F*s+8)   (values ignored)
    ms = timeit(lambda: ops.spmm(raw, x, out, agg=L.AGG_MEAN))
    report("GraphSage mean aggregate (raw A)", ms, raw.nnz, raw.nnz * (4 + d * s) + n * (d * s + 8))
    # GraphSage dense part: [x || agg] W, l2norm, relu: N*(2F+H)*s bytes, 2*N*2F*H flop
    agg = out.clone()
    out2 = torch.empty(n, d, device=dev)
    ms = timeit(lambda: ops.dense(x, w2, bias, "relu", x2=agg, rowop=L.ROWOP_L2NORM, out=out2))
    report("GraphSage [x||agg]W + l2norm + relu (dense, fp32 FFMA)", ms, 0, n * 3 * d * s,
           {"tflops": 2 * n * 2 * d * d / (ms * 1e-3) / 1e12})
    ms = timeit(lambda: ops.sage_dense(x, agg, w2, bias, "relu", n, out=out2))
    report("GraphSage [x||agg]W + l2norm + relu (tcgen05, 3xTF32, two products: the path the layer takes at this scale)", ms, 0,
           n * 3 * d * s, {"tflops_fp32_equivalent": 2 * n * 2 * d * d / (ms * 1e-3) / 1e12})
    # GCN transform
    ms = timeit(lambda: ops.dense(x, w, out=out2))
    report("GCN transform X W (dense, fp32 FFMA)", ms, 0, n * 2 * d * s, {"tflops": 2 * n * d * d / (ms * 1e-3) / 1e12})
    ms = timeit(lambda: ops.dense_tf32x3(x, w, out=out2))
    report("GCN transform X W (tcgen05, 3xTF32, TMA: the kernel the layers use at this scale)", ms, 0, n * 2 * d * s,
           {"tflops_fp32_equivalent": 2 * n * d * d / (ms * 1e-3) / 1e12})
    ms = timeit(lambda: ops.gat_transform(x, w, a_s, a_n, n, out=out2))
    report("GAT transform X W + attention logits (tcgen05, 3xTF32)", ms, 0, n * 2 * d * s + 8 * n)
    ms = timeit(lambda: ops.dense(x, w, rowop=L.ROWOP_ATTN, a_self=a_s, a_neigh=a_n, out=out2))
    report("GAT transform X W + attention logits (dense, fp32 FFMA)", ms, 0, n * 2 * d * s + 8 * n)
    # GAT: transform + logits, then fused edge softmax + aggregate: nnz*(4+4+H*s) + N*(H*s+16)
    z, p, q = ops.dense(x, w, rowop=L.ROWOP_ATTN, a_self=a_s, a_neigh=a_n)
    ms = timeit(lambda: ops.gat(raw, z, p, q, out, bias=bias, relu=True))
    report("GAT fused score+softmax+aggregate (raw A + self loops)", ms, raw.nnz + n, raw.nnz * (8 + d * s) + n * (d * s + 16))
    # bf16 operand storage
    z16 = x.to(torch.bfloat16)
    ms = timeit(lambda: ops.spmm(norm, z16, out, bias=bias, relu=True))
    report("GCN SpMM, bf16 operand", ms, norm.nnz, norm.nnz * (8 + d * 2) + n * (d * s + 8))


if __name__ == "__main__":
    main()
