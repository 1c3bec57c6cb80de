#!/usr/bin/env python
"""Micro-benchmark of the chained tensor-core hybrid catalog scorers on random hoisted tables (run on a B200):
users x items, CUDA events, one warm-up, median of --reps runs.
  --precision bf16: cbrs_score_hybrid_topk_bf16, 40,960 tensor FLOP per pair (4 products of 64 x 64 plus the 128 x 64
                    first classifier layer counted as two);
  --precision fp32: cbrs_score_hybrid_topk_tf32x3, the same products as 3xTF32 = 122,880 tensor FLOP per pair.
With --generic (default shapes only), the same run also times the generic pair pipeline that fp32 used before the
3xTF32 kernel: recommend_top_k(fused=False) of a feature-based HybridBertGCN (econfigs/hybrid-gnn.yaml shapes) at
6,040 x 3,706, propagation cached, next to recommend_top_k(precision='fp32') of the same model.

    python tools/hybrid_tc_bench.py [users items] [--precision {bf16,fp32}] [--exclude {none,empty,ml1m,zipf}]
                                    [--reps R] [--generic]

--exclude other than none alternates runs without and with per-user exclusion lists (the arms of tools/score_bench.py)
and reports both arms and the overhead."""
import argparse
import json
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deep_cbrs_amar_renaissance_b200 import ops  # noqa: E402
from tools.score_bench import alternate, arm_summary, exclusion_lists  # noqa: E402


FLOP_PER_PAIR = {"bf16": 40960, "fp32": 122880}
KERNEL = {"bf16": "score_hybrid_tc_kernel", "fp32": "score_hybrid_tf32_kernel"}


def generic_vs_fused(reps):
    """recommend_top_k of one feature-based HybridBertGCN at MovieLens-1M shape: generic pipeline vs fused fp32 kernel"""
    import numpy as np
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import hybrid
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
    from tools.score_bench import time_ms
    n_users, n_items, k = 6040, 3706, 10
    set_seed(42)
    adj = small_graph(n_users, n_items, 572000, seed=42)
    model = hybrid.HybridBertGCN(adj, n_hiddens=[16, 16], n_layers=2, embedding_dim=16,
                                 dense_units=[[48, 48], [256, 64], [64, 64]], clf_units=[64, 64], feature_based=True)
    rng = np.random.RandomState(0)
    model.set_content_table((rng.standard_normal((n_users + n_items, 768)) * 0.5).astype(np.float32))
    model((rng.randint(0, n_users, 64), rng.randint(0, n_items, 64) + n_users))
    model.cache_propagation = True
    model.propagate()
    out = {}
    for name, kw in (("generic", dict(fused=False)), ("fused_tf32x3", dict(precision="fp32"))):
        ms = sorted(time_ms(lambda: model.recommend_top_k(n_users, n_items, k, **kw), iters=1) for _ in range(reps))
        out[name] = {"ms": ms[len(ms) // 2], "ms_min": ms[0], "ms_max": ms[-1], "pairs_per_s": n_users * n_items / ms[len(ms) // 2] * 1e3}
    gi, gv = model.recommend_top_k(n_users, n_items, k, fused=False)
    fi, fv = model.recommend_top_k(n_users, n_items, k, precision="fp32")
    return {"case": "HybridBertGCN feature-based recommend_top_k, propagation cached", "users": n_users, "items": n_items,
            "k": k, "reps": reps, **out, "speedup": out["generic"]["ms"] / out["fused_tf32x3"]["ms"],
            "max_abs_score_diff": float((gv - fv).abs().max()), "ids_equal_fraction": float((gi == fi).float().mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("shape", type=int, nargs="*", help="users items (default: 6040 x 3706 and 4736 x 200000)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--exclude", default="none", choices=["none", "empty", "ml1m", "zipf"])
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--generic", action="store_true")
    args = ap.parse_args()
    shapes = [(6040, 3706), (4736, 200000)] if len(args.shape) < 2 else [(args.shape[0], args.shape[1])]
    dev = torch.device("cuda", 0)
    print(json.dumps({"device": torch.cuda.get_device_name(dev), "power_limit_w": power_limit()}), flush=True)
    g = torch.Generator(dev).manual_seed(0)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    c = 64
    w = [r(c, c) * 0.2, r(c) * 0.1, r(c, c) * 0.2, r(c) * 0.1, r(2 * c, c) * 0.15, r(c) * 0.1, r(c, c) * 0.2, r(c) * 0.1, r(c) * 0.2,
         torch.zeros(1, device=dev)]
    score = ops.score_hybrid_topk_bf16 if args.precision == "bf16" else ops.score_hybrid_topk_tf32x3
    kernel = KERNEL[args.precision]
    for n_users, n_items in shapes:
        t = [r(n_users, c), r(n_items, c), r(n_users, c), r(n_items, c)]
        score(*t, *w, 10)
        torch.cuda.synchronize()
        if args.exclude != "none":
            top, _ = score(*t, *w, 128)
            excl = exclusion_lists(args.exclude, n_users, n_items, top)
            none, lst = alternate(lambda: score(*t, *w, 10), lambda: score(*t, *w, 10, excl), args.reps)
            print(json.dumps({"kernel": kernel, "precision": args.precision, "users": n_users, "items": n_items, "k": 10,
                              "exclude": args.exclude, "list_items": int(excl[1].numel()), "reps": args.reps,
                              **arm_summary(none, lst)}), flush=True)
            continue
        times = []
        for _ in range(args.reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            score(*t, *w, 10)
            e1.record()
            torch.cuda.synchronize()
            times.append(e0.elapsed_time(e1))
        times.sort()
        ms = times[len(times) // 2]
        pairs = n_users * n_items
        print(json.dumps({"kernel": kernel, "precision": args.precision, "users": n_users, "items": n_items, "k": 10,
                          "reps": args.reps, "ms": ms, "ms_min": times[0], "ms_max": times[-1],
                          "pairs_per_s": pairs / ms * 1e3, "tensor_tflops": pairs * FLOP_PER_PAIR[args.precision] / ms / 1e9}),
              flush=True)
    if args.generic and len(args.shape) < 2:
        print(json.dumps(generic_vs_fused(max(1, min(args.reps, 3)))), flush=True)


def power_limit():
    import subprocess
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


main()
