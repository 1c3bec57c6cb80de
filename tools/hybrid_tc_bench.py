#!/usr/bin/env python
"""Micro-benchmark of the chained tensor-core hybrid catalog scorer (cbrs_score_hybrid_topk_bf16) on random hoisted
tables (run under gpurun): users x items, CUDA events, one warm-up.  40,960 tensor FLOP per pair (4 products of 64 x 64
plus the 128 x 64 first classifier layer counted as two).

    python tools/hybrid_tc_bench.py [users items] [--exclude {none,empty,ml1m,zipf}] [--reps R]

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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("shape", type=int, nargs="*", help="users items (default: 6040 x 3706 and 4736 x 200000)")
    ap.add_argument("--exclude", default="none", choices=["none", "empty", "ml1m", "zipf"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    shapes = [(6040, 3706), (4736, 200000)] if len(args.shape) < 2 else [(args.shape[0], args.shape[1])]
    dev = torch.device("cuda", 0)
    g = torch.Generator(dev).manual_seed(0)
    r = lambda *s: torch.randn(*s, device=dev, generator=g)
    c = 64
    w = [r(c, c) * 0.2, r(c) * 0.1, r(c, c) * 0.2, r(c) * 0.1, r(2 * c, c) * 0.15, r(c) * 0.1, r(c, c) * 0.2, r(c) * 0.1, r(c) * 0.2,
         torch.zeros(1, device=dev)]
    for n_users, n_items in shapes:
        t = [r(n_users, c), r(n_items, c), r(n_users, c), r(n_items, c)]
        ops.score_hybrid_topk_bf16(*t, *w, 10)
        torch.cuda.synchronize()
        if args.exclude != "none":
            top, _ = ops.score_hybrid_topk_bf16(*t, *w, 128)
            excl = exclusion_lists(args.exclude, n_users, n_items, top)
            none, lst = alternate(lambda: ops.score_hybrid_topk_bf16(*t, *w, 10),
                                  lambda: ops.score_hybrid_topk_bf16(*t, *w, 10, excl), args.reps)
            print(json.dumps({"kernel": "score_hybrid_tc_kernel", "users": n_users, "items": n_items, "k": 10,
                              "exclude": args.exclude, "list_items": int(excl[1].numel()), "reps": args.reps,
                              **arm_summary(none, lst)}), flush=True)
            continue
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        ops.score_hybrid_topk_bf16(*t, *w, 10)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1)
        pairs = n_users * n_items
        print(json.dumps({"kernel": "score_hybrid_tc_kernel", "users": n_users, "items": n_items, "ms": ms,
                          "pairs_per_s": pairs / ms * 1e3, "tensor_tflops": pairs * 40960 / ms / 1e9}), flush=True)


main()
