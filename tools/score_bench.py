"""Full-catalog BasicRS scoring + top-10 (cbrs_score_catalog_topk*) at the reference's classifier shape (64 -> 64 -> 1):
FFMA kernel, fp32-accurate 3xTF32 tensor-core kernel, bf16 tensor-core kernel.  CUDA-event timing on the launching stream.

    python tools/score_bench.py [users] [items] [--exclude {none,empty,ml1m,zipf}] [--reps R]   # one JSON line per kernel

--exclude other than none times each kernel without lists and with the chosen per-user exclusion lists, alternating
the two arms R times, and reports both arms' times (median and spread) and the overhead of the lists:
  empty  every list empty (non-null pointers: the search is reached but finds nothing)
  ml1m   20 to 240 seen items per user (mean 130, MovieLens-1M's density over 3,706 items)
  zipf   100 to 5,000 seen items per user, Pareto-distributed lengths (a few heavy users), Zipf item popularity
A user's seen items are the ones its model scores highest (that is what training does to them), so each ml1m / zipf
list starts with the user's own top-128 items of the run without lists - the case where every listed item keeps
beating the threshold and is searched - and is filled up with random items."""
import argparse
import json
import os
import sys

import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, REPO)


def time_ms(fn, iters=3, warmup=1):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def exclusion_lists(kind, n_users, n_items, top_ids, seed=7):
    """(rowptr int64 [n_users + 1], items int32) device CSR of the `kind` arm (module docstring); top_ids [U, >= 128]:
    each user's items by descending score without lists.  Lists are sorted, duplicates kept; lengths are capped at
    half the catalog."""
    dev = top_ids.device
    g = torch.Generator(device=dev).manual_seed(seed)
    if kind == "empty":
        return torch.zeros(n_users + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev)
    u = torch.rand(n_users, device=dev, generator=g)
    if kind == "ml1m":
        lengths = (20 + u * 220).long()
        fill = lambda n: torch.randint(0, n_items, (n,), device=dev, generator=g)
    elif kind == "zipf":
        lengths = (100 * (1 - u * 0.999) ** -1.2).long().clamp(100, 5000)
        # Zipf(1)-like popularity: log-uniform ranks
        fill = lambda n: (torch.exp(torch.rand(n, device=dev, generator=g) * torch.log(torch.tensor(float(n_items)))) - 1
                          ).long().clamp(0, n_items - 1)
    else:
        raise ValueError(kind)
    lengths = lengths.clamp(max=max(1, n_items // 2))
    n_top = min(128, top_ids.shape[1])
    head = lengths.clamp(max=n_top)
    total = int(lengths.sum())
    rowptr = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
    torch.cumsum(lengths, 0, out=rowptr[1:])
    row = torch.repeat_interleave(torch.arange(n_users, device=dev), lengths)
    pos = torch.arange(total, device=dev) - rowptr[:-1][row]
    items = fill(total)
    is_head = pos < head[row]
    items[is_head] = top_ids[row[is_head], pos[is_head]].long()
    items = torch.sort(row * n_items + items).values % n_items   # sorted within each row
    return rowptr, items.to(torch.int32)


def alternate(fn_none, fn_list, reps):
    """reps x (no lists, lists), alternating; times in ms."""
    none, lst = [], []
    for _ in range(reps):
        none.append(time_ms(fn_none))
        lst.append(time_ms(fn_list))
    return none, lst


def arm_summary(none, lst):
    med = lambda x: sorted(x)[len(x) // 2]
    return {"ms_none": med(none), "ms_none_min": min(none), "ms_none_max": max(none), "ms_lists": med(lst),
            "ms_lists_min": min(lst), "ms_lists_max": max(lst), "overhead": med(lst) / med(none) - 1.0,
            "none_spread": (max(none) - min(none)) / med(none)}


def run(n_users=4736, n_items=200000, c1=64, c2=64, k=10, exclude="none", reps=5):
    from deep_cbrs_amar_renaissance_b200 import ops
    dev = torch.device("cuda", torch.cuda.current_device())
    g = torch.Generator(device=dev).manual_seed(1)
    P = torch.randn(n_users, c1, device=dev, generator=g)
    Q = torch.randn(n_items, c1, device=dev, generator=g)
    w2 = torch.randn(c1, c2, device=dev, generator=g) / c1 ** 0.5
    b2 = torch.randn(c2, device=dev, generator=g) * 0.1
    w3 = torch.randn(c2, device=dev, generator=g) / c2 ** 0.5
    b3 = torch.full((1,), 0.05, device=dev)
    out = []
    ref = None
    for precision in ("fp32-ffma", "fp32", "bf16"):
        ids, vals = ops.score_catalog_topk(P, Q, w2, b2, w3, b3, k, precision)
        name = {"fp32-ffma": "cbrs_score_catalog_topk (FFMA)", "fp32": "cbrs_score_catalog_topk_tf32x3 (3xTF32 tcgen05)",
                "bf16": "cbrs_score_catalog_topk_bf16 (bf16 tcgen05)"}[precision]
        if exclude != "none":
            top, _ = ops.score_catalog_topk(P, Q, w2, b2, w3, b3, 128, precision)
            excl = exclusion_lists(exclude, n_users, n_items, top)
            none, lst = alternate(lambda: ops.score_catalog_topk(P, Q, w2, b2, w3, b3, k, precision),
                                  lambda: ops.score_catalog_topk(P, Q, w2, b2, w3, b3, k, precision, excl), reps)
            line = {"kernel": name, "users": n_users, "items": n_items, "c1": c1, "c2": c2, "k": k, "exclude": exclude,
                    "list_items": int(excl[1].numel()), "reps": reps, **arm_summary(none, lst)}
            out.append(line)
            continue
        ms = time_ms(lambda: ops.score_catalog_topk(P, Q, w2, b2, w3, b3, k, precision))
        line = {"kernel": name, "users": n_users, "items": n_items, "c1": c1, "c2": c2, "k": k, "ms": ms,
                "pairs_per_s": n_users * n_items / (ms * 1e-3)}
        if ref is None:
            ref = (ids, vals)
        else:
            line["ids_equal_to_ffma"] = float((ids == ref[0]).float().mean().item())
            line["max_score_diff_vs_ffma"] = float((vals - ref[1]).abs().max().item())
        out.append(line)
    return out


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("users", type=int, nargs="?", default=4736)
    ap.add_argument("items", type=int, nargs="?", default=200000)
    ap.add_argument("--exclude", default="none", choices=["none", "empty", "ml1m", "zipf"])
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    for line in run(args.users, args.items, exclude=args.exclude, reps=args.reps):
        print(json.dumps(line), flush=True)
