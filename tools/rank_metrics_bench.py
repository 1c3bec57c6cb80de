#!/usr/bin/env python
"""Full-catalog ranking metrics: the device kernel (cbrs_rank_metrics) against the host stage it replaces in the
experiment driver (metrics.catalog_predictions + precision_recall_f1_at_k at both cutoffs).  Run on a B200.

For each user count: relevance lists of 10..30 distinct items per user (about 20) drawn from the catalog, and top-k lists
(k = 10) whose slots are one of the user's relevant items with probability 0.2, a random catalog item otherwise, all
generated on the device from a seed.  Prints one JSON line per user count:
  kernel_ms_*   the C call (main kernel + fixed-order reduction), CUDA events around each call, after --warmup calls;
                median / min / max of --reps;
  api_ms        utilities.metrics.catalog_ranking_metrics end to end (host clock, ends with the copy of the sums);
  host_ms       catalog_predictions + precision_recall_f1_at_k at cutoffs 5 and 10 (host clock, one run), or null when
                the user count exceeds --host-max (the host arm is a Python loop over every test and prediction row);
  max_abs_diff  the largest difference of P / R / F1 between the two arms, when both ran.
The card's name and power limit are read at start, in the same process.

    python tools/rank_metrics_bench.py [--users 6040 1000000 10000000] [--reps 20] [--host-max 1000000]"""
import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from deep_cbrs_amar_renaissance_b200 import _lib as L, ops  # noqa: E402
from deep_cbrs_amar_renaissance_b200.scoring import ItemLists  # noqa: E402
from deep_cbrs_amar_renaissance_b200.utilities import metrics as M  # noqa: E402

CUTOFFS = (5, 10)


def power_limit():
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                              capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def make_inputs(n_users, n_items, k, seed, dev):
    g = torch.Generator(device=dev).manual_seed(seed)
    lens = torch.randint(10, 31, (n_users,), generator=g, device=dev)
    user = torch.repeat_interleave(torch.arange(n_users, device=dev), lens)
    item = torch.randint(0, n_items, (user.numel(),), generator=g, device=dev)
    rel = ItemLists.from_ratings(torch.stack([user, item + n_users], 1), n_users, n_items, distinct=True)
    del user, item
    counts = rel.rowptr[1:] - rel.rowptr[:-1]
    pick = (torch.rand(n_users, k, generator=g, device=dev) * counts[:, None]).long()
    own = rel.items[(rel.rowptr[:-1, None] + pick).clamp(max=max(rel.items.numel() - 1, 0))]
    rand = torch.randint(0, n_items, (n_users, k), generator=g, device=dev, dtype=torch.int32)
    ids = torch.where(torch.rand(n_users, k, generator=g, device=dev) < 0.2, own, rand).contiguous()
    return ids, rel


def kernel_times(ids, rel, reps, warmup):
    lib = L.load()
    n, k = ids.shape
    nc = len(CUTOFFS)
    sums = torch.empty(nc, 7, dtype=torch.float64, device=ids.device)
    ws = torch.empty(max(16, lib.cbrs_rank_metrics_workspace_bytes(n, nc)), dtype=torch.uint8, device=ids.device)
    cut = (ctypes.c_int32 * nc)(*CUTOFFS)
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    args = (vp(ids), k, n, k, rel.n_items, None, rel.n_users, vp(rel.rowptr), vp(rel.items), cut, nc, vp(sums), None,
            vp(ws), ws.numel())
    times = []
    for r in range(warmup + reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        L.check(lib.cbrs_rank_metrics(*args, ops._stream()), "cbrs_rank_metrics")
        e1.record()
        e1.synchronize()
        if r >= warmup:
            times.append(e0.elapsed_time(e1))
    return times


def host_arm(ids, rel):
    """the driver's stage before the device path: lists to the host, a frame, then the RiVal restatement per cutoff"""
    n_users, n_items = rel.n_users, rel.n_items
    rowptr, items = rel.rowptr.cpu().numpy(), rel.items.cpu().numpy()
    test = np.stack([np.repeat(np.arange(n_users), np.diff(rowptr)), items, np.ones(len(items), np.int64)], 1)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    vals = torch.arange(ids.shape[1], 0, -1, dtype=torch.float32, device=ids.device).expand(ids.shape)
    frame = M.catalog_predictions(ids, vals, np.arange(n_users), np.arange(n_items)).to_numpy()
    res = {c: M.precision_recall_f1_at_k(test, frame, c) for c in CUTOFFS}
    return (time.perf_counter() - t0) * 1e3, res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--users", type=int, nargs="+", default=[6040, 1_000_000, 10_000_000])
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--host-max", type=int, default=1_000_000)
    ap.add_argument("--seed", type=int, default=0)
    args = ap.parse_args()
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    ops.check_device()
    card = {"device": torch.cuda.get_device_name(dev), "power_limit_w,max_sm_clock": power_limit()}
    for n_users in args.users:
        n_items = 3706 if n_users <= 6040 else 200_000      # MovieLens-1M's catalog at its user count
        ids, rel = make_inputs(n_users, n_items, args.k, args.seed, dev)
        times = kernel_times(ids, rel, args.reps, args.warmup)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        dev_res = M.catalog_ranking_metrics(ids, rel, cutoffs=CUTOFFS)
        api_ms = (time.perf_counter() - t0) * 1e3
        line = dict(card, users=n_users, items=n_items, k=args.k, relevant=int(rel.items.numel()), cutoffs=list(CUTOFFS),
                    kernel_ms_median=statistics.median(times), kernel_ms_min=min(times), kernel_ms_max=max(times),
                    reps=args.reps, api_ms=api_ms, host_ms=None, host_capped_at=args.host_max,
                    ndcg_at_10=dev_res["ndcg_at_10"], recall_at_10=dev_res["recall_at_10"])
        if n_users <= args.host_max:
            host_ms, host = host_arm(ids, rel)
            line["host_ms"] = host_ms
            line["host_over_kernel"] = host_ms / line["kernel_ms_median"]
            line["max_abs_diff"] = max(abs(dev_res["%s_at_%d" % (m, c)] - host[c][m])
                                       for c in CUTOFFS for m in ("precision", "recall", "f1"))
        print(json.dumps(line), flush=True)
        del ids, rel
        torch.cuda.empty_cache()


if __name__ == "__main__":
    main()
