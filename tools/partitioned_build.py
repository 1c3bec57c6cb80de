"""Device memory and time of the graph build, whole and partitioned, at config 5 (bench.py's graph).

Arms, each with torch.cuda's peak-allocation counter reset before it:
  * whole: ops.synth_bipartite + DeviceGraph.norm, what every rank of a RowPartition runs today (bench.py);
  * N = 2, 4, 8 ranks, built one after the other in this process: rank r's pass-1 histogram and
    graph.build_row_blocks of its own row blocks (norm view) from a streamed graph.SyntheticSource.  Every rank's
    degrees come from graph.LoopbackDegrees, run before the arm and handed to the rank as a real all-gather would
    (a fresh [N] device vector inside the arm).  The whole build's CSR stays on the device for the check, so a rank's
    peak is reported as the peak above what was allocated when the arm began.
Each rank's slices are compared with the whole build's row_slice, field for field (torch.equal).  Times end in a
device synchronise.  A multi-GPU run is not part of this tool.

    python tools/partitioned_build.py [--scale c5] [--ranks 2 4 8] [--out result.json]
"""
import argparse
import json
import os
import subprocess
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

SCALES = {"c5": (10_000_000, 1_000_000, 1_000_000_000), "c5-tenth": (1_000_000, 100_000, 100_000_000),
          "c5-hundredth": (100_000, 10_000, 10_000_000)}   # bench.py's scales


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = "nvidia-smi unavailable: %s" % e
    return {"device": torch.cuda.get_device_name(0), "nvidia_smi": q}


def same_slice(got, want):
    if (got.row_offset, got.n_rows, got.blocking) != (want.row_offset, want.n_rows, want.blocking):
        return False
    if not (torch.equal(got.rowptr, want.rowptr) and torch.equal(got.colidx, want.colidx)
            and torch.equal(got.vals, want.vals)):
        return False
    for k in ("n_chunks", "n_heavy", "n_slots"):
        if got.chunks[k] != want.chunks[k]:
            return False
    for k in ("chunk_row", "chunk_begin", "chunk_slot", "heavy_row", "heavy_slot_ptr", "chunk_len"):
        g, w = got.chunks[k], want.chunks[k]
        if (g is None) != (w is None) or (g is not None and not torch.equal(g, w)):
            return False
    return True


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scale", default="c5", choices=sorted(SCALES))
    ap.add_argument("--ranks", type=int, nargs="+", default=[2, 4, 8])
    ap.add_argument("--seed", type=int, default=42)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    from deep_cbrs_amar_renaissance_b200 import graph as G
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.distributed import balanced_ranges, edge_cost_prefix
    torch.cuda.set_device(0)
    dev = torch.device("cuda", 0)
    ops.check_device()
    nu, ni, ne = SCALES[args.scale]
    n = nu + ni
    sizes = [nu, ni]
    gib = float(1 << 30)
    res = {"tool": "partitioned_build", "scale": args.scale, "n_users": nu, "n_items": ni, "coo_entries": 2 * ne,
           "card": card(), "piece_edges": G.PIECE_EDGES}

    # ---- whole build (bench.py's path)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    torch.cuda.reset_peak_memory_stats()
    base = torch.cuda.memory_allocated()
    t0 = time.perf_counter()
    row, col = ops.synth_bipartite(nu, ni, ne, args.seed, dev)
    whole = G.DeviceGraph(row, col, None, n)
    del row, col
    norm = whole.norm
    whole.release_coo()
    torch.cuda.synchronize()
    res["whole"] = {"seconds": time.perf_counter() - t0,
                    "peak_gib": (torch.cuda.max_memory_allocated() - base) / gib,
                    "kept_gib": (torch.cuda.memory_allocated() - base) / gib, "nnz": norm.nnz,
                    "blocking": list(norm.blocking)}
    print(json.dumps({"whole": res["whole"]}), flush=True)

    src = G.SyntheticSource(nu, ni, ne, args.seed)
    hist = G.row_histogram(src, dev)
    est = G.estimated_rowptr(hist)
    res["partitioned"] = []
    for world in args.ranks:
        ranges = balanced_ranges(sizes, world, edge_cost_prefix(est, sizes, G.blocking_policy(n)[1]))
        t0 = time.perf_counter()
        d_host = G.LoopbackDegrees(src, ranges, hist, dev).d.cpu()
        loop_s = time.perf_counter() - t0
        ranks = []
        for r in range(world):
            mine = [rg for rg in ranges[r] if rg[1] > rg[0]]
            torch.cuda.synchronize()
            torch.cuda.empty_cache()
            torch.cuda.reset_peak_memory_stats()
            base = torch.cuda.memory_allocated()
            t0 = time.perf_counter()
            h = G.row_histogram(src, dev)
            slices = G.build_row_blocks(src, mine, lambda local: d_host.to(dev), ("norm",), h, device=dev)["norm"]
            del h
            torch.cuda.synchronize()
            secs = time.perf_counter() - t0
            peak = (torch.cuda.max_memory_allocated() - base) / gib
            kept = (torch.cuda.memory_allocated() - base) / gib
            ok = all(same_slice(sl, norm.row_slice(a, b)) for (a, b), sl in zip(mine, slices))
            ranks.append({"rank": r, "blocks": mine, "entries": sum(s.nnz for s in slices), "seconds": secs,
                          "peak_gib": peak, "kept_gib": kept, "bit_identical": ok})
            del slices
        line = {"ranks": world, "loopback_degrees_seconds": loop_s, "per_rank": ranks,
                "max_peak_gib": max(x["peak_gib"] for x in ranks), "max_seconds": max(x["seconds"] for x in ranks),
                "bit_identical": all(x["bit_identical"] for x in ranks)}
        res["partitioned"].append(line)
        print(json.dumps(line), flush=True)
    res["bit_identical"] = all(x["bit_identical"] for x in res["partitioned"])
    res["multi_gpu"] = "not run by this tool (one process, one GPU)"
    text = json.dumps(res, indent=1)
    print(text)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    return 0 if res["bit_identical"] else 1


if __name__ == "__main__":
    sys.exit(main())
