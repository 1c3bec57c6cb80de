#!/usr/bin/env python
"""Benchmark of the hot path: GNN propagation -> gather -> MLP -> sigmoid (-> catalog top-k).

    python bench.py --gpus N --steps K --warmup W            # this implementation (B200)
    python bench.py --impl reference --gpus N --steps K ...  # CPU restatement of the reference path
    python bench.py --gpus 1 --steps K --warmup W --dump-outputs DIR   # + DIR/scores.npy of the last timed step

A step = one pass of the hot path over one batch: the model call the reference makes per
batch (/root/reference/src/models/basic.py:61-63: full-graph propagation, embedding lookup,
BasicRS MLP, sigmoid).  Headline metric (BASELINE.json): propagation edges/s, i.e.
K_layers * nnz(A_hat) / step time, whole job; scored pairs/s for full-catalog top-k is
measured in the same run and reported under "pairs".

Workload at every N: config 5 of BASELINE.json, the scaled synthetic bipartite graph
(10M users x 1M items x 1e9 edges, dim 128, 3 GCN layers, fp32) - it fits one B200 - so the
graph is fixed and N GPUs split its rows ("scaling": "strong").  Inputs are larger than L2
(5.6 GB of features per layer), so no L2 flush is needed between iterations.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

SCALES = {  # name: users, items, undirected edges
    "c5": (10_000_000, 1_000_000, 1_000_000_000),
    "c5-tenth": (1_000_000, 100_000, 100_000_000),
    "c5-hundredth": (100_000, 10_000, 10_000_000),
}
DIM, LAYERS = 128, 3
DENSE_UNITS, CLF_UNITS = [48, 48], [64, 64]  # econfigs/basic-gnn.yaml grid2 scorer
PAIR_BATCH = 65536


BF16_SCORER_FLOPS = 2 * (64 + 16) * 64 + 2 * 64 * 16   # per pair, cbrs_score_catalog_topk_bf16 at the reference's 64 -> 64 -> 1 classifier


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scale", default=os.environ.get("CBRS_BENCH_SCALE", "c5"), choices=sorted(SCALES))
    ap.add_argument("--cpu-scale", default="c5-hundredth", choices=sorted(SCALES))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-bf16", action="store_true", help="skip the bf16-operand variant of the step")
    ap.add_argument("--no-small-configs", action="store_true", help="skip the MovieLens-1M-shaped configs 1-4 block")
    ap.add_argument("--unscattered", action="store_true",
                    help="item id = popularity rank (no scattering of hot items over the id space): the adversarial case for "
                         "the row partition; cuts are balanced by edge count either way")
    ap.add_argument("--row-count-cuts", action="store_true", help="N > 1: cut node types at equal ROW counts (round-1 behaviour)")
    ap.add_argument("--edge-count-cuts", action="store_true", help="N > 1: cut at equal EDGE counts (default: equal edge COST, "
                                                                   "edges of rows that stream from HBM weigh 2.4)")
    ap.add_argument("--no-parity-check", action="store_true", help="N > 1: skip the bit-identity self-check that precedes timing")
    ap.add_argument("--catalog-users", type=int, default=4736,
                    help="users per rank scored against the whole catalog (4736 = 148 SMs x 2 CTAs x 16 users: one full wave of "
                         "the fp32 kernel; the bf16 kernel gets 4x as many)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the scores the model call returned in the last one as "
                         "DIR/scores.npy (float32, one per pair of the seeded batch; DIR/scores_rank<r>.npy per rank when N > 1)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


# ----------------------------------------------------------------------------- CPU arm
def cpu_reference_run(scale, steps, warmup, threads):
    """K-layer GCN forward + BasicRS scoring of one batch on the host cores with the oracle
    (torch-CPU twin, all threads): the CPU restatement of the reference path."""
    import torch
    from oracle import synth as osynth
    from oracle import torch_cpu as oc
    torch.set_num_threads(threads)
    n_users, n_items, n_edges = SCALES[scale]
    row, col = osynth.synth_bipartite(n_users, n_items, n_edges, 42)
    a_hat, nnz = oc.gcn_filter_torch(row, col, n_users + n_items)
    rng = np.random.RandomState(0)
    n = n_users + n_items
    emb = torch.from_numpy((rng.standard_normal((n, DIM)) * 0.02).astype(np.float32))
    layers = [(torch.from_numpy(oc.glorot(rng, (DIM, DIM))), torch.zeros(DIM)) for _ in range(LAYERS)]
    mlp = oc.random_basic_rs(rng, DIM * (LAYERS + 1), DENSE_UNITS, CLF_UNITS)
    u = torch.from_numpy(rng.randint(0, n_users, size=PAIR_BATCH))
    i = torch.from_numpy(rng.randint(0, n_items, size=PAIR_BATCH) + n_users)

    def step():
        x = oc.gcn_forward(emb, a_hat, layers)
        return oc.basic_rs(x, u, i, mlp)

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return dict(edges_per_s=LAYERS * nnz / dt, ms_per_step=dt * 1e3, nnz=nnz,
                sample="GCN %d layers dim %d on the %s graph (%d users x %d items, nnz(A_hat)=%d) + %d scored pairs per step"
                       % (LAYERS, DIM, scale, n_users, n_items, nnz, PAIR_BATCH))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    r = cpu_reference_run(args.cpu_scale, args.steps, args.warmup, threads)
    n_users, n_items, n_edges = SCALES[args.scale]
    line = {
        "impl": "reference", "metric": "propagation_edges_per_s", "value": r["edges_per_s"], "unit": "edges/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": r["ms_per_step"],
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args.scale, args.gpus),
        "cpu_baseline": {"value": r["edges_per_s"], "unit": "edges/s", "cores": threads, "kind": "port",
                         "sample": r["sample"]},
        "e2e": {"value": r["edges_per_s"], "unit": "edges/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "TensorFlow/Spektral cannot be installed here; this is the CPU restatement (oracle, torch-CPU, "
                "all host threads) on a bounded sample of the workload; the rate is per edge.",
    }
    print(json.dumps(line), flush=True)


NCU_SPMM = os.path.join("profiles", "r02_ncu_spmm_blocked_tf32x3_c5.json")


def ncu_traffic(scale, world):
    """dram bytes per sparse-kernel launch from the committed `ncu --set full` capture of this same workload (one GPU,
    config 5): a CITATION of profiles/r02_ncu_spmm_blocked_tf32x3_c5.json, not something measured in this run (ncu
    cannot run inside a timed bench); the line says so in roofline.traffic_source."""
    if scale != "c5" or world != 1:
        return None
    try:
        for k in json.load(open(os.path.join(REPO, NCU_SPMM))):
            if "spmm_chunk_kernel" in k["kernel"]:
                return (float(k["dram__bytes_read.sum [Gbyte]"]) + float(k["dram__bytes_write.sum [Gbyte]"])) * 1e9
    except Exception:
        pass
    return None


def workload_config(scale, gpus):
    n_users, n_items, n_edges = SCALES[scale]
    return {"workload": "%s scaled synthetic bipartite graph, BasicGCN %d layers dim %d fp32, concatenation, "
                        "BasicRS %s/%s, %d scored pairs per step" % (scale, LAYERS, DIM, DENSE_UNITS, CLF_UNITS, PAIR_BATCH),
            "users": n_users, "items": n_items, "undirected_edges": n_edges, "dim": DIM, "layers": LAYERS,
            "parallelism": ("rows x%d" % gpus) if gpus > 1 else "single",
            "l2": "inputs larger than L2 (no flush needed)"}


def mark_variant(cfg, args):
    if args.unscattered:
        cfg["item_ids"] = "unscattered (id = popularity rank)"
    return cfg


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc = [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def stop(self, t0, t1):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        rows = [r for t, r in self.rows if t0 <= t <= t1] or [r for _, r in self.rows]
        try:
            sm = sorted(float(r[0]) for r in rows)
            names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
            reasons = [n for k, n in enumerate(names) if any(r[3 + k].lower().startswith("active") for r in rows)]
            return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(rows[0][1]), "reasons": reasons,
                    "power_w_max": max(float(r[2]) for r in rows), "samples": len(rows)}
        except Exception as e:  # pragma: no cover
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["parse error: %s" % e]}


# ----------------------------------------------------------------------------- configs 1-4 (MovieLens-1M shape)
def nvlink_counters(local):
    """Cumulative NVLink payload bytes (tx, rx) of this rank's GPU summed over its links, read from NVML field values
    (NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX / RX, KiB, scope = all links); None when NVML does not expose them."""
    try:
        import pynvml
        import torch
        pynvml.nvmlInit()
        try:
            handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + str(torch.cuda.get_device_properties(local).uuid)).encode())
        except Exception:
            handle = pynvml.nvmlDeviceGetHandleByIndex(local)
        vals = pynvml.nvmlDeviceGetFieldValues(handle, [(pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_TX, 0xFFFFFFFF),
                                                        (pynvml.NVML_FI_DEV_NVLINK_THROUGHPUT_DATA_RX, 0xFFFFFFFF)])
        out = []
        for v in vals:
            if v.nvmlReturn != 0:
                return None
            kib = {pynvml.NVML_VALUE_TYPE_UNSIGNED_LONG_LONG: v.value.ullVal, pynvml.NVML_VALUE_TYPE_UNSIGNED_LONG: v.value.ulVal,
                   pynvml.NVML_VALUE_TYPE_UNSIGNED_INT: v.value.uiVal}.get(v.valueType)
            if kib is None:
                return None
            out.append(int(kib) * 1024)
        return tuple(out)
    except Exception:
        return None


def small_configs(dev):
    """BASELINE configs 1-4 on one GPU: the per-batch model call (batch 2048, econfigs grid2 shapes) eager and as a
    CUDA-graph replay, and full-catalog top-10 for every user with HOST ids in and HOST (ids, scores) out.  These
    graphs are L2-resident (~67 MB of algorithmic traffic per layer) and launch-latency-bound: the numbers are times
    against the launch count, never an HBM fraction (SURVEY section 0).  Published context (BASELINE.md, other
    hardware, whole training loop): BasicRS-GCN 16/2 trains in 211 s / 25 epochs on an RTX 3060 = ~11.4 ms per step."""
    import torch
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.data.preprocess import RelationalAdjacency
    from deep_cbrs_amar_renaissance_b200.graphed import GraphedForward
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic, hybrid
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph

    def timeit(fn, n=30, warm=3):
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

    n_users, n_items, batch, k = 6040, 3706, 2048, 10
    n_props, n_links = 17554, 70341                      # doc.pdf Table 3
    adj = small_graph(n_users, n_items, 572000, seed=42)
    uip = small_graph(n_users, n_items, 572000, seed=42, n_props=n_props, n_links=n_links, dup_links=400)
    is_prop = (uip.row >= n_users + n_items) | (uip.col >= n_users + n_items)
    uip_rel = RelationalAdjacency(uip, is_prop.astype(np.int32), 2)
    rng = np.random.RandomState(0)
    u = rng.randint(0, n_users, size=batch)
    i = rng.randint(0, n_items, size=batch) + n_users
    bert = (rng.standard_normal((n_users + n_items, 768)) * 0.5).astype(np.float32)
    all_users = torch.arange(n_users, dtype=torch.int64).pin_memory()
    hyb = dict(dense_units=[[48, 48], [256, 64], [64, 64]], feature_based=True)
    cases = [("config 1: BasicGCN", basic.BasicGCN, adj, {}, "fp32"),
             ("config 2: BasicGraphSage", basic.BasicGraphSage, adj, {}, "fp32"),
             ("config 2: BasicGAT", basic.BasicGAT, adj, {}, "fp32"),
             ("config 3: BasicGCN on the user-item-properties graph (untyped, as the reference)", basic.BasicGCN, uip, {}, "fp32"),
             ("config 3: BasicRGCN, 2 relation types (node-range)", basic.BasicRGCN, uip_rel, {}, "fp32"),
             ("config 4: HybridBertGCN feature-based, fp32 scorer", hybrid.HybridBertGCN, adj, hyb, "fp32"),
             ("config 4: HybridBertGCN feature-based, bf16 tensor-core scorer", hybrid.HybridBertGCN, adj, hyb, "bf16")]
    out = []
    for name, cls, a, extra, precision in cases:
        set_seed(42)
        kw = dict(n_hiddens=[16, 16], n_layers=2, embedding_dim=16, dense_units=[48, 48], clf_units=[64, 64])
        kw.update(extra)
        model = cls(a, **kw)
        if cls is hybrid.HybridBertGCN:
            # the bf16 case keeps the static content table as bf16: its towers are fed by TMA (cbrs_dense_tc_bf16)
            model.set_content_table(bert, dtype="bf16" if precision == "bf16" else "fp32")
            model.set_scorer_precision(precision)
        model((u, i))
        before = ops.LAUNCHES
        model((u, i))
        kernels = ops.LAUNCHES - before
        eager = timeit(lambda: model((u, i)))
        g = GraphedForward(model, batch)
        graphed = timeit(lambda: g((u, i)))
        gph = model.gnn.gnn_layers.adj_matrix
        nnz = (gph.raw if ("Sage" in name or "GAT" in name) else gph.norm).nnz

        def catalog():
            users = all_users.to(dev, non_blocking=True)              # H2D: the ids to rank for
            ids, vals = model.recommend_top_k(n_users, n_items, k, users=users, precision=precision)
            return ids.cpu(), vals.cpu()                              # D2H: the lists
        cat = timeit(catalog, n=3, warm=1)                            # propagation recomputed inside: end to end
        out.append({"case": name, "nnz": nnz, "layers": 2, "batch": batch, "kernels_per_call": kernels,
                    "eager_ms": eager, "graph_replay_ms": graphed, "us_per_kernel_in_graph": graphed * 1e3 / max(kernels, 1),
                    "edges_per_s_graph_replay": 2 * nnz / (graphed * 1e-3),
                    "catalog_top10_e2e_ms": cat, "catalog_pairs_per_s_e2e": n_users * n_items / (cat * 1e-3),
                    "catalog_h2d_bytes": n_users * 8, "catalog_d2h_bytes": n_users * k * 8, "scorer_precision": precision})
        del model, g
    return out


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args):
    import torch
    import torch.distributed as dist
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.distributed import RowPartition
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    L.load()
    ops.check_device()
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(REPO, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, peak_src = (peaks.get("hbm_gbs"), "measured") if peaks.get("hbm_gbs") else (6650.0, "fallback")

    # ---- multi-GPU self-check BEFORE anything is timed: the row-partitioned propagation must equal the single-GPU
    # one bit for bit (all layer families, both exchanges, pipelines, fused kernel, blocked schedule; small graphs)
    parity = None
    if world > 1 and not args.no_parity_check:
        from deep_cbrs_amar_renaissance_b200.selfcheck import partition_parity
        t_par0 = time.perf_counter()
        parity = partition_parity()
        parity["seconds"] = time.perf_counter() - t_par0
        if not parity["bit_identical"]:
            if rank == 0:
                print(json.dumps({"metric": "propagation_edges_per_s", "value": None, "n_gpus": world,
                                  "partition_parity": parity, "error": "partitioned result differs from the single-GPU result"}),
                      flush=True)
            dist.destroy_process_group()
            raise SystemExit(3)
        torch.cuda.empty_cache()

    n_users, n_items, n_edges = SCALES[args.scale]
    n = n_users + n_items
    t_build0 = time.perf_counter()
    row, col = ops.synth_bipartite(n_users, n_items, n_edges, 42, dev, scatter_items=not args.unscattered)
    graph = DeviceGraph(row, col, None, n)
    del row, col
    set_seed(42)
    model = basic.BasicGCN(graph, n_hiddens=[DIM] * LAYERS, embedding_dim=DIM, dense_units=DENSE_UNITS,
                           clf_units=CLF_UNITS, final_node="concatenation")
    seq = model.gnn.gnn_layers
    nnz_total = graph.norm.nnz  # builds the normalised CSR on device
    heavy = graph.norm.chunks["n_heavy"]
    part = None
    if world > 1:
        # CBRS_EXCHANGE=nccl|peer; each node type is cut into N blocks of equal EDGE count (SURVEY 8e)
        part = RowPartition([n_users, n_items], final_types=[1],
                            balance_rowptr=None if args.row_count_cuts else graph.norm.rowptr,
                            balance_min_len=0 if args.edge_count_cuts else graph.norm.blocking[1]).attach(seq)
        exchange_label = part.exchange + ("+" + part.pipeline if part.exchange == "peer" else "")
        if part.heap is not None:
            exchange_label += ", %s buffers" % part.heap.backend + (", NVSwitch multicast stores" if part.heap.flags.mc_ptr else "")
        part.csr_slices("norm", graph)
        part.release_full_views(graph)
    else:
        graph.release_coo()
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    build_s = time.perf_counter() - t_build0

    # the batch: pairs whose users this rank owns (scoring is sharded by user)
    rng = np.random.RandomState(1234 + rank)
    if part is not None:
        u_lo, u_hi = part.ranges[rank][0]
    else:
        u_lo, u_hi = 0, n_users
    u_host = torch.from_numpy(rng.randint(u_lo, max(u_hi, u_lo + 1), size=PAIR_BATCH)).pin_memory()
    i_host = torch.from_numpy(rng.randint(0, n_items, size=PAIR_BATCH) + n_users).pin_memory()
    u_dev, i_dev = u_host.to(dev), i_host.to(dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        t1 = time.perf_counter()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return ms.item(), t0, t1

    # ---- device-resident timing (value) -------------------------------------------------
    sampler = ClockSampler(local) if rank == 0 else None
    ops.PROFILE.clear()
    ops.PROFILE_ON = False
    ops.LAUNCHES = 0
    for _ in range(args.warmup):
        model((u_dev, i_dev))
    barrier()
    ops.PROFILE_ON = True
    ops.LAUNCHES = 0
    nvl0 = nvlink_counters(local) if world > 1 else None
    last = {}

    def step():
        last["scores"] = model((u_dev, i_dev))
    ms, t0, t1 = timed(step, args.steps, 0)
    nvl1 = nvlink_counters(local) if world > 1 else None
    launches = ops.LAUNCHES
    ops.PROFILE_ON = False
    clocks = sampler.stop(t0, t1) if sampler else None
    if args.dump_outputs:
        # copied out before anything else runs the model: two builds compare their scores for the same seeded inputs
        os.makedirs(args.dump_outputs, exist_ok=True)
        fname = "scores.npy" if world == 1 else "scores_rank%d.npy" % rank
        np.save(os.path.join(args.dump_outputs, fname), last["scores"].float().cpu().numpy())
    spmm_ms = [a.elapsed_time(b) for (name, a, b, _) in ops.PROFILE if name == "spmm"]
    spmm_meta = [meta for (name, _, _, meta) in ops.PROFILE if name == "spmm"]
    breakdown = {}
    for (name, a, b, _) in ops.PROFILE:
        breakdown[name] = breakdown.get(name, 0.0) + a.elapsed_time(b) / args.steps
    ms_per_step = ms / args.steps
    value = LAYERS * nnz_total / (ms_per_step * 1e-3)

    # per-rank time in the sparse kernels (balance of the row partition)
    rank_sparse = None
    if world > 1:
        mine = torch.tensor([sum(spmm_ms) / max(args.steps, 1)], device=dev, dtype=torch.float64)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        per = [float(t.item()) for t in every]
        rank_sparse = {"ms_per_step": per, "min": min(per), "max": max(per), "max_over_min": max(per) / max(min(per), 1e-9),
                       "local_edges": part.local_edges("norm"),
                       "cuts": "equal row counts" if args.row_count_cuts else ("equal edge counts per node type" if args.edge_count_cuts else "equal edge cost per node type (edges of rows that stream from HBM weigh 2.4)")}

    # NVLink payload bytes this rank's GPU sent / received during the timed steps (NVML counters), next to what the
    # exchange must move: every layer's output rows reach the other G-1 ranks ((G-1)/G * N * H * 4 bytes received per
    # layer and rank); sent = own rows once when the stores go through the NVSwitch multicast mapping, G-1 times otherwise
    nvlink = None
    if world > 1:
        mine = torch.tensor([(nvl1[0] - nvl0[0]) / args.steps, (nvl1[1] - nvl0[1]) / args.steps] if nvl0 and nvl1 else [-1.0, -1.0],
                            device=dev, dtype=torch.float64)
        every = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(every, mine)
        if not all(float(t[0]) >= 0 for t in every):
            nvlink = {"unavailable": "NVML reports NVLINK_THROUGHPUT_DATA_TX/RX as NOT_SUPPORTED on this (virtualised) pool and "
                                     "`nvidia-smi nvlink -gt d` prints N/A (profiles/r02_nvlink_counters_unavailable.txt)",
                      "expected_rx_bytes_per_step_per_rank":
                          sum((n if l < LAYERS - 1 else n_items) * (world - 1) / world for l in range(LAYERS)) * DIM * 4}
        else:
            own_rows = sum(hi - lo for lo, hi in part.ranges[rank])
            rows_out = [(n if l < LAYERS - 1 else n_items) for l in range(LAYERS)]   # last layer: items only (scoring is user-sharded)
            nvlink = {"tx_bytes_per_step": [float(t[0]) for t in every], "rx_bytes_per_step": [float(t[1]) for t in every],
                      "expected_rx_bytes_per_step_per_rank": sum(r * (world - 1) / world for r in rows_out) * DIM * 4,
                      "expected_tx_multicast": sum(r / world for r in rows_out) * DIM * 4,
                      "expected_tx_unicast": sum(r * (world - 1) / world for r in rows_out) * DIM * 4,
                      "rank0_own_rows": own_rows, "source": "NVML NVLINK_THROUGHPUT_DATA_TX/RX, all links, around the timed steps"}

    # ---- end to end through the public model call with HOST buffers (e2e) --------------------
    def e2e_step():
        out = model((u_host, i_host))       # H2D of the id vectors inside
        return out.cpu()                    # D2H of the scores
    ms_e2e, _, _ = timed(e2e_step, args.steps, 1)
    e2e_value = LAYERS * nnz_total / (ms_e2e / args.steps * 1e-3)

    # ---- roofline of the dominant kernel (SpMM) -------------------------------------------
    # algorithmic bytes of one SpMM launch (SURVEY 8d): nnz*(4 col + 4 val + D*4 row) + rows*(D*4 out + 8 rowptr),
    # summed over exactly the launches that were timed (a rank's user slice and item slice are separate launches)
    avg_ms = float(np.mean(spmm_ms)) if spmm_ms else float("nan")
    alg_bytes = float(np.mean([m["bytes"] for m in spmm_meta])) if spmm_meta else float("nan")
    achieved = (sum(m["bytes"] for m in spmm_meta) / (sum(spmm_ms) * 1e-3) / 1e9) if spmm_ms else float("nan")
    traffic = ncu_traffic(args.scale, world)
    roofline = {"bound": "hbm", "kernel": "spmm_chunk_kernel<32,4,4,4> on the column-blocked schedule (+heavy-row merge)",
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic,
                "traffic_source": (NCU_SPMM + " (ncu --set full of this workload, committed; not measured in this run)") if traffic else None,
                "peak_source": peak_src, "launch_ms": avg_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "bytes_per_edge": 8 + DIM * 4, "launches_timed": len(spmm_ms),
                "share_of_step": (sum(spmm_ms) / args.steps) / ms_per_step if spmm_ms else None,
                "note": "achieved = algorithmic bytes (no-reuse gather model, SURVEY 8d) / measured launch time; it exceeds the "
                        "DRAM peak because the blocked schedule serves heavy rows from an L2-resident window and hot item "
                        "rows hit in L2 - `traffic` is what ncu saw cross the HBM pins (the kernel is bound by the L2 -> SM "
                        "path, DESIGN.md section 4)"}

    # ---- the same step with bf16 STORAGE of the gathered operand (config 5's "bf16 feature variant") -------
    # Z = X W is written as bf16 by the dense kernel (and travels as bf16 between GPUs); products and sums stay
    # fp32.  Not the headline: the reference computes in fp32.  Tolerance vs the fp32 result: tests/test_gpu_bf16.py.
    bf16_block = None
    if not args.no_bf16:
        seq.set_feature_dtype("bf16")
        ops.PROFILE.clear()
        for _ in range(2):
            model((u_dev, i_dev))
        barrier()
        ops.PROFILE_ON = True
        ms16, _, _ = timed(lambda: model((u_dev, i_dev)), args.steps, 0)
        ops.PROFILE_ON = False
        s_ms = [a.elapsed_time(b) for (name, a, b, _) in ops.PROFILE if name == "spmm"]
        s_meta = [meta for (name, _, _, meta) in ops.PROFILE if name == "spmm"]
        ach16 = (sum(m["bytes"] for m in s_meta) / (sum(s_ms) * 1e-3) / 1e9) if s_ms else float("nan")
        bd16 = {}
        for (name, a, b, _) in ops.PROFILE:
            bd16[name] = bd16.get(name, 0.0) + a.elapsed_time(b) / args.steps
        bf16_block = {"value": LAYERS * nnz_total / (ms16 / args.steps * 1e-3), "unit": "edges/s",
                      "ms_per_step": ms16 / args.steps, "what": "same step, Z = X W stored as bf16 (264 B/edge), fp32 accumulate",
                      "spmm_launch_ms": float(np.mean(s_ms)) if s_ms else None, "bytes_per_edge": 8 + DIM * 2,
                      "roofline": {"bound": "hbm", "achieved": ach16, "peak": hbm_peak, "unit": "GB/s",
                                   "frac": ach16 / hbm_peak}, "step_breakdown_ms": bd16}
        seq.set_feature_dtype("fp32")
        ops.PROFILE.clear()

    # ---- full-catalog scoring + top-10 for a block of this rank's users --------------------
    model.cache_propagation = True
    model.propagate()
    cu = min(args.catalog_users, u_hi - u_lo)
    users = torch.arange(u_lo, u_lo + cu, device=dev)
    # fp32 FFMA kernel (round 1's parity path), for reference next to the headline
    ffma_ms, _, _ = timed(lambda: model.recommend_top_k(n_users, n_items, 10, users=users, precision="fp32-ffma"), 1, 1)
    pairs_ffma = world * cu * n_items / (ffma_ms * 1e-3)
    # tensor-core scorers (tcgen05): more users per launch so the grid fills the chip.  fp32 = the 3xTF32 kernel
    # (fp32-accurate, the default of recommend_top_k: same parity tests as the FFMA kernel); bf16 = bf16 operands
    cu_tc = min(args.catalog_users * 4, u_hi - u_lo)
    users_tc = torch.arange(u_lo, u_lo + cu_tc, device=dev)
    cat_ms, _, _ = timed(lambda: model.recommend_top_k(n_users, n_items, 10, users=users_tc), 1, 1)
    pairs_per_s = world * cu_tc * n_items / (cat_ms * 1e-3)
    tc_ms, _, _ = timed(lambda: model.recommend_top_k(n_users, n_items, 10, users=users_tc, precision="bf16"), 1, 1)
    pairs_tc = world * cu_tc * n_items / (tc_ms * 1e-3)
    model.cache_propagation = False
    model.invalidate()

    if part is not None and part.heap is not None:
        part.heap.check()  # raises if any flag barrier timed out during the run
        torch.cuda.synchronize()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    line = {
        "metric": "propagation_edges_per_s", "value": value, "unit": "edges/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": mark_variant(workload_config(args.scale, world), args),
        "edges_per_s_per_gpu": value / world, "nnz_a_hat": nnz_total, "heavy_rows": heavy,
        "graph_build_s": build_s, "gpu_launches": launches, "clocks": clocks,
        "step_breakdown_ms": breakdown, "bf16_operands": bf16_block,
        "e2e": {"value": e2e_value, "unit": "edges/s", "h2d_bytes_per_step": 2 * PAIR_BATCH * 8,
                "d2h_bytes_per_step": PAIR_BATCH * 4, "ms_per_step": ms_e2e / args.steps},
        "roofline": roofline, "partition_parity": parity, "rank_sparse_ms": rank_sparse,
        "exchange": exchange_label if world > 1 else None, "nvlink": nvlink,
        "pairs": {"value": pairs_per_s, "unit": "pairs/s",
                  "what": "full-catalog BasicRS scoring + top-10, %d users x %d items per rank, fp32-accurate 3xTF32 tcgen05 "
                          "kernel (cbrs_score_catalog_topk_tf32x3; 1e-5 parity vs the oracle in tests/test_gpu_kernels.py)" % (cu_tc, n_items),
                  "ms": cat_ms, "tensor_flops_per_pair": 3 * 2 * CLF_UNITS[0] * CLF_UNITS[1],
                  "fp32_ffma": {"value": pairs_ffma, "unit": "pairs/s", "users_per_rank": cu, "ms": ffma_ms,
                                "what": "cbrs_score_catalog_topk (CUDA-core FFMA kernel, round 1's parity path)"},
                  # v3 kernel: h1 . [W2; b2] (K = 64 + 16 for the bias row) and relu(.) . w3 (N = 16) both on the tensor core
                  "bf16_tcgen05": {"value": pairs_tc, "unit": "pairs/s", "users_per_rank": cu_tc, "ms": tc_ms,
                                   "tensor_flops_per_pair": BF16_SCORER_FLOPS,
                                   "frac_of_bf16_peak": pairs_tc / world * BF16_SCORER_FLOPS / 1e12 / (peaks.get("bf16_tflops_sustained") or 1398.0)}},
    }
    if world == 1:
        # hybrid scorer towers (BASELINE config 4: Dense 768 -> 256 -> 64 over BERT rows, bf16): cbrs_dense_tc (tcgen05)
        # next to the fp32 FFMA kernel, 2^20 rows (3.2 GB of fp32 input: larger than L2).  Reported, not part of `value`.
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("cbrs_dense_tc_bench", os.path.join(REPO, "tools", "dense_tc_bench.py"))
            towers = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(towers)
            line["hybrid_towers"] = towers.run(1 << 20)
        except Exception as e:  # noqa: BLE001  (never let the side measurement take the headline line down)
            line["hybrid_towers"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if world == 1 and not args.no_small_configs:
        try:
            sc = small_configs(dev)
            line["small_configs"] = sc
            hyb = [c for c in sc if c["case"].startswith("config 4")]
            line["pairs"]["hybrid"] = [{"value": c["catalog_pairs_per_s_e2e"], "unit": "pairs/s", "ms": c["catalog_top10_e2e_ms"],
                                        "what": c["case"] + ": propagation + 6040 x 3706 full-catalog top-10, host ids in, host "
                                        "lists out (MovieLens-1M shape, BASELINE config 4)",
                                        "tolerance": "fp32: 2e-5 vs the oracle; bf16: 2e-3 vs an oracle rounding the same operands "
                                                     "(tests/test_zz_gpu_dense_tc.py, tests/test_gpu_models.py)"} for c in hyb]
        except Exception as e:  # noqa: BLE001
            line["small_configs"] = {"error": "%s: %s" % (type(e).__name__, e)}
    if not args.no_cpu_baseline and world == 1:
        threads = os.cpu_count() or 1
        r = cpu_reference_run(args.cpu_scale, 2, 1, threads)
        line["cpu_baseline"] = {"value": r["edges_per_s"], "unit": "edges/s", "cores": threads, "kind": "port",
                                "sample": r["sample"], "ms_per_step": r["ms_per_step"]}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def main():
    args = parse()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
