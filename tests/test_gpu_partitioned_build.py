"""Partitioned graph build, tested on one GPU.

A rank of a row partition builds only its own row blocks of the graph (RowPartition.build_graph,
graph.build_row_blocks): the COO streamed in pieces, the rank's entries selected in input order, each block built by
the whole build's kernels with a row offset, the degrees gathered between the two phases of the normalised view.

A. The edge-range generator: the pieces of any split of [0, E) make up ops.synth_bipartite bit for bit.
B. Row selection and the row histogram against numpy.
C. Every rank's slices equal DeviceGraph(...).<view>.row_slice(a, b) field for field, for 1-4 ranks emulated in one
   process (the loopback degree exchange), ragged and empty blocks, row-major and column-blocked schedules.
D. Two processes on one GPU, each building its own blocks with the real exchange (gloo): propagation of GCN, LightGCN,
   GraphSage and GAT and user-sharded catalog top-k equal the single-GPU model's bit for bit.
E. What has no partitioned form, and every whole-graph accessor, is refused before any launch."""
import json
import os

import numpy as np
import pytest
import torch
from scipy import sparse

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


def _directed_graph(n, n_entries, seed):
    """A directed multigraph on n nodes whose COO holds what a build must get right: duplicates with values other than
    1.0 (the order of their sum matters), explicit self loops, hub rows of many entries, isolated nodes."""
    rng = np.random.RandomState(seed)
    live = np.sort(rng.choice(n, size=n - n // 7, replace=False))        # the other nodes never appear: isolated
    hubs = live[rng.randint(0, live.size, size=3)]
    row = np.concatenate([live[rng.randint(0, live.size, size=n_entries)], np.repeat(hubs, 150)])
    col = live[rng.randint(0, live.size, size=row.size)]
    dup = rng.randint(0, row.size, size=row.size // 5)                    # repeated entries, new values
    loops = live[rng.randint(0, live.size, size=40)]
    row = np.concatenate([row, row[dup], loops, loops[:10]])
    col = np.concatenate([col, col[dup], loops, loops[:10]])
    val = rng.uniform(0.1, 3.0, size=row.size).astype(np.float32)
    perm = rng.permutation(row.size)
    return sparse.coo_matrix((val[perm], (row[perm], col[perm])), shape=(n, n))


# ------------------------------------------------------------------------------------------ A. edge-range generator
@pytest.mark.parametrize("scatter", [True, False], ids=["scattered", "unscattered"])
def test_edge_ranges_make_up_the_whole_generator_output(dev, scatter):
    from deep_cbrs_amar_renaissance_b200 import ops
    nu, ni, e = 5003, 1201, 40_000
    row, col = ops.synth_bipartite(nu, ni, e, 7, dev, scatter_items=scatter)
    for cuts in ([0, e], [0, 0, 1, 256, 255 * 33, 255 * 33, e - 1, e, e], list(range(0, e, 9973)) + [e]):
        parts = [ops.synth_bipartite_range(nu, ni, e, 7, lo, hi, dev, scatter_items=scatter)
                 for lo, hi in zip(cuts[:-1], cuts[1:])]
        ms = [hi - lo for lo, hi in zip(cuts[:-1], cuts[1:])]
        got_r = torch.cat([r[:m] for (r, _), m in zip(parts, ms)] + [r[m:] for (r, _), m in zip(parts, ms)])
        got_c = torch.cat([c[:m] for (_, c), m in zip(parts, ms)] + [c[m:] for (_, c), m in zip(parts, ms)])
        assert torch.equal(got_r, row) and torch.equal(got_c, col), cuts
    # the synthetic source streams the same entries in the same order
    from deep_cbrs_amar_renaissance_b200.graph import SyntheticSource
    pieces = [(r.clone(), c.clone()) for r, c, _ in SyntheticSource(nu, ni, e, 7, scatter, piece_edges=6000).pieces(dev)]
    assert torch.equal(torch.cat([p[0] for p in pieces]), row) and torch.equal(torch.cat([p[1] for p in pieces]), col)


def test_edge_range_outside_the_graph_is_refused(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    for lo, hi in ((-1, 5), (6, 5), (0, 101)):
        with pytest.raises(L.CbrsError, match="edge range"):
            ops.synth_bipartite_range(50, 20, 100, 1, lo, hi, dev)


# ------------------------------------------------------------------------------------ B. selection and histogram
def test_selection_keeps_input_order_and_histogram_counts_rows(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(3)
    n, n_rows = 30_000, 997
    row = rng.randint(0, n_rows + 40, size=n).astype(np.int32)      # some rows outside [0, n_rows)
    col = rng.randint(0, n_rows, size=n).astype(np.int32)
    val = rng.standard_normal(n).astype(np.float32)
    t = lambda a: torch.from_numpy(a).to(dev)  # noqa: E731
    hist = ops.coo_row_histogram(t(row), n_rows)
    keep = (row >= 0) & (row < n_rows)
    assert torch.equal(hist.cpu(), torch.from_numpy(np.bincount(row[keep], minlength=n_rows).astype(np.int64)))
    # accumulates over pieces
    ops.coo_row_histogram(t(row[:1000]), n_rows, hist)
    k2 = keep[:1000]
    want = np.bincount(row[keep], minlength=n_rows) + np.bincount(row[:1000][k2], minlength=n_rows)
    assert torch.equal(hist.cpu(), torch.from_numpy(want.astype(np.int64)))

    for lo, hi in ((100, 350), (0, 0), (n_rows + 100, n_rows + 200), (0, n_rows + 40), (500, 501)):
        for rebase in (False, True):
            m = (row >= lo) & (row < hi)
            cap = int(m.sum())
            out = [torch.full((cap + 3,), -7, dtype=torch.int32, device=dev) for _ in range(2)]
            out_v = torch.full((cap + 3,), -7.0, device=dev)
            cursor = torch.zeros(1, dtype=torch.int64, device=dev)
            for a in range(0, n, 7001):                                      # appended piece by piece
                b = min(a + 7001, n)
                ops.coo_select_rows(t(row[a:b]), t(col[a:b]), t(val[a:b]), lo, hi, out[0], out[1], out_v, cursor,
                                    rebase=rebase)
            assert int(cursor.item()) == cap
            assert torch.equal(out[0][:cap].cpu(), torch.from_numpy(row[m] - (lo if rebase else 0)))
            assert torch.equal(out[1][:cap].cpu(), torch.from_numpy(col[m]))
            assert torch.equal(out_v[:cap].cpu(), torch.from_numpy(val[m]))
            assert bool((out[0][cap:] == -7).all()) and bool((out_v[cap:] == -7.0).all())
    # capacity: nothing is written past it, the cursor still counts
    out = [torch.full((10,), -7, dtype=torch.int32, device=dev) for _ in range(2)]
    cursor = torch.zeros(1, dtype=torch.int64, device=dev)
    ops.coo_select_rows(t(row), t(col), None, 0, n_rows, out[0][:4], out[1][:4], None, cursor)
    assert int(cursor.item()) == int(keep.sum()) and bool((out[0][4:] == -7).all())
    assert torch.equal(out[0][:4].cpu(), torch.from_numpy(row[keep][:4]))


# ------------------------------------------------------------------------- C. slices equal the whole build's slices
def _same_slice(got, want, what):
    assert got.row_offset == want.row_offset and got.n_rows == want.n_rows and got.n_cols == want.n_cols, what
    assert got.blocking == want.blocking and got.chunk_edges == want.chunk_edges, what
    assert torch.equal(got.rowptr, want.rowptr), what + ": rowptr"
    assert torch.equal(got.colidx, want.colidx), what + ": colidx"
    assert (got.vals is None) == (want.vals is None), what + ": vals kept"
    if want.vals is not None:
        assert torch.equal(got.vals, want.vals), what + ": vals"
    for k in ("n_chunks", "n_heavy", "n_slots"):
        assert got.chunks[k] == want.chunks[k], what + ": " + k
    for k in ("chunk_row", "chunk_begin", "chunk_slot", "heavy_row", "heavy_slot_ptr", "chunk_len"):
        g, w = got.chunks[k], want.chunks[k]
        assert (g is None) == (w is None) and (g is None or torch.equal(g, w)), what + ": " + k


def _ragged(sizes, world, seed):
    """cuts that leave some blocks empty and put the others anywhere"""
    rng = np.random.RandomState(seed)
    out = [[] for _ in range(world)]
    base = 0
    for t, n in enumerate(sizes):
        cuts = [int(c) for c in np.sort(rng.randint(0, n + 1, size=world - 1))]
        if world > 1 and t == 0:
            cuts[0] = 0                         # rank 0 holds no row of the first type
        cuts = [0] + cuts + [n]
        for r in range(world):
            out[r].append((base + cuts[r], base + max(cuts[r + 1], cuts[r])))
        base += n
    return out


GRAPHS = ["directed", "synthetic"]


def _graph(kind, dev):
    """(source, DeviceGraph of the same COO, node counts by type)"""
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import CooSource, DeviceGraph, SyntheticSource
    if kind == "directed":
        adj = _directed_graph(1500, 12_000, 9)
        return CooSource(adj, piece_entries=2500), DeviceGraph.from_scipy(adj, dev, chunk_edges=16), [1000, 500]
    nu, ni, e = 2000, 600, 15_000
    row, col = ops.synth_bipartite(nu, ni, e, 5, dev, scatter_items=False)
    return SyntheticSource(nu, ni, e, 5, False, piece_edges=4000), DeviceGraph(row, col, None, nu + ni, 16), [nu, ni]


@pytest.mark.parametrize("blocking", [None, (97, 25)], ids=["row-major", "blocked"])
@pytest.mark.parametrize("kind", GRAPHS)
def test_every_rank_builds_the_rows_of_the_whole_build(dev, monkeypatch, kind, blocking):
    from deep_cbrs_amar_renaissance_b200 import graph as G
    from deep_cbrs_amar_renaissance_b200.distributed import balanced_ranges, block_ranges, edge_cost_prefix
    monkeypatch.setattr(G, "FORCED_BLOCKING", blocking)
    src, whole, sizes = _graph(kind, dev)
    n = sum(sizes)
    assert not whole.symmetric or kind == "synthetic"
    hist = G.row_histogram(src, dev)
    assert int(hist.sum().item()) == (whole.row.numel())
    norm, raw = whole.norm, whole.raw
    assert norm.chunks["n_heavy"] > 0
    if blocking:
        assert norm.blocking == tuple(blocking) and norm.chunks["chunk_len"] is not None
    cases = 0
    for world in (1, 2, 3, 4):
        est = G.estimated_rowptr(hist)
        for ranges in (balanced_ranges(sizes, world, edge_cost_prefix(est, sizes, G.blocking_policy(n)[1])),
                       block_ranges(sizes, world), _ragged(sizes, world, world)):
            loop = G.LoopbackDegrees(src, ranges, hist, dev)
            for rank in range(world):
                mine = [rg for rg in ranges[rank] if rg[1] > rg[0]]
                if not mine:
                    continue
                got = G.build_row_blocks(src, mine, loop, ("norm", "raw"), hist, chunk_edges=16, device=dev)
                for view, full in (("norm", norm), ("raw", raw)):
                    assert len(got[view]) == len(mine)
                    for (a, b), sl in zip(mine, got[view]):
                        _same_slice(sl, full.row_slice(a, b), "%s world %d rank %d rows [%d, %d)" % (view, world, rank, a, b))
                        cases += 1
    assert cases > 40


def test_hist_free_call_and_single_view(dev):
    """build_row_blocks makes its own histogram, and builds only the views asked for"""
    from deep_cbrs_amar_renaissance_b200 import graph as G
    src, whole, sizes = _graph("directed", dev)
    blocks = [(3, 700), (1000, 1400)]
    got = G.build_row_blocks(src, blocks, lambda local: pytest.fail("raw needs no degrees"), ("raw",), chunk_edges=16,
                             device=dev)
    assert list(got) == ["raw"]
    for (a, b), sl in zip(blocks, got["raw"]):
        _same_slice(sl, whole.raw.row_slice(a, b), "raw [%d, %d)" % (a, b))
    with pytest.raises(ValueError, match="views"):
        G.build_row_blocks(src, blocks, None, ("plain",), device=dev)


# ------------------------------------------------------------------------- D. two processes, one GPU, real exchange
FAMILIES = ["BasicGCN", "BasicLightGCN", "BasicGraphSage", "BasicGAT"]


def _model(name, adj, seed=31):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic
    set_seed(seed)
    kw = dict(embedding_dim=16, dense_units=[32, 16], clf_units=[16, 16], final_node="concatenation")
    if name == "BasicLightGCN":
        m = basic.BasicLightGCN(adj, n_layers=2, **kw)
    else:
        m = getattr(basic, name)(adj, n_hiddens=[16, 16], **kw)
    m.build_weights()
    return m


def _worker(rank, world, init, out_dir, sizes):
    import torch.distributed as dist
    from deep_cbrs_amar_renaissance_b200 import graph as G
    from deep_cbrs_amar_renaissance_b200.distributed import RowPartition
    from deep_cbrs_amar_renaissance_b200.selfcheck import small_graph
    torch.cuda.set_device(0)
    dist.init_process_group("gloo", init_method=init, rank=rank, world_size=world)
    dev = torch.device("cuda", 0)
    adj = small_graph(sizes[0], sizes[1], 6000, seed=5)
    nu, ni = sizes
    failures, cases = [], 0
    try:
        for blocking in (None, (97, 25)):
            G.FORCED_BLOCKING = blocking
            hist = G.row_histogram(adj, dev)
            part = RowPartition(sizes, exchange="nccl", final_types=[1], balance_rowptr=G.estimated_rowptr(hist),
                                balance_min_len=G.blocking_policy(nu + ni)[1])
            graph = part.build_graph(G.CooSource(adj, piece_entries=3000), views=("norm", "raw"), hist=hist)
            assert isinstance(graph, G.PartitionedGraph) and graph.shape == (nu + ni, nu + ni)
            u_lo, u_hi = part.ranges[rank][0]
            users = torch.arange(u_lo, u_hi, dtype=torch.int64, device=dev)
            for name in FAMILIES:
                tag = "%s %s" % (name, "blocked" if blocking else "row-major")
                ref = _model(name, adj)
                want = ref.propagate().clone()
                want_ids, want_sc = ref.recommend_top_k(nu, ni, k=10, users=users)
                model = _model(name, graph)
                part.attach(model.gnn.gnn_layers)
                got = model.propagate()
                got_ids, got_sc = model.recommend_top_k(nu, ni, k=10, users=users)
                torch.cuda.synchronize()
                rows = [rg for rg in part.mine] + [(nu, nu + ni)]             # own blocks + every item row
                for what, ok in [("rows [%d, %d)" % (a, b), torch.equal(got[a:b], want[a:b])) for a, b in rows] + \
                        [("top-k ids", torch.equal(got_ids, want_ids)), ("top-k scores", torch.equal(got_sc, want_sc))]:
                    cases += 1
                    if not ok:
                        failures.append("%s rank %d: %s differ" % (tag, rank, what))
            part.close()
    except Exception as e:  # noqa: BLE001
        failures.append("rank %d: %r" % (rank, e))
    finally:
        G.FORCED_BLOCKING = None
        with open(os.path.join(out_dir, "rank%d.json" % rank), "w") as f:
            json.dump({"cases": cases, "failures": failures}, f)
        dist.destroy_process_group()


def test_two_processes_on_one_gpu_build_and_propagate_bit_identically(dev, tmp_path):
    """Both ranks share cuda:0 and a gloo group; each builds only its own row blocks, the degrees travel by broadcast."""
    import torch.multiprocessing as mp
    sizes = (301, 199)
    mp.spawn(_worker, args=(2, "file://" + str(tmp_path / "store"), str(tmp_path), sizes), nprocs=2, join=True)
    for r in range(2):
        res = json.load(open(tmp_path / ("rank%d.json" % r)))
        assert not res["failures"], res["failures"]
        assert res["cases"] == 2 * len(FAMILIES) * 5


# ------------------------------------------------------------------------------------------------ E. refusals
def _refused(call, match):
    from deep_cbrs_amar_renaissance_b200 import ops
    torch.cuda.synchronize()
    launches = ops.LAUNCHES
    with pytest.raises(NotImplementedError, match=match):
        call()
    assert ops.LAUNCHES == launches


def test_what_a_partitioned_build_cannot_serve_is_refused_before_any_launch(dev):
    from deep_cbrs_amar_renaissance_b200.graph import PartitionedGraph
    from deep_cbrs_amar_renaissance_b200.models import basic
    nu, ni = 40, 30
    g = PartitionedGraph(nu + ni, ("norm", "raw"))
    for what, call in (("norm", lambda: g.norm), ("raw", lambda: g.raw), ("plain", lambda: g.plain),
                       ("dgcf", lambda: g.dgcf), ("symmetric", lambda: g.symmetric),
                       ("transposed", lambda: g.transposed()), ("row_subset", lambda: g.row_subset(torch.arange(3)))):
        _refused(call, "partitioned graph build")
    u, i = np.arange(8), np.arange(8) + nu
    y = np.ones(8, np.float32)
    m = basic.BasicGCN(g, n_hiddens=[8, 8], embedding_dim=8, dense_units=[16], clf_units=[8])
    m.build_weights()
    m.compile()
    _refused(lambda: m.train_on_batch((u, i), y), "training on a partitioned graph build")
    _refused(lambda: m.make_graphed_train_step(8), "training on a partitioned graph build")
    batches = [((u, i), y), ((u, i), y)]
    seq = type("S", (), {"__len__": lambda s: 2, "__getitem__": lambda s, k: batches[k]})()
    _refused(lambda: m.fit(seq, epochs=1), "training on a partitioned graph build")
    _refused(lambda: m.fit(seq, epochs=1, cuda_graph=True), "training on a partitioned graph build")
    # with no partition attached, the model's call reaches the whole-graph view and stops there
    _refused(lambda: m((u, i)), "partitioned graph build")
    _refused(lambda: basic.BasicRGCN(g, n_hiddens=[8, 8], embedding_dim=8, dense_units=[16], clf_units=[8]), "RGCN")
    _refused(lambda: basic.BasicDGCF(g, embedding_dim=8, n_layers=2, dense_units=[16], clf_units=[8]), "DGCFConv")
    n_props = 20
    ip = PartitionedGraph(ni + n_props, ("norm",))
    up = PartitionedGraph(nu + n_props, ("norm",))
    _refused(lambda: basic.BasicTSGCN(nu, ni, (g, ip), n_hiddens=[8, 8], embedding_dim=8, dense_units=[16],
                                      clf_units=[8]), "TwoStep")
    _refused(lambda: basic.BasicTWGCN(nu, ni, (g, ip, up), n_hiddens=[8, 8], embedding_dim=8, dense_units=[16],
                                      clf_units=[8]), "TwoWay")
