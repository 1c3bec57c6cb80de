"""GPU: the per-batch call computes its last GCN / LightGCN layer only at the rows the batch scores
(graph.CsrSubset, cbrs_csr_subset_*).  The scores must equal, bit for bit, scoring the full propagation; the needed
rows of the last layer must equal the full layer's rows bit for bit; the subset descriptor must equal a numpy
restatement of its definition; and every call that hands the table out (propagate, the cache, CUDA-graph replays)
must keep computing every row."""
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


@pytest.fixture
def forced():
    """force the size condition of the policy on; restore both overrides afterwards"""
    from deep_cbrs_amar_renaissance_b200 import graph
    saved = graph.FORCED_SUBSET, graph.FORCED_BLOCKING
    graph.FORCED_SUBSET = True
    yield graph
    graph.FORCED_SUBSET, graph.FORCED_BLOCKING = saved


N_USERS, N_ITEMS = 300, 200


def hub_graph(seed=3):
    """bipartite, symmetric, with hub rows: items 0-4 are linked to every user and user 0 to every item, so that with
    16-edge chunks and 32-column windows there are multi-chunk rows and column-blocked rows of many slots"""
    rng = np.random.RandomState(seed)
    keys = np.unique(rng.randint(0, N_USERS * N_ITEMS, size=2500))
    u, i = keys // N_ITEMS, keys % N_ITEMS
    u = np.concatenate([u, np.repeat(np.arange(N_USERS), 5), np.zeros(N_ITEMS, np.int64)])
    i = np.concatenate([i, np.tile(np.arange(5), N_USERS), np.arange(N_ITEMS)])
    keys = np.unique(u * N_ITEMS + i)
    u, i = keys // N_ITEMS, keys % N_ITEMS + N_USERS
    r = np.concatenate([u, i]).astype(np.int32)
    c = np.concatenate([i, u]).astype(np.int32)
    n = N_USERS + N_ITEMS
    return sparse.coo_matrix((np.ones(len(r), np.float32), (r, c)), shape=(n, n))


def _device_graph(blocked, graph):
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    graph.FORCED_BLOCKING = (32, 48) if blocked else (0, 0)
    return DeviceGraph.from_scipy(hub_graph(), chunk_edges=16)


def _model(kind, dtype, blocked, graph):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.layers import ReductionLayer
    from deep_cbrs_amar_renaissance_b200.models import basic
    set_seed(7)
    adj = _device_graph(blocked, graph)
    kw = dict(embedding_dim=32, dense_units=[48, 48], clf_units=[64, 64])
    if kind == "gcn":
        model = basic.BasicGCN(adj, n_hiddens=[32, 32, 32], final_node="concatenation", **kw)
    else:
        model = basic.BasicLightGCN(adj, n_layers=3, **kw)
        seq = model.gnn.gnn_layers
        seq.final_node = "concatenation"          # BasicLightGCN forces 'mean' (gnn.py:378); the stack supports both
        seq.reduce = ReductionLayer("concatenation")
    if dtype == "bf16":
        model.gnn.gnn_layers.set_feature_dtype("bf16")
    return model


def _batches():
    rng = np.random.RandomState(11)
    n = N_USERS + N_ITEMS
    u = rng.randint(0, N_USERS, size=96)
    i = rng.randint(0, N_ITEMS, size=96) + N_USERS
    u[:10] = u[10]                                    # duplicate ids
    i[20:30] = u[20:30]                               # ids shared between u and i
    every = np.arange(n)
    return {"random": (u, i), "every_row": (every, every[::-1].copy()), "one_pair": (u[:1], i[:1]),
            "hubs": (np.zeros(4, np.int64), np.arange(4) + N_USERS)}


def _full(model, graph):
    """the full propagation's table (what every pruned call must agree with)"""
    graph.FORCED_SUBSET = False
    emb = model.gnn(None).clone()
    graph.FORCED_SUBSET = True
    return emb


@pytest.mark.parametrize("kind,dtype", [("gcn", "fp32"), ("gcn", "bf16"), ("lightgcn", "fp32")])
@pytest.mark.parametrize("blocked", [False, True])
def test_pruned_call_is_bit_identical(dev, forced, kind, dtype, blocked):
    from deep_cbrs_amar_renaissance_b200 import ops
    model = _model(kind, dtype, blocked, forced)
    seq = model.gnn.gnn_layers
    csr = seq.adj_matrix.norm
    if blocked:
        assert csr.blocking == (32, 48) and csr.chunks["n_heavy"] > 0 and csr.desc.chunk_len
    assert seq.last_layer_subset()
    model(_batches()["random"])              # builds the scorer's weights
    full = _full(model, forced)
    last = slice(full.shape[1] - 32, full.shape[1])
    lens = (csr.rowptr[1:] - csr.rowptr[:-1]).cpu().numpy()
    for name, (u, i) in _batches().items():
        ops.PROFILE.clear()
        ops.PROFILE_ON = True
        try:
            got = model((u, i))
        finally:
            ops.PROFILE_ON = False
        torch.cuda.synchronize()
        table = seq._buf.clone()
        want = model.embed_recommend(full, (u, i))
        assert torch.equal(got, want), name
        needed = np.unique(np.concatenate([u, i]))
        idx = torch.from_numpy(needed).to(dev)
        assert torch.equal(table[idx][:, last], full[idx][:, last]), name
        assert torch.equal(table[:, :last.start], full[:, :last.start]), name   # layers before the last are full
        meta = [m for (k, _, _, m) in ops.PROFILE if k == "spmm"][-1]         # what the last launch processed
        assert meta["rows"] == len(needed) and meta["nnz"] == int(lens[needed].sum()), name
        ops.PROFILE.clear()


def _expected_subset(full, needed):
    """numpy restatement: the needed rows' chunks in list order; needed heavy rows in order, slots renumbered
    compactly keeping each row's slot order"""
    row = full["chunk_row"].cpu().numpy()
    keep = needed[row]
    hrow = full["heavy_row"].cpu().numpy()
    hptr = full["heavy_slot_ptr"].cpu().numpy()
    hkeep = needed[hrow]
    new_ptr = [0]
    slot_map = {}
    for h in np.nonzero(hkeep)[0]:
        for s in range(hptr[h], hptr[h + 1]):
            slot_map[s] = new_ptr[-1] + (s - hptr[h])
        new_ptr.append(new_ptr[-1] + hptr[h + 1] - hptr[h])
    slot = full["chunk_slot"].cpu().numpy()[keep]
    exp = dict(chunk_row=row[keep], chunk_begin=full["chunk_begin"].cpu().numpy()[keep],
               chunk_slot=np.array([slot_map[s] if s >= 0 else -1 for s in slot], np.int32),
               heavy_row=hrow[hkeep], heavy_slot_ptr=np.array(new_ptr, np.int64))
    if full["chunk_len"] is not None:
        exp["chunk_len"] = full["chunk_len"].cpu().numpy()[keep]
    return exp


@pytest.mark.parametrize("blocked", [False, True])
def test_subset_descriptor_matches_its_definition(dev, forced, blocked):
    csr = _device_graph(blocked, forced).norm
    n = csr.n_rows
    rng = np.random.RandomState(5)
    cases = [rng.randint(0, n, size=40), np.arange(n), np.array([0]), np.array([], np.int64),
             np.array([-1, n, n + 7, 3, 3, N_USERS])]             # ids outside [0, n) select nothing
    lens = (csr.rowptr[1:] - csr.rowptr[:-1]).cpu().numpy()
    for ids in cases:
        sub = csr.row_subset(torch.from_numpy(ids.astype(np.int64)).to(dev))
        needed = np.zeros(n, bool)
        valid = ids[(ids >= 0) & (ids < n)]
        needed[valid] = True
        exp = _expected_subset(csr.chunks, needed)
        c = sub.chunks
        assert c["n_chunks"] == len(exp["chunk_row"]) and c["n_heavy"] == len(exp["heavy_row"])
        assert c["n_slots"] == exp["heavy_slot_ptr"][-1]
        for key, want in exp.items():
            np.testing.assert_array_equal(c[key].cpu().numpy(), want, err_msg=key)
        assert sub.n_needed == needed.sum() and sub.nnz == int(lens[needed].sum())
        assert (c["chunk_len"] is None) == (not blocked)


def test_cached_propagation_stays_full(dev, forced):
    model = _model("gcn", "fp32", True, forced)
    u, i = _batches()["random"]
    model((u, i))
    full = _full(model, forced)
    model.cache_propagation = True
    emb = model.propagate()                  # cached from here on
    assert torch.equal(emb, full)
    model.cache_propagation = False
    model((u[:3], i[:3]))                    # pruned: overwrites the shared table, drops the cache
    assert model._cached is None
    model.cache_propagation = True
    assert torch.equal(model.propagate(), full)
    assert torch.equal(model((u, i)), model.embed_recommend(full, (u, i)))
    ids, vals = model.recommend_top_k(N_USERS, N_ITEMS, 5)
    model.cache_propagation = False
    model.invalidate()
    ids2, vals2 = model.recommend_top_k(N_USERS, N_ITEMS, 5)
    assert torch.equal(ids, ids2) and torch.equal(vals, vals2)


def test_graphed_forward_replays_the_full_layer(dev, forced):
    from deep_cbrs_amar_renaissance_b200.graphed import GraphedForward
    model = _model("gcn", "fp32", True, forced)
    u, i = _batches()["random"]
    g = GraphedForward(model, len(u))        # the capture takes the full path (any ids may come)
    full = _full(model, forced)
    rng = np.random.RandomState(2)
    for _ in range(3):
        u2 = rng.randint(0, N_USERS, size=len(u))
        i2 = rng.randint(0, N_ITEMS, size=len(u)) + N_USERS
        got = g((u2, i2)).clone()
        assert torch.equal(got, model.embed_recommend(full, (u2, i2)))


def test_other_stacks_keep_the_full_path(dev, forced):
    from deep_cbrs_amar_renaissance_b200.models import basic
    adj = _device_graph(False, forced)
    kw = dict(embedding_dim=16, dense_units=[16], clf_units=[16])
    assert not basic.BasicGAT(adj, n_hiddens=[16, 16], final_node="concatenation", **kw).gnn.gnn_layers.last_layer_subset()
    assert not basic.BasicGraphSage(adj, n_hiddens=[16, 16], final_node="concatenation", **kw).gnn.gnn_layers.last_layer_subset()
    assert not basic.BasicGCN(adj, n_hiddens=[16, 16], final_node="mean", **kw).gnn.gnn_layers.last_layer_subset()
    assert not basic.BasicLightGCN(adj, n_layers=2, **kw).gnn.gnn_layers.last_layer_subset()   # 'mean'
    forced.FORCED_SUBSET = None
    assert not basic.BasicGCN(adj, n_hiddens=[16, 16], **kw).gnn.gnn_layers.last_layer_subset()  # small graph
