"""GPU parity: every kernel of the C ABI against the CPU oracle on the same seeded inputs.
Integer outputs bit-exact; float outputs within 1e-5 of the tensor scale (north star)."""
import os

import numpy as np
import pytest
import torch
from scipy import sparse

from oracle import graph as og
from oracle import layers as ol
from tests.helpers import assert_close, glorot, random_bipartite

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


def _t(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(dev) if dtype is None else t.to(dev, dtype)


# ------------------------------------------------------------------ sort / scan
@pytest.mark.parametrize("n,bits", [(1, 8), (31, 8), (4096, 16), (4097, 24), (100003, 40), (1 << 20, 64)])
def test_radix_sort_is_stable(dev, n, bits):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(n)
    hi = min(bits, 62)
    keys = rng.randint(0, 1 << 62, size=n, dtype=np.int64) & ((1 << hi) - 1)
    if n >= 8:  # force duplicates so stability is observable
        src = rng.randint(0, n, size=n // 2)
        dst = rng.randint(0, n, size=n // 2)
        keys[dst] = keys[src]
    k, p = ops.sort_pairs_u64(_t(keys, dev), _t(np.arange(n, dtype=np.int32), dev), bits)
    order = np.argsort(keys, kind="stable")
    assert np.array_equal(k.cpu().numpy(), keys[order])
    assert np.array_equal(p.cpu().numpy(), order.astype(np.int32))


def test_sort_ignores_bits_above_key_bits_only_if_zero(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    keys = np.array([3, 1, 2, 1, 0], np.int64)
    k, p = ops.sort_pairs_u64(_t(keys, dev), _t(np.arange(5, dtype=np.int32), dev), 2)
    assert k.cpu().tolist() == [0, 1, 1, 2, 3] and p.cpu().tolist() == [4, 1, 3, 2, 0]


# ------------------------------------------------------------------ graph build
def _golden_adj(golden_dir, case):
    g = np.load(os.path.join(golden_dir, case, "golden.npz"))
    return sparse.coo_matrix((g["adj_data"], (g["adj_row"], g["adj_col"])), shape=tuple(g["adj_shape"]))


def _check_graph(adj, dev, chunk_edges=1024):
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=chunk_edges)
    want = og.gcn_filter(adj)
    norm = g.norm
    assert np.array_equal(norm.rowptr.cpu().numpy(), want.indptr.astype(np.int64))
    assert np.array_equal(norm.colidx.cpu().numpy(), want.indices.astype(np.int32))
    assert np.array_equal(norm.vals.cpu().numpy(), want.data), "normalised values must be bit-exact for 0/1 graphs"
    ptr, idx, _ = og.reorder_raw(adj)
    raw = g.raw
    assert np.array_equal(raw.rowptr.cpu().numpy(), ptr) and np.array_equal(raw.colidx.cpu().numpy(), idx)
    return g


@pytest.mark.parametrize("case", ["ui_small", "uip_small", "hybrid_small"])
def test_graph_build_matches_reference_fixtures(dev, golden_dir, case):
    adj = _golden_adj(golden_dir, case)
    g = _check_graph(adj, dev)
    # and against scipy's own duplicate summing of the reference's matrix
    gold = np.load(os.path.join(golden_dir, case, "golden.npz"))
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    rowptr, colidx, vals = ops.graph_build_csr(g.row, g.col, g.val, g.n_nodes, L.GRAPH_DEDUP_SUM)
    assert np.array_equal(rowptr.cpu().numpy(), gold["csr_indptr"].astype(np.int64))
    assert np.array_equal(colidx.cpu().numpy(), gold["csr_indices"]) and np.array_equal(vals.cpu().numpy(), gold["csr_data"])


@pytest.mark.parametrize("shape", [(7, 5, 20, 0, 0, 0), (300, 200, 9000, 150, 700, 60), (6040, 3706, 570000, 0, 0, 0),
                                   (6040, 3706, 570000, 17554, 70341, 400)])
def test_graph_build_random(dev, shape):
    u, i, pos, p, links, dups = shape
    _check_graph(random_bipartite(u, i, pos, seed=pos, n_props=p, n_links=links, dup_links=dups), dev)


def test_graph_build_edge_cases(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    # empty adjacency: A_hat = I
    empty = sparse.coo_matrix((5, 5), dtype=np.float32)
    _check_graph(empty, dev)
    # existing self loops and isolated nodes, non-unit values
    rows = np.array([0, 0, 2, 2, 2, 4], np.int32)
    cols = np.array([0, 3, 2, 2, 0, 1], np.int32)
    vals = np.array([1, 1, 1, 1, 1, 1], np.float32)
    adj = sparse.coo_matrix((vals, (rows, cols)), shape=(6, 6))
    _check_graph(adj, dev)
    # DROP_DIAG: the GAT edge set without the appended loops
    r, c, v = ops.graph_build_csr(_t(rows, dev), _t(cols, dev), None, 6, L.GRAPH_DROP_DIAG)
    assert r.cpu().tolist() == [0, 1, 1, 2, 2, 3, 3] and c.cpu().tolist() == [3, 0, 1]
    # out-of-range entries are dropped, not written out of bounds
    r, c, v = ops.graph_build_csr(_t(np.array([0, 9], np.int32), dev), _t(np.array([1, 1], np.int32), dev), None, 3, 0)
    assert r.cpu().tolist() == [0, 1, 1, 1] and c.cpu().tolist() == [1]
    # float duplicates are summed in input order
    rr = np.zeros(4, np.int32)
    vv = np.array([1e8, 1.0, -1e8, 1.0], np.float32)
    _, _, v = ops.graph_build_csr(_t(rr, dev), _t(rr, dev), _t(vv, dev), 1, L.GRAPH_DEDUP_SUM)
    acc = np.float32(0)
    for x in vv:
        acc = np.float32(acc + x)
    assert v.cpu().numpy()[0] == acc


def test_chunk_decomposition(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    lens = np.array([0, 5, 8, 9, 17, 1, 0, 24, 3], np.int64)
    rowptr = np.concatenate([[0], np.cumsum(lens)])
    c = ops.build_chunks(_t(rowptr, dev), 8)
    nc = np.where(lens <= 8, 1, -(-lens // 8))
    assert c["n_chunks"] == nc.sum() and c["n_heavy"] == (nc > 1).sum() and c["n_slots"] == nc[nc > 1].sum()
    want_row = np.repeat(np.arange(len(lens)), nc)
    assert np.array_equal(c["chunk_row"].cpu().numpy(), want_row)
    k_in_row = np.arange(nc.sum()) - np.repeat(np.cumsum(nc) - nc, nc)
    assert np.array_equal(c["chunk_begin"].cpu().numpy(), rowptr[want_row] + 8 * k_in_row)
    slot = c["chunk_slot"].cpu().numpy()
    assert (slot[np.repeat(nc, nc) == 1] == -1).all()
    assert np.array_equal(slot[slot >= 0], np.arange(c["n_slots"]))
    assert c["heavy_row"].cpu().tolist() == [3, 4, 7] and c["heavy_slot_ptr"].cpu().tolist() == [0, 2, 5, 8]


# ------------------------------------------------------------------ propagation
@pytest.mark.parametrize("d", [8, 16, 32, 48, 128, 100, 130, 6, 256])
@pytest.mark.parametrize("chunk_edges", [16, 1024])
def test_spmm_weighted_matches_oracle(dev, d, chunk_edges):
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    adj = random_bipartite(120, 40, 2500, seed=d, n_props=20, n_links=100, dup_links=10)
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=chunk_edges)
    rng = np.random.RandomState(d)
    x = rng.standard_normal((adj.shape[0], d)).astype(np.float32)
    b = rng.standard_normal(d).astype(np.float32)
    a_hat = og.gcn_filter(adj)
    assert g.norm.chunks["n_heavy"] > 0 or chunk_edges > 16
    out = torch.empty(adj.shape[0], d, device=dev)
    ops.spmm(g.norm, _t(x, dev), out)
    assert_close(out.cpu().numpy(), ol.lightgcn_conv(x, a_hat), what="A_hat x")
    ops.spmm(g.norm, _t(x, dev), out, bias=_t(b, dev), relu=True)
    assert_close(out.cpu().numpy(), np.maximum(a_hat @ x + b, 0), what="relu(A_hat x + b)")


@pytest.mark.parametrize("agg,name", [(1, "sum"), (2, "mean")])
@pytest.mark.parametrize("chunk_edges", [8, 1024])
def test_spmm_aggregators_ignore_values_and_keep_duplicates(dev, agg, name, chunk_edges):
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    adj = random_bipartite(50, 30, 600, seed=3, n_props=12, n_links=80, dup_links=25)
    adj = sparse.coo_matrix((adj.data, (adj.row, adj.col)), shape=(adj.shape[0] + 3, adj.shape[1] + 3))  # isolated tail
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=chunk_edges)
    x = np.random.RandomState(1).standard_normal((adj.shape[0], 32)).astype(np.float32)
    ptr, idx, _ = og.reorder_raw(adj)
    out = torch.full((adj.shape[0], 32), 7.0, device=dev)
    ops.spmm(g.raw, _t(x, dev), out, agg=agg)
    assert_close(out.cpu().numpy(), ol.sage_aggregate(x, ptr, idx, name), what=name)
    assert (out[-3:] == 0).all()


def test_spmm_writes_into_a_column_slice(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    adj = random_bipartite(40, 25, 400, seed=5)
    g = DeviceGraph.from_scipy(adj, dev)
    x = np.random.RandomState(2).standard_normal((65, 16)).astype(np.float32)
    buf = torch.full((65, 48), -1.0, device=dev)
    buf[:, :16] = _t(x, dev)
    ops.spmm(g.norm, buf[:, :16], buf[:, 16:32])
    assert_close(buf[:, 16:32].cpu().numpy(), ol.lightgcn_conv(x, og.gcn_filter(adj)))
    assert (buf[:, 32:] == -1).all() and np.array_equal(buf[:, :16].cpu().numpy(), x)


def test_spmm_row_slices_are_bit_identical_to_the_full_run(dev):
    """Rank-count independence (SURVEY 8e): a row partition computes the same bits."""
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    adj = random_bipartite(200, 50, 5000, seed=9)
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=32)
    x = _t(np.random.RandomState(3).standard_normal((250, 64)).astype(np.float32), dev)
    full = torch.empty(250, 64, device=dev)
    ops.spmm(g.norm, x, full, relu=True)
    for cuts in ([0, 250], [0, 100, 250], [0, 7, 130, 131, 250]):
        part = torch.empty(250, 64, device=dev)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            ops.spmm(g.norm.row_slice(r0, r1), x, part[r0:r1], relu=True)
        assert torch.equal(part, full)


@pytest.mark.parametrize("h", [8, 16, 32, 128, 20])
@pytest.mark.parametrize("chunk_edges", [8, 1024])
def test_gat_matches_oracle(dev, h, chunk_edges):
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    adj = random_bipartite(60, 30, 900, seed=h, n_props=10, n_links=60, dup_links=20)
    # add a few explicit self loops: the layer must drop them and add its own
    rows = np.concatenate([adj.row, [0, 5, 5]]).astype(np.int32)
    cols = np.concatenate([adj.col, [0, 5, 5]]).astype(np.int32)
    adj = sparse.coo_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=adj.shape)
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=chunk_edges)
    rng = np.random.RandomState(h)
    f = 12
    x = rng.standard_normal((adj.shape[0], f)).astype(np.float32)
    w, a_s, a_n = glorot(rng, (f, h)), rng.standard_normal(h).astype(np.float32), rng.standard_normal(h).astype(np.float32)
    b = rng.standard_normal(h).astype(np.float32)
    ptr, idx, _ = og.reorder_raw(adj)
    want = ol.gat_conv(x, ptr, idx, w, a_s, a_n, b)
    z, p, q = ops.dense(_t(x, dev), _t(w, dev), rowop=L.ROWOP_ATTN, a_self=_t(a_s, dev), a_neigh=_t(a_n, dev))
    assert_close(z.cpu().numpy(), x @ w, what="z")
    assert_close(p.cpu().numpy(), (x @ w) @ a_s, what="p")
    out = torch.empty(adj.shape[0], h, device=dev)
    ops.gat(g.raw, z, p, q, out, bias=_t(b, dev), relu=True)
    assert_close(out.cpu().numpy(), want, what="gat")


# ------------------------------------------------------------------ dense
@pytest.mark.parametrize("m,f1,f2,n", [(1, 3, 0, 1), (1000, 48, 0, 48), (777, 96, 0, 64), (513, 64, 64, 64),
                                        (300, 768, 0, 256), (129, 17, 5, 130), (2048, 64, 0, 1), (50, 16, 16, 200)])
@pytest.mark.parametrize("act", [None, "relu", "sigmoid"])
def test_dense_matches_oracle(dev, m, f1, f2, n, act):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(m + n)
    x1 = rng.standard_normal((m, f1)).astype(np.float32)
    x2 = rng.standard_normal((m, f2)).astype(np.float32) if f2 else None
    w, b = glorot(rng, (f1 + f2, n)), rng.standard_normal(n).astype(np.float32)
    xin = np.concatenate([x1, x2], 1) if f2 else x1
    got = ops.dense(_t(x1, dev), _t(w, dev), _t(b, dev), act, x2=_t(x2, dev) if f2 else None)
    assert_close(got.cpu().numpy(), ol.dense(xin, w, b, act), what="dense")


def test_dense_fused_gather_concat_and_l2norm(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(0)
    table = rng.standard_normal((500, 48)).astype(np.float32)
    other = rng.standard_normal((90, 24)).astype(np.float32)
    i1 = rng.randint(0, 500, size=1234)
    i2 = rng.randint(0, 90, size=1234)
    w, b = glorot(rng, (72, 40)), rng.standard_normal(40).astype(np.float32)
    got = ops.dense(_t(table, dev), _t(w, dev), _t(b, dev), "relu", x2=_t(other, dev), idx1=_t(i1, dev), idx2=_t(i2, dev))
    want = ol.dense(np.concatenate([table[i1], other[i2]], 1), w, b, "relu")
    assert_close(got.cpu().numpy(), want, what="gather+concat+dense")
    # GraphSage epilogue: l2-normalise then relu; narrow (fused) and wide (two-pass) outputs
    for n in (40, 200):
        w2, b2 = glorot(rng, (48, n)), rng.standard_normal(n).astype(np.float32)
        got = ops.dense(_t(table, dev), _t(w2, dev), _t(b2, dev), "relu", rowop=L.ROWOP_L2NORM)
        pre = table @ w2 + b2
        want = np.maximum(pre / np.sqrt(np.maximum((pre * pre).sum(1, keepdims=True), 1e-12)), 0)
        assert_close(got.cpu().numpy(), want, what="l2norm n=%d" % n)
    # strided output slice
    buf = torch.zeros(500, 100, device=dev)
    ops.dense(_t(table, dev), _t(w2[:, :32].copy(), dev), None, None, out=buf[:, 10:42])
    assert_close(buf[:, 10:42].cpu().numpy(), table @ w2[:, :32])
    assert (buf[:, :10] == 0).all() and (buf[:, 42:] == 0).all()


def test_ops_refuse_cpu_tensors(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib as L
    from deep_cbrs_amar_renaissance_b200 import ops
    with pytest.raises(L.CbrsError):
        ops.dense(torch.zeros(4, 4), torch.zeros(4, 4))
    with pytest.raises(L.CbrsError):
        ops.dense(torch.zeros(4, 4, device=dev), torch.zeros(5, 4, device=dev))


def test_reduce_and_gather(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(1)
    hs = [rng.standard_normal((300, 24)).astype(np.float32) for _ in range(4)]
    ths = [_t(h, dev) for h in hs]
    assert_close(ops.reduce_layers(ths, divide_by=4.0).cpu().numpy(), ol.reduce_layers(hs, "mean"), rtol=1e-6)
    assert_close(ops.reduce_layers(ths).cpu().numpy(), ol.reduce_layers(hs, "sum"), rtol=1e-6)
    w = [1.0, 0.5, 2.0, 1.5]
    assert_close(ops.reduce_layers(ths, coefs=[v * v for v in w]).cpu().numpy(), ol.reduce_layers(hs, "w-sum", w), rtol=1e-6)
    idx = rng.randint(0, 300, size=77)
    assert np.array_equal(ops.gather_rows(ths[0], _t(idx, dev)).cpu().numpy(), hs[0][idx])


# ------------------------------------------------------------------ top-k
@pytest.mark.parametrize("n_users,n_items,k", [(1, 1, 1), (37, 3706, 10), (64, 1000, 5), (3, 7, 10), (5, 70000, 10)])
def test_topk_rows_is_bit_exact_with_stable_sort(dev, n_users, n_items, k):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(n_items)
    s = rng.random_sample((n_users, n_items)).astype(np.float32)
    s[:, ::3] = np.round(s[:, ::3], 2)  # plenty of exact ties
    if n_items > 10:
        s[0, :] = 0.5  # all tied: ids must be 0..k-1
        s[-1, 5] = np.inf
        s[-1, 6] = -np.inf
    ids, vals = ops.topk_rows(_t(s, dev), k)
    kk = min(k, n_items)
    want_ids, want_vals = ol.top_k_catalog(s, kk)
    assert np.array_equal(ids.cpu().numpy()[:, :kk], want_ids)
    assert np.array_equal(vals.cpu().numpy()[:, :kk], want_vals)
    assert (ids.cpu().numpy()[:, kk:] == -1).all()


def test_topk_pairs_matches_the_reference_semantics(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(5)
    n, n_users = 50000, 613
    u = rng.randint(0, n_users, size=n).astype(np.int64)
    i = rng.randint(0, 900, size=n) + n_users
    s = np.round(rng.random_sample(n), 3).astype(np.float32)  # ties inside users
    for k in (5, 10):
        keep = ops.topk_pairs(_t(u, dev), _t(s, dev), n_users, k).cpu().numpy()
        uu, ii, ss, rows = ol.top_k_pairs(u, i, s, k)
        assert np.array_equal(keep, rows)


def test_top_k_predictions_frame(dev):
    from deep_cbrs_amar_renaissance_b200.utilities.metrics import top_k_predictions
    users = np.array([100, 200, 300])
    items = np.array([7, 8, 9, 10])
    preds = np.array([[1, 3, 0.2], [0, 4, 0.9], [1, 5, 0.8], [1, 6, 0.8], [0, 3, 0.1], [2, 6, 0.5]])
    df = top_k_predictions(preds, users, items, k=2)
    assert df['users'].tolist() == [100, 100, 200, 200, 300]
    assert df['items'].tolist() == [8, 7, 9, 10, 10]
    assert df['scores'].tolist() == [0.9, 0.1, 0.8, 0.8, 0.5]


@pytest.mark.parametrize("n_users,n_items,c1,c2,k", [(1, 1, 4, 1, 1), (37, 3706, 64, 64, 10), (50, 1000, 48, 48, 5),
                                                      (16, 333, 64, 128, 128), (70, 2049, 128, 96, 10),
                                                      (5, 7, 64, 64, 10), (33, 40000, 64, 64, 10),
                                                      (45, 1500, 32, 64, 10), (21, 777, 64, 48, 7), (18, 600, 32, 24, 5)])
@pytest.mark.parametrize("precision", ["fp32", "fp32-ffma"])
def test_fused_catalog_scorer_matches_oracle(dev, n_users, n_items, c1, c2, k, precision):
    """'fp32' takes the 3xTF32 tensor-core kernel for c1 in {32, 64}, c2 <= 64 (fp32-accurate: same oracle, same
    tolerance, same tie rule) and the FFMA kernel otherwise; 'fp32-ffma' forces the FFMA kernel on every shape."""
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    if precision == "fp32":
        launches = ops.LAUNCHES
        tensor = bool(_lib.load().cbrs_score_catalog_topk_tf32x3_eligible(c1, c2))
        assert tensor == (c1 in (32, 64) and c2 <= 64)
    from tests.helpers import assert_topk_equivalent, basic_chain
    rng = np.random.RandomState(n_items + c2)
    P = rng.standard_normal((n_users, c1)).astype(np.float32)
    Q = rng.standard_normal((n_items, c1)).astype(np.float32)
    if n_items > 100:
        Q[50:60] = Q[40:50]  # exact duplicates: exact score ties, lower index must win
    w2, b2 = glorot(rng, (c1, c2)), rng.standard_normal(c2).astype(np.float32) * 0.1
    w3, b3 = glorot(rng, (c2, 1)).reshape(-1), np.array([0.05], np.float32)
    ids, vals = ops.score_catalog_topk(_t(P, dev), _t(Q, dev), _t(w2, dev), _t(b2, dev), _t(w3, dev), _t(b3, dev), k,
                                       precision=precision)
    if precision == "fp32":
        assert ops.LAUNCHES - launches == (2 if tensor else 1)   # operand-image prep + scorer | the FFMA scorer
    scores = basic_chain(P, Q, w2, b2, w3, b3)
    kk = min(k, n_items)
    ids_np, vals_np = ids.cpu().numpy(), vals.cpu().numpy()
    assert (ids_np[:, kk:] == -1).all()
    assert_topk_equivalent(ids_np[:, :kk], vals_np[:, :kk], scores, kk)
    if n_items > 100:  # among exactly tied duplicates the lower index comes first
        for u in range(n_users):
            pos = {int(i): r for r, i in enumerate(ids_np[u, :kk])}
            for a in range(40, 50):
                if a in pos and a + 10 in pos:
                    assert pos[a] < pos[a + 10]
                assert not (a + 10 in pos and a not in pos)


@pytest.mark.parametrize("n_users,n_items,c1,c2,k", [(37, 3706, 64, 64, 10), (50, 1000, 48, 48, 5), (5, 7, 64, 64, 10),
                                                      (40, 333, 128, 128, 20), (130, 2049, 64, 32, 10),
                                                      (33, 500, 8, 16, 3), (20, 700, 72, 80, 10),
                                                      (41, 1500, 64, 128, 10), (9, 300, 32, 96, 7)])
def test_tensor_core_catalog_scorer_matches_bf16_oracle(dev, n_users, n_items, c1, c2, k):
    """tcgen05 path: operands rounded to bf16, fp32 accumulate.  Oracle = the same rounding in numpy;
    tolerance 2e-5 on scores (fp32 summation order inside the MMA is unspecified; 1e-4 for the v3 kernel, where an
    activation within an fp32 ulp of a bf16 rounding boundary may round the other way before the output product)."""
    from deep_cbrs_amar_renaissance_b200 import ops
    from tests.helpers import assert_topk_equivalent, bf16_basic_chain
    rng = np.random.RandomState(n_items + c2)
    P = rng.standard_normal((n_users, c1)).astype(np.float32)
    Q = rng.standard_normal((n_items, c1)).astype(np.float32)
    w2, b2 = glorot(rng, (c1, c2)), rng.standard_normal(c2).astype(np.float32) * 0.1
    w3, b3 = glorot(rng, (c2, 1)).reshape(-1), np.array([0.05], np.float32)
    ids, vals = ops.score_catalog_topk(_t(P, dev), _t(Q, dev), _t(w2, dev), _t(b2, dev), _t(w3, dev), _t(b3, dev), k,
                                       precision="bf16")
    scores = bf16_basic_chain(P, Q, w2, b2, w3, b3)
    kk = min(k, n_items)
    ids_np, vals_np = ids.cpu().numpy(), vals.cpu().numpy()
    assert (ids_np[:, kk:] == -1).all()
    assert_topk_equivalent(ids_np[:, :kk], vals_np[:, :kk], scores, kk, tol=1e-4 if (c1 <= 64 and c2 <= 64) else 2e-5)
    # and it stays within bf16 distance of the exact fp32 scorer
    exact = ol.sigmoid(np.maximum(np.maximum(P[:, None, :] + Q[None, :, :], 0).reshape(-1, c1) @ w2 + b2, 0) @ w3 + b3)
    got_exact = np.take_along_axis(exact.reshape(n_users, n_items), ids_np[:, :kk].astype(np.int64), axis=1)
    assert np.abs(got_exact - vals_np[:, :kk]).max() < 3e-2


# ------------------------------------------------------------------ synthetic generator
def _splitmix(x):
    x = (x + np.uint64(0x9E3779B97F4A7C15))
    x = (x ^ (x >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)
    x = (x ^ (x >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)
    return x ^ (x >> np.uint64(31))


def test_synthetic_generator_is_the_documented_hash(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    import math
    n_users, n_items, n_edges, seed = 5000, 3000, 20000, 42
    row, col = ops.synth_bipartite(n_users, n_items, n_edges, seed, dev)
    with np.errstate(over="ignore"):
        e = np.arange(n_edges, dtype=np.uint64)
        h0 = _splitmix(np.uint64(seed) ^ (e * np.uint64(0x2545F4914F6CDD1D)))
        h1 = _splitmix(h0)
        h2 = _splitmix(h1)
    c = max(n_items // 1024, 1)
    levels = 1
    while c * ((1 << levels) - 1) < n_items:
        levels += 1
    mult = 0x9E3779B1 % n_items or 1
    while math.gcd(mult, n_items) != 1:
        mult += 1
    u = (h0 % np.uint64(n_users)).astype(np.int64)
    lvl = (h1 % np.uint64(levels)).astype(np.int64)
    span = (c << lvl).astype(np.uint64)
    rank = ((span - np.uint64(c) + (h2 % span)) % np.uint64(n_items)).astype(np.int64)
    it = (rank * mult) % n_items
    assert np.array_equal(row.cpu().numpy()[:n_edges], u.astype(np.int32))
    assert np.array_equal(col.cpu().numpy()[:n_edges], (n_users + it).astype(np.int32))
    assert torch.equal(row[n_edges:], col[:n_edges]) and torch.equal(col[n_edges:], row[:n_edges])


# ------------------------------------------------------------------ id compaction (rows G0 / (f)-2)
@pytest.mark.parametrize("n,span", [(1, 5), (1000, 50), (200_000, 6040), (300_000, 2 ** 40)])
def test_compact_ids_equals_numpy_unique(n, span):
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(n % 97)
    raw = rng.randint(-span, span, size=n).astype(np.int64) * 3 + 7  # negative and non-contiguous ids
    uniq, inv = ops.compact_ids(torch.from_numpy(raw).cuda())
    want_u, want_inv = np.unique(raw, return_inverse=True)
    assert np.array_equal(uniq.cpu().numpy(), want_u)
    assert np.array_equal(inv.cpu().numpy(), want_inv)


def test_lookup_ids_equals_broadcast_argwhere():
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(3)
    vocab = np.unique(rng.randint(0, 10 ** 6, size=5000).astype(np.int64))
    ids = np.concatenate([vocab[rng.randint(0, len(vocab), size=3000)], np.array([-5, 10 ** 7], np.int64)])
    got = ops.lookup_ids(torch.from_numpy(vocab).cuda(), torch.from_numpy(ids).cuda()).cpu().numpy()
    want = np.argwhere(ids[:3000, None] == vocab)[:, 1]  # the reference's formulation (loaders.py:53-54)
    assert np.array_equal(got[:3000], want)
    assert (got[3000:] == -1).all()


def test_loader_device_ids_give_the_same_arrays(tmp_path):
    from deep_cbrs_amar_renaissance_b200.data import loaders
    rng = np.random.RandomState(5)
    n = 5000
    tr = np.stack([rng.randint(0, 300, n) * 11 + 1000, rng.randint(0, 200, n) * 7 + 50000, rng.randint(0, 2, n)], 1)
    te = tr[rng.randint(0, n, 800)]
    pr = np.stack([tr[rng.randint(0, n, 600), 1], rng.randint(0, 90, 600) + 90000, rng.randint(0, 5, 600)], 1)
    for name, arr in (("train", tr), ("test", te), ("props", pr)):
        np.savetxt(tmp_path / (name + ".tsv"), arr, fmt="%d", delimiter="\t")
    args = (str(tmp_path / "train.tsv"), str(tmp_path / "test.tsv"), str(tmp_path / "props.tsv"))
    host = loaders.load_train_test_ratings(*args, return_adjacency=True, type_adjacency='unary-uip', device_ids=False)
    dev = loaders.load_train_test_ratings(*args, return_adjacency=True, type_adjacency='unary-uip', device_ids=True)
    for a, b in zip(host[0] + host[1], dev[0] + dev[1]):
        assert a.dtype == b.dtype and np.array_equal(a, b)
    assert (host[2] != dev[2]).nnz == 0 and np.array_equal(host[2].row, dev[2].row)


@pytest.mark.parametrize("m,f,h,r", [(300, 16, 16, 2), (1000, 64, 64, 3), (77, 10, 6, 2), (513, 128, 128, 2), (200, 32, 8, 5)])
def test_dense_grouped_writes_every_relation_block_in_one_launch(dev, m, f, h, r):
    """cbrs_dense_grouped (row R): X . [W_0 | ... | W_{R-1}] stored straight into the stacked [R*N, H] operand; same
    bits as R separate cbrs_dense calls, rows outside the written blocks untouched, bf16 output = rounded fp32 output"""
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(m + f)
    x = _t(rng.standard_normal((m, f)).astype(np.float32), dev)
    ws = [_t(glorot(rng, (f, h)), dev) for _ in range(r)]
    n_stack = m + 37                                   # the stack is taller than this row block (a rank's slice)
    z = torch.full((r * n_stack, h), -5.0, device=dev)
    ops.dense_grouped(x, ws, z[11:], n_stack)          # block written at row offset 11
    for k, w in enumerate(ws):
        want = ops.dense(x, w)
        assert torch.equal(z[k * n_stack + 11:k * n_stack + 11 + m], want), k
    mask = torch.ones(r * n_stack, dtype=torch.bool, device=dev)
    for k in range(r):
        mask[k * n_stack + 11:k * n_stack + 11 + m] = False
    assert (z[mask] == -5.0).all()
    assert_close(z[11:11 + m].cpu().numpy(), x.cpu().numpy() @ ws[0].cpu().numpy(), what="relation 0 vs numpy")
    zb = torch.zeros(r * n_stack, h, device=dev, dtype=torch.bfloat16)
    ops.dense_grouped(x, ws, zb, n_stack)
    for k, w in enumerate(ws):
        assert torch.equal(zb[k * n_stack:k * n_stack + m], ops.dense(x, w).to(torch.bfloat16)), k
