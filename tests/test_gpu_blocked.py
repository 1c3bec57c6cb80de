"""GPU parity for the column-blocked work decomposition (cbrs_chunks_blocked_*, round 2).

The schedule only re-orders and re-cuts the work of the sparse kernels, so every consumer (weighted SpMM, sum / mean
aggregators, bf16 operands, the fused GCN kernel, GAT) is checked against the same CPU oracle as the row-major
schedule, at 1e-5 of the tensor scale, with windows small enough that every heavy row crosses many of them; the
decomposition itself (integer work) is checked exactly against a numpy restatement of its definition; and a row
partition must give the same bits as the full run (SURVEY 8e)."""
import numpy as np
import pytest
import torch

from oracle import graph as og
from oracle import layers as ol
from tests.helpers import assert_close, random_bipartite

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


def _t(a, dev, dtype=None):
    t = torch.from_numpy(np.ascontiguousarray(a))
    return t.to(dev) if dtype is None else t.to(dev, dtype)


def _expected_chunks(rowptr, colidx, chunk_edges, n_cols, block_cols, min_len):
    """numpy restatement of the definition in include/cbrs_b200.h: (row, begin, len, slot) in list order."""
    n_rows = len(rowptr) - 1
    plain, blocked, heavy, slot_ptr = [], [], [], [0]
    n_blocks = -(-n_cols // block_cols)
    slot = 0
    for i in range(n_rows):
        b, e = int(rowptr[i]), int(rowptr[i + 1])
        if e - b >= min_len:
            heavy.append(i)
            for cb in range(n_blocks):
                lo = b + int(np.searchsorted(colidx[b:e], cb * block_cols, "left"))
                hi = e if cb + 1 == n_blocks else b + int(np.searchsorted(colidx[b:e], (cb + 1) * block_cols, "left"))
                for s in range(lo, hi, chunk_edges):
                    blocked.append((cb, i, s, min(chunk_edges, hi - s), slot))
                    slot += 1
            slot_ptr.append(slot)
        else:
            nc = 1 if e - b <= chunk_edges else -(-(e - b) // chunk_edges)
            for k in range(nc):
                s = b + k * chunk_edges
                plain.append((i, s, min(chunk_edges, e - s), slot + k if nc > 1 else -1))
            if nc > 1:
                heavy.append(i)
                slot += nc
                slot_ptr.append(slot)
    blocked.sort(key=lambda t: (t[0], t[1], t[2]))
    return plain + [t[1:] for t in blocked], heavy, slot_ptr


@pytest.mark.parametrize("chunk_edges,block_cols,min_len", [(8, 16, 6), (1024, 32, 10), (4, 7, 1), (16, 1000, 5)])
def test_blocked_decomposition_matches_its_definition(dev, chunk_edges, block_cols, min_len):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj = random_bipartite(90, 35, 1800, seed=chunk_edges, n_props=10, n_links=60, dup_links=8)
    rowptr, colidx, _ = og.reorder_raw(adj)
    n_cols = adj.shape[1]
    c = ops.build_chunks(_t(rowptr, dev, torch.int64), chunk_edges, _t(colidx, dev, torch.int32), n_cols, block_cols, min_len)
    want, heavy, slot_ptr = _expected_chunks(rowptr, colidx, chunk_edges, n_cols, block_cols, min_len)
    got = list(zip(c["chunk_row"].cpu().tolist(), c["chunk_begin"].cpu().tolist(), c["chunk_len"].cpu().tolist(),
                   c["chunk_slot"].cpu().tolist()))
    assert c["n_chunks"] == len(want) and got == want
    assert c["heavy_row"].cpu().tolist() == heavy and c["heavy_slot_ptr"].cpu().tolist() == slot_ptr
    assert c["n_heavy"] == len(heavy) and c["n_slots"] == slot_ptr[-1]
    # every edge is covered exactly once
    cover = np.zeros(len(colidx), np.int32)
    for _, s, n, _ in got:
        cover[s:s + n] += 1
    assert (cover == 1).all()


def test_blocked_decomposition_handles_empty_rows_and_no_blocked_rows(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    lens = np.array([0, 5, 0, 9, 0], np.int64)
    rowptr = np.concatenate([[0], np.cumsum(lens)])
    colidx = np.concatenate([np.sort(np.random.RandomState(0).choice(50, n, replace=False)) for n in lens]).astype(np.int32)
    for min_len in (100, 9, 1):
        c = ops.build_chunks(_t(rowptr, dev), 4, _t(colidx, dev), 50, 10, min_len)
        want, heavy, slot_ptr = _expected_chunks(rowptr, colidx, 4, 50, 10, min_len)
        got = list(zip(c["chunk_row"].cpu().tolist(), c["chunk_begin"].cpu().tolist(), c["chunk_len"].cpu().tolist(),
                       c["chunk_slot"].cpu().tolist()))
        assert got == want and c["heavy_row"].cpu().tolist() == heavy and c["heavy_slot_ptr"].cpu().tolist() == slot_ptr


def _graphs(adj, dev, blocking, chunk_edges=16):
    from deep_cbrs_amar_renaissance_b200.graph import CsrSlice, DeviceGraph
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=chunk_edges)

    def reblock(v):
        return CsrSlice(v.rowptr, v.colidx, v.vals, v.n_cols, chunk_edges, blocking=blocking)
    return g, reblock


@pytest.mark.parametrize("d", [16, 128, 100, 6])
@pytest.mark.parametrize("blocking", [(16, 8), (50, 1), (7, 30)])
def test_spmm_blocked_matches_oracle(dev, d, blocking):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj = random_bipartite(120, 40, 2500, seed=d, n_props=20, n_links=100, dup_links=10)
    g, reblock = _graphs(adj, dev, blocking)
    norm = reblock(g.norm)
    assert norm.chunks["chunk_len"] is not None and norm.chunks["n_heavy"] > 0
    rng = np.random.RandomState(d)
    x = rng.standard_normal((adj.shape[0], d)).astype(np.float32)
    b = rng.standard_normal(d).astype(np.float32)
    a_hat = og.gcn_filter(adj)
    out = torch.empty(adj.shape[0], d, device=dev)
    ops.spmm(norm, _t(x, dev), out, bias=_t(b, dev), relu=True)
    assert_close(out.cpu().numpy(), np.maximum(a_hat @ x + b, 0), what="blocked relu(A_hat x + b)")
    # the schedule changes the reduction tree of blocked rows only: rows below min_len keep their bits
    ref = torch.empty_like(out)
    ops.spmm(g.norm, _t(x, dev), ref, bias=_t(b, dev), relu=True)
    lens = (g.norm.rowptr[1:] - g.norm.rowptr[:-1]).cpu().numpy()
    light = lens < blocking[1]
    assert torch.equal(out[torch.from_numpy(light).to(dev)], ref[torch.from_numpy(light).to(dev)])
    raw = reblock(g.raw)
    ptr, idx, _ = og.reorder_raw(adj)
    for agg, name in ((1, "sum"), (2, "mean")):
        ops.spmm(raw, _t(x, dev), out, agg=agg)
        assert_close(out.cpu().numpy(), ol.sage_aggregate(x, ptr, idx, name), what="blocked " + name)


def test_spmm_blocked_bf16_equals_fp32_kernel_on_widened_values(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj = random_bipartite(150, 40, 3000, seed=4)
    g, reblock = _graphs(adj, dev, (24, 12))
    norm = reblock(g.norm)
    x = torch.randn(adj.shape[0], 128, device=dev, generator=torch.Generator(dev).manual_seed(1))
    xb = x.to(torch.bfloat16)
    a, b = torch.empty_like(x), torch.empty_like(x)
    ops.spmm(norm, xb, a)
    ops.spmm(norm, xb.float(), b)
    assert torch.equal(a, b)


def test_blocked_row_partition_is_bit_identical(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    adj = random_bipartite(200, 50, 5000, seed=9)
    g, reblock = _graphs(adj, dev, (32, 20), chunk_edges=32)
    norm, raw = reblock(g.norm), reblock(g.raw)
    x = _t(np.random.RandomState(3).standard_normal((250, 64)).astype(np.float32), dev)
    full, full_mean = torch.empty(250, 64, device=dev), torch.empty(250, 64, device=dev)
    ops.spmm(norm, x, full, relu=True)
    ops.spmm(raw, x, full_mean, agg=2)
    for cuts in ([0, 250], [0, 100, 250], [0, 7, 130, 131, 250], [0, 210, 250]):
        part, part_mean = torch.empty(250, 64, device=dev), torch.empty(250, 64, device=dev)
        for r0, r1 in zip(cuts[:-1], cuts[1:]):
            s = norm.row_slice(r0, r1)
            assert s.blocking == (32, 20) and s.chunks["chunk_len"] is not None
            ops.spmm(s, x, part[r0:r1], relu=True)
            ops.spmm(raw.row_slice(r0, r1), x, part_mean[r0:r1], agg=2)
        assert torch.equal(part, full) and torch.equal(part_mean, full_mean)


def test_gat_blocked_matches_oracle_and_partition(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph, CsrSlice
    adj = random_bipartite(100, 40, 2200, seed=11, n_props=15, n_links=80, dup_links=12)
    n, h = adj.shape[0], 32
    g = DeviceGraph.from_scipy(adj, dev, chunk_edges=16)
    v = g.raw
    blk = CsrSlice(v.rowptr, v.colidx, None, v.n_cols, 16, blocking=(20, 10))
    rng = np.random.RandomState(5)
    z = rng.standard_normal((n, h)).astype(np.float32)
    p = rng.standard_normal(n).astype(np.float32)
    q = rng.standard_normal(n).astype(np.float32)
    bias = rng.standard_normal(h).astype(np.float32)
    ref = torch.empty(n, h, device=dev)
    out = torch.empty(n, h, device=dev)
    ops.gat(v, _t(z, dev), _t(p, dev), _t(q, dev), ref, bias=_t(bias, dev), relu=True)
    ops.gat(blk, _t(z, dev), _t(p, dev), _t(q, dev), out, bias=_t(bias, dev), relu=True)
    assert_close(out.cpu().numpy(), ref.cpu().numpy(), what="blocked GAT vs row-major GAT (oracle-checked elsewhere)")
    part = torch.empty_like(out)
    for r0, r1 in ((0, 33), (33, 101), (101, n)):
        ops.gat(blk.row_slice(r0, r1), _t(z, dev), _t(p, dev), _t(q, dev), part[r0:r1], bias=_t(bias, dev), relu=True,
                row_offset=r0)
    assert torch.equal(part, out)


def test_default_policy_leaves_small_graphs_row_major(dev):
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph, blocking_policy
    assert blocking_policy(9746) == (0, 0) and blocking_policy(11_000_000)[0] > 0
    g = DeviceGraph.from_scipy(random_bipartite(40, 25, 400, seed=5), dev)
    assert g.norm.blocking == (0, 0) and g.norm.chunks["chunk_len"] is None


def test_unscattered_generator_equals_its_numpy_twin_and_concentrates_hot_items(dev):
    """scatter_items=0 (bench.py --unscattered): item id = popularity rank; same hash as the scattered generator"""
    from deep_cbrs_amar_renaissance_b200 import ops
    from oracle import synth as osynth
    n_users, n_items, n_edges = 5000, 3000, 40000
    for scatter in (True, False):
        row, col = ops.synth_bipartite(n_users, n_items, n_edges, 42, dev, scatter_items=scatter)
        r, c = osynth.synth_bipartite(n_users, n_items, n_edges, 42, scatter_items=scatter)
        assert np.array_equal(row.cpu().numpy(), r) and np.array_equal(col.cpu().numpy(), c)
    deg = np.bincount(c[:n_edges] - n_users, minlength=n_items)
    assert deg[:n_items // 8].sum() > 0.25 * n_edges  # the first eighth of the ids holds far more than an eighth


def test_transposed_view_and_symmetry_flag(dev):
    from deep_cbrs_amar_renaissance_b200.graph import DeviceGraph
    from scipy import sparse
    adj = random_bipartite(60, 30, 700, seed=1, n_props=10, n_links=50, dup_links=10)
    g = DeviceGraph.from_scipy(adj, dev)
    assert g.symmetric
    half = sparse.coo_matrix((adj.data[:len(adj.data) // 2], (adj.row[:len(adj.data) // 2], adj.col[:len(adj.data) // 2])),
                             shape=adj.shape)
    gd = DeviceGraph.from_scipy(half, dev)
    assert not gd.symmetric
    t = gd.plain.transposed()
    want = half.tocsr().T.tocsr()
    want.sort_indices()
    got = t.to_scipy()
    assert np.array_equal(got.indptr, want.indptr) and np.array_equal(got.indices, want.indices)
    assert np.array_equal(got.data, want.data)
