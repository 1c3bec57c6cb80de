"""CPU: the host side of the partitioned graph build (graph.build_row_blocks, graph.PartitionedGraph): what it refuses
before touching a device, and the cuts it derives from the row histogram."""
import numpy as np
import pytest
import torch
from scipy import sparse

from deep_cbrs_amar_renaissance_b200 import graph as G
from deep_cbrs_amar_renaissance_b200.distributed import balanced_ranges, edge_cost_prefix


def test_whole_graph_access_names_the_partitioned_build():
    g = G.PartitionedGraph(70, ("norm",))
    assert g.shape == (70, 70) and g.n_nodes == 70 and g.n_rel == 1
    assert isinstance(g, G.DeviceGraph)        # the model constructors pass it through as they pass a DeviceGraph
    for call in (lambda: g.norm, lambda: g.raw, lambda: g.plain, lambda: g.dgcf, lambda: g.symmetric,
                 lambda: g.transposed(), lambda: g.row_subset(torch.arange(3))):
        with pytest.raises(NotImplementedError, match="partitioned graph build"):
            call()
    g.release_coo()                            # RowPartition.release_full_views stays harmless
    with pytest.raises(NotImplementedError, match="RGCN on a partitioned graph build"):
        G.refuse_partitioned([None, g], "RGCN")
    G.refuse_partitioned([None, sparse.eye(3)], "RGCN")


def test_bad_blocks_and_views_are_refused_before_any_device_work():
    adj = sparse.coo_matrix((np.ones(4, np.float32), ([0, 1, 2, 3], [1, 2, 3, 0])), shape=(5, 5))
    for blocks in ([(2, 2)], [(3, 1)], [(0, 6)], [(-1, 2)]):
        with pytest.raises(ValueError, match="row blocks"):
            G.build_row_blocks(adj, blocks, None)
    with pytest.raises(ValueError, match="views"):
        G.build_row_blocks(adj, [(0, 5)], None, views=("norm", "dgcf"))


def test_cuts_from_the_histogram_are_rank_independent_and_cover_every_row():
    rng = np.random.RandomState(2)
    sizes = [700, 300]
    hist = torch.from_numpy(rng.zipf(1.6, size=sum(sizes)).clip(0, 5000).astype(np.int64))
    est = G.estimated_rowptr(hist)
    assert est.shape == (1001,) and int(est[0]) == 0
    assert torch.equal(est[1:] - est[:-1], hist + 1)
    assert torch.equal(G.estimated_rowptr(hist, self_loops=False)[1:] - G.estimated_rowptr(hist, False)[:-1], hist)
    for world in (1, 2, 3, 8):
        ranges = balanced_ranges(sizes, world, edge_cost_prefix(est, sizes, 25))
        assert ranges == balanced_ranges(sizes, world, edge_cost_prefix(est.clone(), sizes, 25))
        for t, (lo, hi) in enumerate(((0, 700), (700, 1000))):
            blocks = [ranges[r][t] for r in range(world)]
            assert blocks[0][0] == lo and blocks[-1][1] == hi
            assert all(a[1] == b[0] for a, b in zip(blocks[:-1], blocks[1:]))
