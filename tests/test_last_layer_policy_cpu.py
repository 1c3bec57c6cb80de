"""CPU: when the per-batch call may compute its last layer at the batch's rows only (graph.last_layer_subset_policy).
Row-partitioned stacks, other reductions and other layer families keep the full product; graphs below the row
threshold (the MovieLens-1M-shaped ones) keep it too, and the test override decides only the size condition."""
import pytest

from deep_cbrs_amar_renaissance_b200 import graph


@pytest.fixture
def restore():
    saved = graph.FORCED_SUBSET
    yield
    graph.FORCED_SUBSET = saved


@pytest.mark.parametrize("forced", [None, True, False])
def test_partitioned_or_other_stacks_never_prune(restore, forced):
    graph.FORCED_SUBSET = forced
    big = 11_000_000
    assert not graph.last_layer_subset_policy(big, True, True, True)       # row partition attached
    assert not graph.last_layer_subset_policy(big, False, False, True)     # sum / mean / w-sum / last reduction
    assert not graph.last_layer_subset_policy(big, False, True, False)     # GraphSage / GAT / RGCN / DGCF last layer


def test_small_graphs_keep_the_full_product(restore):
    graph.FORCED_SUBSET = None
    assert graph.SUBSET_MIN_ROWS > 6040 + 3706 + 17554                    # MovieLens-1M users + items + properties
    assert not graph.last_layer_subset_policy(6040 + 3706, False, True, True)
    assert not graph.last_layer_subset_policy(graph.SUBSET_MIN_ROWS - 1, False, True, True)
    graph.FORCED_SUBSET = False
    assert not graph.last_layer_subset_policy(11_000_000, False, True, True)
