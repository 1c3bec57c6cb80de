"""Host side of the catalog exclusion lists: scoring.ItemLists (built with torch on CPU tensors here, against a numpy
construction), the row selection for a user subset, and metrics.catalog_predictions."""
import numpy as np
import pytest
import torch

from deep_cbrs_amar_renaissance_b200.scoring import ItemLists, _exclusion_rows
from deep_cbrs_amar_renaissance_b200.utilities.metrics import catalog_predictions


def _numpy_lists(ratings, n_users, n_items):
    lists = [[] for _ in range(n_users)]
    for u, i in ratings[:, :2]:
        lists[u].append(i - n_users)
    rowptr = np.zeros(n_users + 1, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    return rowptr, np.array([i for x in lists for i in sorted(x)], np.int64)


def _ratings(n_users, n_items, n, seed):
    rng = np.random.RandomState(seed)
    r = np.stack([rng.randint(0, n_users, n), rng.randint(0, n_items, n) + n_users, rng.randint(0, 2, n)], 1)
    r = np.concatenate([r, r[:7]])              # duplicated pairs stay duplicated
    r[:, 0][r[:, 0] == 3] = 4                   # user 3 has no ratings: an empty row
    return r[rng.permutation(len(r))]           # any input order


@pytest.mark.parametrize("as_tensor", [True, False])
def test_from_ratings_matches_numpy(as_tensor):
    n_users, n_items = 23, 41
    r = _ratings(n_users, n_items, 300, 1)
    assert (r[:, 2] == 0).any()                 # rating-0 rows are seen items too
    lists = ItemLists.from_ratings(torch.from_numpy(r) if as_tensor else r, n_users, n_items, device="cpu")
    rowptr, items = _numpy_lists(r, n_users, n_items)
    assert lists.rowptr.dtype == torch.int64 and lists.items.dtype == torch.int32 and lists.n_items == n_items
    assert np.array_equal(lists.rowptr.numpy(), rowptr) and np.array_equal(lists.items.numpy(), items)
    assert lists.rowptr[3] == lists.rowptr[4] and lists.n_users == n_users


def test_from_ratings_rejects_out_of_range_ids():
    r = _ratings(10, 12, 50, 2)
    for col, bad in ((0, 10), (0, -1), (1, 9), (1, 10 + 12)):
        x = r.copy()
        x[0, col] = bad
        with pytest.raises(ValueError):
            ItemLists.from_ratings(torch.from_numpy(x), 10, 12)


def test_rowptr_of_the_wrong_length_is_rejected():
    items = torch.tensor([1, 2, 3], dtype=torch.int32)
    with pytest.raises(ValueError):
        ItemLists(torch.tensor([0, 1, 2], dtype=torch.int64), items, 5)       # ends at 2, not len(items)
    with pytest.raises(ValueError):
        ItemLists(torch.tensor([0, 1, 2, 3], dtype=torch.int32), items, 5)    # not int64
    lists = ItemLists(torch.tensor([0, 1, 2, 3], dtype=torch.int64), items, 5)
    with pytest.raises(ValueError):                                          # lists for 3 users, catalog of 4
        _exclusion_rows(lists, 4, 5, torch.arange(4), True)


def test_user_subsets_select_their_rows():
    n_users, n_items = 15, 30
    lists = ItemLists.from_ratings(torch.from_numpy(_ratings(n_users, n_items, 200, 3)), n_users, n_items)
    want = [lists.items[lists.rowptr[u]:lists.rowptr[u + 1]].tolist() for u in range(n_users)]
    for sub in ([9, 2, 14, 2, 0], [4, 5, 6, 7], [3]):
        rowptr, items = _exclusion_rows(lists, n_users, n_items, torch.tensor(sub), False)
        got = [items[rowptr[r]:rowptr[r + 1]].tolist() for r in range(len(sub))]
        assert got == [want[u] for u in sub]
    rowptr, _ = _exclusion_rows(lists, n_users, n_items, torch.tensor([4, 5, 6, 7]), False)
    assert rowptr.data_ptr() == lists.rowptr[4:].data_ptr()    # a contiguous range is a view, not a copy
    with pytest.raises(ValueError):
        _exclusion_rows(lists, n_users, n_items, torch.tensor([1, n_users]), False)


def test_catalog_predictions_drops_padding():
    ids = torch.tensor([[2, 0, -1], [-1, -1, -1], [1, 2, 0]], dtype=torch.int32)
    vals = torch.tensor([[0.9, 0.5, -np.inf], [-np.inf] * 3, [0.7, 0.6, 0.1]])
    df = catalog_predictions(ids, vals, np.array([10, 20, 30]), np.array([7, 8, 9]))
    assert df["users"].tolist() == [10, 10, 30, 30, 30] and df["items"].tolist() == [9, 7, 8, 9, 7]
    assert np.allclose(df["scores"].to_numpy(), [0.9, 0.5, 0.7, 0.6, 0.1])
