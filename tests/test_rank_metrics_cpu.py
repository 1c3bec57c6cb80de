"""Host side of the full-catalog ranking metrics: a plain-numpy restatement of the definitions above cbrs_rank_metrics
(include/cbrs_b200.h), checked on a hand-worked case and against precision_recall_f1_at_k; the relevance lists built by
ItemLists.from_ratings(min_rating=1, distinct=True); the refusal of bad cutoffs before any device work.
tests/test_gpu_rank_metrics.py checks the kernel against the same restatement."""
import numpy as np
import pytest
import torch

from deep_cbrs_amar_renaissance_b200 import _lib as L
from deep_cbrs_amar_renaissance_b200 import ops
from deep_cbrs_amar_renaissance_b200.scoring import ItemLists
from deep_cbrs_amar_renaissance_b200.utilities import metrics as M

COLS = ("precision", "recall", "hit_rate", "mrr", "ndcg", "map")   # ops.RANK_METRICS


def restate(ids, rowptr, items, users, cutoffs, n_items):
    """(per_user [n_rows, n_cutoffs, 6] with NaN rows for users without relevant items, sums [n_cutoffs, 7]) of the lists
    ids [n_rows, k] against the CSR relevance lists (rows = global user ids, sorted distinct catalog indices)."""
    ids = np.asarray(ids, np.int64)
    n_rows, k = ids.shape
    n_users = len(rowptr) - 1
    users = np.arange(n_rows) if users is None else np.asarray(users, np.int64)
    ok_user = (users >= 0) & (users < n_users)
    uu = np.where(ok_user, users, 0)
    n_rel = np.where(ok_user, rowptr[uu + 1] - rowptr[uu], 0)
    # hit_r: the slot's id is a catalog index in the user's list (one search over the global (user, item) keys)
    keys = np.repeat(np.arange(n_users, dtype=np.int64), np.diff(rowptr)) * n_items + np.asarray(items, np.int64)
    q = uu[:, None] * n_items + ids
    hit = np.zeros((n_rows, k))
    if len(keys):
        found = keys[np.minimum(np.searchsorted(keys, q), len(keys) - 1)] == q
        hit[(ids >= 0) & (ids < n_items) & ok_user[:, None] & found] = 1.0
    r = np.arange(k)
    disc = 1.0 / np.log2(r + 2.0)
    cum = np.cumsum(hit, axis=1)
    any_rel = n_rel > 0
    per_user = np.full((n_rows, len(cutoffs), 6), np.nan)
    sums = np.zeros((len(cutoffs), 7))
    for ci, c in enumerate(cutoffs):
        h = hit[:, :c]
        tp = h.sum(1)
        first = np.where(tp > 0, np.argmax(h > 0, axis=1), c)
        ideal = np.minimum(c, n_rel)
        idcg = np.array([disc[:m].sum() for m in ideal])
        vals = np.stack([
            tp / c,
            tp / np.maximum(n_rel, 1),
            (tp > 0).astype(np.float64),
            np.where(tp > 0, 1.0 / (first + 1.0), 0.0),
            (h * disc[:c]).sum(1) / np.where(ideal > 0, idcg, 1.0),
            (h * cum[:, :c] / (r[:c] + 1.0)).sum(1) / np.maximum(ideal, 1),
        ], 1)
        per_user[any_rel, ci] = vals[any_rel]
        sums[ci, :6] = vals[any_rel].sum(0)
        sums[ci, 6] = any_rel.sum()
    return per_user, sums


def _csr(lists):
    rowptr = np.zeros(len(lists) + 1, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.asarray(x, np.int64) for x in lists] + [np.zeros(0, np.int64)])
    return rowptr, items


def test_restatement_hand_case():
    a, b, c, x, y = 3, 7, 11, 1, 9
    rowptr, items = _csr([sorted([a, b, c])])
    per_user, sums = restate([[a, x, b, y, -1]], rowptr, items, None, [1, 2, 5], n_items=20)
    p5, r5, hr5, mrr5, ndcg5, ap5 = per_user[0, 2]
    assert p5 == pytest.approx(0.4, abs=1e-15) and r5 == pytest.approx(2 / 3, abs=1e-15)
    assert hr5 == 1.0 and mrr5 == 1.0
    assert ndcg5 == pytest.approx(1.5 / (1 + 1 / np.log2(3) + 0.5), abs=1e-15)
    assert ndcg5 == pytest.approx(0.7039, abs=1e-4)
    assert ap5 == pytest.approx((1 + 2 / 3) / 3, abs=1e-15)
    # cutoff 1: one slot, a hit; cutoff 2: [a, x]
    assert np.allclose(per_user[0, 0], [1, 1 / 3, 1, 1, 1, 1], rtol=0, atol=1e-15)
    assert np.allclose(per_user[0, 1], [0.5, 1 / 3, 1, 1, 1 / (1 + 1 / np.log2(3)), 0.5], rtol=0, atol=1e-15)
    assert np.array_equal(sums[:, 6], [1, 1, 1])
    # no hit before the cutoff: MRR, HR, NDCG and AP are 0; a user without relevant items is not counted
    rowptr, items = _csr([[a], []])
    per_user, sums = restate([[x, y, a], [a, b, c]], rowptr, items, None, [2, 3], n_items=20)
    assert np.array_equal(per_user[0, 0], [0, 0, 0, 0, 0, 0]) and np.isnan(per_user[1]).all()
    assert np.allclose(per_user[0, 1], [1 / 3, 1, 1, 1 / 3, 0.5, 1 / 3], rtol=0, atol=1e-15)
    assert np.array_equal(sums[:, 6], [1, 1])


def test_restatement_ignores_empty_and_out_of_range_slots():
    rowptr, items = _csr([[0, 4]])
    got, _ = restate([[-1, 4, 5, -7, 0]], rowptr, items, None, [5], n_items=5)
    want, _ = restate([[2, 4, 3, 1, 0]], rowptr, items, None, [5], n_items=5)
    assert np.array_equal(got, want)
    got, _ = restate([[4, 9]], rowptr, items, None, [2], n_items=4)     # 4 is outside [0, n_items = 4)
    assert got[0, 0, 0] == 0


@pytest.mark.parametrize("seed", [0, 1, 2])
def test_restatement_precision_recall_f1_match_the_rival_restatement(seed):
    """on random lists for a subset of users, against precision_recall_f1_at_k on the catalog_predictions frame"""
    rng = np.random.RandomState(seed)
    n_users, n_items, k = 57, 90, 10
    users_orig, items_orig = np.arange(300, 300 + n_users) * 3, np.arange(9000, 9000 + n_items)
    test = np.stack([rng.randint(0, n_users, 800), rng.randint(0, n_items, 800), rng.randint(0, 3, 800)], 1)
    test = np.concatenate([test, test[:50]])                        # duplicated test rows
    rel = [sorted(set(test[(test[:, 0] == u) & (test[:, 2] >= 1), 1].tolist())) for u in range(n_users)]
    rowptr, items = _csr(rel)
    scored = np.sort(rng.choice(n_users, 40, replace=False))          # the others count 0
    ids = np.stack([rng.choice(n_items, k, replace=False) for _ in scored])
    ids[::7, 8:] = -1                                                 # fewer eligible items than k
    vals = np.tile(-np.arange(k, dtype=np.float32), (len(scored), 1))
    frame = M.catalog_predictions(ids, vals, users_orig[scored], items_orig)
    test_orig = np.stack([users_orig[test[:, 0]], items_orig[test[:, 1]], test[:, 2]], 1)
    _, sums = restate(ids, rowptr, items, scored, [5, 10], n_items)
    n_rel = sum(1 for x in rel if x)
    for ci, c in enumerate((5, 10)):
        want = M.precision_recall_f1_at_k(test_orig, frame.to_numpy(), c)
        p, r = sums[ci, 0] / n_rel, sums[ci, 1] / n_rel
        assert want["users"] == n_rel
        assert np.allclose([p, r, 2 * p * r / (p + r)], [want["precision"], want["recall"], want["f1"]], rtol=0, atol=1e-12)


def test_from_ratings_relevance_sets():
    n_users, n_items = 9, 13
    r = np.array([[0, 9 + 4, 1], [0, 9 + 4, 1], [0, 9 + 2, 0], [0, 9 + 1, 2], [2, 9 + 0, 0], [2, 9 + 0, 0],
                  [5, 9 + 12, 1], [5, 9 + 3, 1], [5, 9 + 12, 0], [8, 9 + 7, 1]])
    rel = ItemLists.from_ratings(r, n_users, n_items, device="cpu", min_rating=1, distinct=True)
    lists = [rel.items[rel.rowptr[u]:rel.rowptr[u + 1]].tolist() for u in range(n_users)]
    assert lists == [[1, 4], [], [], [], [], [3, 12], [], [], [7]]
    # the rows precision_recall_f1_at_k treats as relevant, as sets
    want = {}
    for u, i, x in r:
        if x >= 1:
            want.setdefault(u, set()).add(i - n_users)
    assert {u: set(x) for u, x in enumerate(lists) if x} == want
    # defaults unchanged: every row, duplicates kept
    seen = ItemLists.from_ratings(torch.from_numpy(r), n_users, n_items, device="cpu")
    assert seen.items.tolist() == [1, 2, 4, 4, 0, 0, 3, 12, 12, 7]
    # each keyword alone, on a tensor
    t = torch.from_numpy(r)
    assert ItemLists.from_ratings(t, n_users, n_items, min_rating=1).items.tolist() == [1, 4, 4, 3, 12, 7]
    assert ItemLists.from_ratings(t, n_users, n_items, distinct=True).items.tolist() == [1, 2, 4, 0, 3, 12, 7]
    with pytest.raises(ValueError, match="rating column"):
        ItemLists.from_ratings(r[:, :2], n_users, n_items, device="cpu", min_rating=1)


@pytest.mark.parametrize("cutoffs", [[], [0], [11], [5, 5], [10, 5], list(range(1, 10)), [5, "x"]])
def test_bad_cutoffs_are_refused_before_any_device_work(cutoffs, monkeypatch):
    def no_device(*a, **kw):
        raise AssertionError("the library was loaded")
    monkeypatch.setattr(L, "load", no_device)
    ids = torch.zeros(4, 10, dtype=torch.int32)
    rel = ItemLists(torch.zeros(5, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), 20)
    with pytest.raises((L.CbrsError, ValueError)):
        M.catalog_ranking_metrics(ids, rel, cutoffs=cutoffs)
    with pytest.raises((L.CbrsError, ValueError)):
        ops.rank_metrics(ids, (rel.rowptr, rel.items), None, cutoffs)


def test_other_refusals_before_any_device_work(monkeypatch):
    monkeypatch.setattr(L, "load", lambda: (_ for _ in ()).throw(AssertionError("the library was loaded")))
    rel = ItemLists(torch.zeros(5, dtype=torch.int64), torch.zeros(0, dtype=torch.int32), 20)
    with pytest.raises(L.CbrsError, match="k = 129"):
        M.catalog_ranking_metrics(torch.zeros(4, 129, dtype=torch.int32), rel, cutoffs=[5])
    with pytest.raises(L.CbrsError, match="int32"):
        M.catalog_ranking_metrics(torch.zeros(4, 10, dtype=torch.int64), rel)
    with pytest.raises(ValueError, match="unknown ranking metrics"):
        M.catalog_ranking_metrics(torch.zeros(4, 10, dtype=torch.int32), rel, metrics=("ndcg", "auc"))
    with pytest.raises(TypeError):
        M.catalog_ranking_metrics(torch.zeros(4, 10, dtype=torch.int32), (rel.rowptr, rel.items))


def test_workspace_query_needs_no_device():
    lib = L.load()
    assert lib.cbrs_rank_metrics_workspace_bytes(0, 2) == 0
    one = lib.cbrs_rank_metrics_workspace_bytes(1, 2)
    assert one >= 2 * 7 * 8
    big = lib.cbrs_rank_metrics_workspace_bytes(10_000_000, 2)
    assert big >= 2 * 7 * 8 * (10_000_000 // 128) and big < 2 * 7 * 8 * 10_000_000 // 64
