"""cbrs_rank_metrics on the GPU: sums and per-user values against the numpy restatement of tests/test_rank_metrics_cpu.py,
the model path against precision_recall_f1_at_k, determinism, guard bands, the argument refusals and the driver's
`catalog_metrics: all`."""
import ctypes
import os

import numpy as np
import pytest
import torch

from tests.test_rank_metrics_cpu import restate

pytestmark = pytest.mark.gpu
N_ITEMS = 3000


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _relevance(n_users, seed):
    """sorted distinct rows of 0..300 items; every fifth user has none"""
    rng = np.random.RandomState(seed)
    lens = rng.randint(0, 301, n_users)
    lens[::5] = 0
    lens[1::5] = rng.randint(1, 4, len(lens[1::5]))
    rowptr = np.zeros(n_users + 1, np.int64)
    rowptr[1:] = np.cumsum(lens)
    items = np.concatenate([np.sort(rng.choice(N_ITEMS, n, replace=False)) for n in lens] + [np.zeros(0, np.int64)])
    return rowptr, items.astype(np.int32)


def _lists(rowptr, items, users, k, seed):
    """lists mixing the user's relevant items (at random ranks) with other items, -1 tails and out-of-range ids"""
    rng = np.random.RandomState(seed)
    n = len(users)
    ids = rng.randint(0, N_ITEMS, (n, k)).astype(np.int64)
    for r, u in enumerate(users):
        if 0 <= u < len(rowptr) - 1 and rowptr[u + 1] > rowptr[u]:
            own = items[rowptr[u]:rowptr[u + 1]]
            m = min(len(own), rng.randint(0, k + 1))
            ids[r, rng.choice(k, m, replace=False)] = rng.choice(own, m, replace=False)
    if k > 2:
        ids[::3, -2:] = -1                                    # fewer eligible items than k
        ids[1::7, 0] = N_ITEMS + 5                            # out of the catalog
        ids[2::11, 1] = -9
        ids[4::13, k // 2] = 2 ** 31 - 1
    return ids.astype(np.int32)


def _run(dev, ids, rowptr, items, users, cutoffs, per_user=True):
    from deep_cbrs_amar_renaissance_b200 import ops
    u = None if users is None else _t(np.asarray(users, np.int64), dev)
    sums, pu = ops.rank_metrics(ids, (_t(rowptr, dev), _t(items, dev)), u, cutoffs, per_user=per_user, n_items=N_ITEMS)
    torch.cuda.synchronize()
    return sums.cpu().numpy(), None if pu is None else pu.cpu().numpy()


def _check(got_sums, got_pu, want_pu, want_sums):
    assert np.array_equal(np.isnan(got_pu), np.isnan(want_pu))
    assert np.allclose(np.nan_to_num(got_pu), np.nan_to_num(want_pu), rtol=0, atol=1e-12)
    assert np.array_equal(got_sums[:, 6], want_sums[:, 6])
    assert np.allclose(got_sums, want_sums, rtol=1e-12, atol=1e-12)


CASES = [(1, 1, [1]), (1, 10, [5, 10]), (31, 10, [1, 3, 5, 10]), (31, 128, [1, 10, 32, 33, 64, 100, 127, 128]),
         (1000, 10, [5, 10]), (1000, 128, [20, 50, 128]), (1000, 1, [1]), (70000, 10, [5, 10]), (70000, 128, [10, 96])]


@pytest.mark.parametrize("n_rows,k,cutoffs", CASES)
def test_kernel_matches_the_restatement(dev, n_rows, k, cutoffs):
    rowptr, items = _relevance(n_rows, seed=n_rows + k)
    ids = _lists(rowptr, items, np.arange(n_rows), k, seed=k)
    sums, pu = _run(dev, _t(ids, dev), rowptr, items, None, cutoffs)
    want_pu, want_sums = restate(ids, rowptr, items, None, cutoffs, N_ITEMS)
    assert want_sums[:, 4].max() > 0 or n_rows == 1
    _check(sums, pu, want_pu, want_sums)


@pytest.mark.parametrize("k", [10, 128])
def test_user_subsets(dev, k):
    n_users = 5000
    rowptr, items = _relevance(n_users, seed=7)
    rng = np.random.RandomState(k)
    for users in (np.arange(1200, 1200 + 777),                                    # contiguous
                  rng.choice(n_users, 1500, replace=False),                       # scattered, unsorted
                  np.array([n_users + 3, 4, -2, 4999, 0, 2 ** 40])):              # users outside the lists: no relevance
        ids = _lists(rowptr, items, users, k, seed=3)
        sums, pu = _run(dev, _t(ids, dev), rowptr, items, users, [1, 5, k])
        want_pu, want_sums = restate(ids, rowptr, items, users, [1, 5, k], N_ITEMS)
        _check(sums, pu, want_pu, want_sums)


def test_no_rows_and_no_lists(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    rowptr, items = _relevance(50, seed=1)
    sums, pu = _run(dev, torch.zeros(0, 10, dtype=torch.int32, device=dev), rowptr, items, None, [5, 10])
    assert np.array_equal(sums, np.zeros((2, 7))) and pu.shape == (0, 2, 6)
    empty = (torch.zeros(51, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    s, p = ops.rank_metrics(torch.zeros(50, 10, dtype=torch.int32, device=dev), empty, None, [5, 10], per_user=True)
    assert not s.any() and torch.isnan(p).all()


def test_model_lists_match_precision_recall_f1_at_k(dev):
    """the setting of test_catalog_metrics_match_a_numpy_restatement: a BasicGCN's catalog lists, training items
    excluded; device P/R/F1 == the RiVal restatement on the catalog_predictions frame"""
    from deep_cbrs_amar_renaissance_b200.scoring import ItemLists
    from deep_cbrs_amar_renaissance_b200.utilities.metrics import (catalog_predictions, catalog_ranking_metrics,
                                                                   precision_recall_f1_at_k)
    from tests.test_gpu_catalog_exclusion import _basic_model
    n_users, n_items = 80, 120
    model, adj = _basic_model(n_users, n_items, seed=21)
    rng = np.random.RandomState(3)
    coo = adj.tocoo() if hasattr(adj, "tocoo") else adj.coo
    mask = (coo.row < n_users) & (coo.col >= n_users)
    train = np.stack([coo.row[mask], coo.col[mask], rng.randint(0, 2, mask.sum())], 1)
    test = np.stack([rng.randint(0, n_users, 600), rng.randint(0, n_items, 600) + n_users, rng.randint(0, 2, 600)], 1)
    users, items = np.arange(1000, 1000 + n_users), np.arange(5000, 5000 + n_items)
    seen = ItemLists.from_ratings(train, n_users, n_items, device=dev)
    ids, vals = model.recommend_top_k(n_users, n_items, 10, exclude=seen)
    rel = ItemLists.from_ratings(test, n_users, n_items, device=dev, min_rating=1, distinct=True)
    got = catalog_ranking_metrics(ids, rel, cutoffs=(5, 10))
    frame = catalog_predictions(ids, vals, users, items)
    test_orig = np.stack([users[test[:, 0]], items[test[:, 1] - n_users], test[:, 2]], 1)
    for k in (5, 10):
        want = precision_recall_f1_at_k(test_orig, frame.to_numpy(), k)
        assert got["users"] == want["users"]
        for m in ("precision", "recall", "f1"):
            assert abs(got["%s_at_%d" % (m, k)] - want[m]) <= 1e-12, (m, k, got, want)
    # a subset of users: the unscored relevant users count 0
    sub = torch.tensor([5, 77, 0, 31], device=dev)
    got = catalog_ranking_metrics(ids[sub], rel, users=sub, cutoffs=(10,), metrics=("precision",))
    frame = catalog_predictions(ids[sub], vals[sub], users[sub.cpu().numpy()], items)
    want = precision_recall_f1_at_k(test_orig, frame.to_numpy(), 10)
    assert set(got) == {"precision_at_10", "users"} and abs(got["precision_at_10"] - want["precision"]) <= 1e-12


def test_bit_identical_across_calls_and_strides(dev):
    n_rows, k = 70000, 64
    rowptr, items = _relevance(n_rows, seed=5)
    ids = _lists(rowptr, items, np.arange(n_rows), k, seed=5)
    a = _run(dev, _t(ids, dev), rowptr, items, None, [5, 10, 64])
    b = _run(dev, _t(ids, dev), rowptr, items, None, [5, 10, 64])
    wide = torch.full((n_rows, k + 37), 7, dtype=torch.int32, device=dev)
    wide[:, 13:13 + k] = _t(ids, dev)
    c = _run(dev, wide[:, 13:13 + k], rowptr, items, None, [5, 10, 64])
    for other in (b, c):
        assert np.array_equal(a[0].view(np.int64), other[0].view(np.int64))
        assert np.array_equal(a[1].view(np.int64), other[1].view(np.int64))


SENT = -7.25e30
GUARD = 2048


class _Arena:
    """one sentinel-filled float32 buffer; every output, workspace and input is carved from it with guard words around"""

    def __init__(self, dev, floats):
        self.buf = torch.full((floats,), SENT, device=dev, dtype=torch.float32)
        self.used = torch.zeros(floats, dtype=torch.bool, device=dev)
        self.off = GUARD

    def take(self, n, dtype):
        words = max(1, -(-n * torch.empty(0, dtype=dtype).element_size() // 4))
        self.off = (self.off + 7) // 8 * 8
        view = self.buf[self.off:self.off + words]
        self.used[self.off:self.off + words] = True
        self.off += words + GUARD
        assert self.off + GUARD <= self.buf.numel()
        return view.view(dtype)[:n]

    def check(self, what):
        sent = torch.tensor([SENT], dtype=torch.float32).view(torch.int32).item()
        bad = (~self.used) & (self.buf.view(torch.int32) != sent)
        assert not bool(bad.any()), "%s wrote outside its buffers: %d stray words" % (what, int(bad.sum()))


@pytest.mark.parametrize("n_rows,k,cutoffs", [(37, 11, [3, 11]), (129, 128, [1, 7, 33, 128]), (1001, 5, [1, 2, 3, 4, 5])])
def test_outputs_and_workspace_stay_inside_their_buffers(dev, n_rows, k, cutoffs):
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    rowptr, items = _relevance(n_rows + 3, seed=k)
    ids_np = _lists(rowptr, items, np.arange(n_rows) + 3, k, seed=k)
    nc = len(cutoffs)
    ws_bytes = lib.cbrs_rank_metrics_workspace_bytes(n_rows, nc)
    a = _Arena(dev, 16 * GUARD + 4 * (rowptr.size + items.size + ids_np.size + n_rows * 2 + nc * 14 + n_rows * nc * 12)
               + ws_bytes)
    rp, it, ids, users = a.take(rowptr.size, torch.int64), a.take(items.size, torch.int32), a.take(ids_np.size, torch.int32), \
        a.take(n_rows, torch.int64)
    rp.copy_(_t(rowptr, dev)); it.copy_(_t(items, dev)); ids.copy_(_t(ids_np.reshape(-1), dev))
    users.copy_(torch.arange(3, n_rows + 3, device=dev))
    sums, pu, ws = a.take(nc * 7, torch.float64), a.take(n_rows * nc * 6, torch.float64), a.take(ws_bytes, torch.uint8)
    rc = lib.cbrs_rank_metrics(vp(ids), k, n_rows, k, N_ITEMS, vp(users), n_rows + 3, vp(rp), vp(it),
                               (ctypes.c_int32 * nc)(*cutoffs), nc, vp(sums), vp(pu), vp(ws), ws_bytes, ops._stream())
    _lib.check(rc, "cbrs_rank_metrics")
    torch.cuda.synchronize()
    a.check("cbrs_rank_metrics")
    want_pu, want_sums = restate(ids_np, rowptr, items, np.arange(n_rows) + 3, cutoffs, N_ITEMS)
    _check(sums.view(nc, 7).cpu().numpy(), pu.view(n_rows, nc, 6).cpu().numpy(), want_pu, want_sums)


def test_invalid_arguments_are_refused_before_any_launch(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    ids = torch.zeros(4, 130, dtype=torch.int32, device=dev)
    rp = torch.zeros(5, dtype=torch.int64, device=dev)
    it = torch.zeros(1, dtype=torch.int32, device=dev)
    sums = torch.full((9, 7), 3.5, dtype=torch.float64, device=dev)
    ws = torch.empty(1 << 16, dtype=torch.uint8, device=dev)

    def call(k=10, cutoffs=(5, 10), rpp=vp(rp), itp=vp(it), ws_bytes=ws.numel()):
        c = (ctypes.c_int32 * max(1, len(cutoffs)))(*cutoffs)
        return lib.cbrs_rank_metrics(vp(ids), 130, 4, k, 100, None, 4, rpp, itp, c, len(cutoffs), vp(sums), None, vp(ws),
                                     ws_bytes, ops._stream())

    invalid = [dict(cutoffs=(10, 5)), dict(cutoffs=(5, 5)), dict(cutoffs=(0, 5)), dict(cutoffs=(5, 11)), dict(cutoffs=()),
               dict(k=129, cutoffs=(5,)), dict(k=0, cutoffs=(5,)), dict(cutoffs=tuple(range(1, 10))),
               dict(rpp=None), dict(itp=None)]
    for kw in invalid:
        assert call(**kw) == -1, kw           # CBRS_E_INVALID
    assert b"rel_items is null" in (call(itp=None) and lib.cbrs_last_error())
    assert call(ws_bytes=8) == -2             # CBRS_E_WORKSPACE
    torch.cuda.synchronize()
    assert bool((sums == 3.5).all())          # nothing was launched
    assert call() == 0 and call(k=128, cutoffs=(1, 128), rpp=None, itp=None) == 0


BASE_KEYS = {"trainable_params", "non_trainable_params", "batch_time", "training_time", "history", "test_loss",
             "test_accuracy"} | {"%s_at_%d" % (m, k) for m in ("precision", "recall", "f1") for k in (5, 10)}
CATALOG_KEYS = {"catalog_%s_at_%d" % (m, k) for m in ("precision", "recall", "f1") for k in (5, 10)}
RANKING_KEYS = {"catalog_%s_at_%d" % (m, k) for m in ("ndcg", "map", "hit_rate", "mrr") for k in (5, 10)}


def test_driver_catalog_metrics_all(dev, tmp_path):
    import yaml

    from deep_cbrs_amar_renaissance_b200 import experiment as ex
    from tests.test_zz_gpu_experiment import write_inputs
    cfg, _, paths = write_inputs(tmp_path / "data")
    graph = {"load_function_name": "load_user_item_graph"}
    exps = os.path.join(str(tmp_path), "exps.yaml")
    with open(exps, "w") as fp:
        yaml.safe_dump({"linear": {
            "all": {"model": {"name": "basic.BasicGCN"}, "dataset": graph, "catalog_metrics": "all"},
            "true": {"model": {"name": "basic.BasicGCN"}, "dataset": graph, "catalog_metrics": True},
        }}, fp)
    res = ex.main(["-c", cfg, "-e", exps, "--out", str(tmp_path / "runs"), "--exp_name", "ranking"])
    assert set(res["true"]) == BASE_KEYS | CATALOG_KEYS
    got = res["all"]
    assert set(got) == BASE_KEYS | CATALOG_KEYS | RANKING_KEYS
    for key in CATALOG_KEYS | RANKING_KEYS:
        assert 0.0 <= got[key] <= 1.0, key
    assert got["catalog_hit_rate_at_10"] >= got["catalog_hit_rate_at_5"]
    for k in (5, 10):
        assert got["catalog_mrr_at_%d" % k] <= got["catalog_hit_rate_at_%d" % k]
