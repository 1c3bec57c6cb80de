"""Per-user exclusion lists in full-catalog top-k (include/cbrs_b200.h, above cbrs_score_catalog_topk_ex): every fused
scorer variant, the chained hybrid scorer at each users-per-CTA width, and the generic item-blocked path.

Exactness oracle, tolerance-free: a kernel's per-pair score depends neither on k, nor on the lists, nor on which users
share its CTA.  So each path runs once WITHOUT lists at k = 128 on a catalog of ~300 items; the lists then remove items
inside that top-128 (the first one, every third one, the items around the 32-item tile borders, and the edge rows
below), and the top-k WITH lists (k = 1, 10, 64) must equal the filtered k = 128 list bit for bit, ids and scores."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import graph as og
from oracle import layers as ol
from tests.helpers import assert_topk_equivalent, export_weights, glorot, random_bipartite

pytestmark = pytest.mark.gpu
KS = (1, 10, 64)


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _csr(lists):
    """list of per-row item lists -> (rowptr int64, items int32) numpy, rows kept as given"""
    rowptr = np.zeros(len(lists) + 1, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.asarray(x, np.int64) for x in lists] + [np.zeros(0, np.int64)]).astype(np.int32)
    return rowptr, items


def _lists(top, n_items, seed=0):
    """Lists per user from its no-list top-128 `top` [U, 128] (ids by rank): the edge rows first, then the regular
    pattern (first item, every third, the tile-border items 31..33 / 63..65, items 0 and n_items - 1, out-of-range
    values); every list sorted ascending."""
    rng = np.random.RandomState(seed)
    lists = []
    for u in range(len(top)):
        t = [int(i) for i in top[u] if i >= 0]
        kind = u % 11
        if kind == 0:
            lst = []                                               # no list
        elif kind == 1:
            lst = t[:64]                                           # the user's whole unexcluded top-64
        elif kind == 2:
            keep = {t[5], t[50], t[100]}
            lst = [i for i in range(n_items) if i not in keep]     # all items but 3 (all of them inside the top-128)
        elif kind == 3:
            lst = list(range(n_items))                             # all items
        elif kind == 4:
            lst = [i for r, i in enumerate(t) if r % 3 == 0] * 2   # duplicates
        elif kind == 5:
            lst = [x for i in t[:60] for x in [i] * 20]            # hub: 1,200 entries that keep beating the threshold
        else:
            lst = [t[0]] + t[::3] + [31, 32, 33, 63, 64, 65, 0, n_items - 1] + list(rng.choice(n_items, 5))
            if kind == 6:
                lst += [n_items, n_items + 5, 2 ** 31 - 1, -1, -7]    # out of range: never match
        lists.append(sorted(lst))
    return lists


def _filtered(ids, vals, lists, k):
    """the k = 128 no-list result with each row's listed items removed, cut to k, padded with -1 / -inf"""
    out_i = np.full((len(ids), k), -1, np.int32)
    out_v = np.full((len(ids), k), -np.inf, np.float32)
    for u in range(len(ids)):
        s = set(lists[u])
        keep = [r for r in range(ids.shape[1]) if ids[u, r] >= 0 and int(ids[u, r]) not in s][:k]
        out_i[u, :len(keep)] = ids[u, keep]
        out_v[u, :len(keep)] = vals[u, keep]
    return out_i, out_v


def _check_exact(run, n_users, n_items, dev, seed=0):
    """run(k, exclude) -> (ids, vals) tensors.  Exactness oracle over KS; empty lists == no lists, bit for bit."""
    ids0, vals0 = (x.cpu().numpy() for x in run(128, None))
    lists = _lists(ids0, n_items, seed)
    # the filtered top-128 stands for the full ranking only as far as it reaches: at least max(KS) entries, except in
    # the rows whose whole eligible set lies inside it (all items but 3, all items)
    kept = (_filtered(ids0, vals0, lists, 128)[0] >= 0).sum(1)
    assert all(kept[u] >= max(KS) for u in range(n_users) if u % 11 not in (2, 3))
    rowptr, items = _csr(lists)
    excl = (_t(rowptr, dev), _t(items, dev))
    for k in KS:
        want_i, want_v = _filtered(ids0, vals0, lists, k)
        got_i, got_v = (x.cpu().numpy() for x in run(k, excl))
        assert np.array_equal(got_i, want_i), "k=%d: ids differ in rows %s" % (k, np.nonzero((got_i != want_i).any(1))[0][:8])
        assert np.array_equal(got_v.view(np.uint32), want_v.view(np.uint32)), "k=%d: scores differ" % k
    for u in range(min(n_users, 44)):      # edge rows with a known result
        if u % 11 == 2:
            assert (got_i[u, 3:] == -1).all() and np.isneginf(got_v[u, 3:]).all() and (got_i[u, :3] >= 0).all()
        if u % 11 == 3:
            assert (got_i[u] == -1).all() and np.isneginf(got_v[u]).all()
    empty = (torch.zeros(n_users + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev))
    for k in (10, 64):
        a, b = run(k, None), run(k, empty)
        assert torch.equal(a[0], b[0]) and torch.equal(a[1].view(torch.int32), b[1].view(torch.int32))


# (precision, c1, c2): FFMA c2 <= 64 / c2 > 64, 3xTF32 c1 = 32 / 64, bf16 v3 / v2 / v1 with the Q row in registers / v1
FUSED = [("fp32-ffma", 64, 48), ("fp32-ffma", 32, 96), ("fp32", 32, 64), ("fp32", 64, 64),
         ("bf16", 64, 64), ("bf16", 64, 128), ("bf16", 64, 192), ("bf16", 128, 64)]


@pytest.mark.parametrize("precision,c1,c2", FUSED)
def test_fused_scorers_exclude_bit_exactly(dev, precision, c1, c2):
    from deep_cbrs_amar_renaissance_b200 import ops
    n_users, n_items = 53, 301          # not multiples of the CTA's 16 users / the 32-item tile
    rng = np.random.RandomState(c1 + c2)
    P, Q = (_t(rng.standard_normal((n, c1)).astype(np.float32), dev) for n in (n_users, n_items))
    w2, b2 = _t(glorot(rng, (c1, c2)), dev), _t(rng.standard_normal(c2).astype(np.float32) * 0.1, dev)
    w3, b3 = _t(glorot(rng, (c2, 1)).reshape(-1), dev), _t(np.array([0.05], np.float32), dev)
    _check_exact(lambda k, ex: ops.score_catalog_topk(P, Q, w2, b2, w3, b3, k, precision, exclude=ex), n_users, n_items, dev)


def _hybrid_tables(dev, n_users, n_items, seed=0):
    rng = np.random.RandomState(seed)
    c = 64
    r = lambda *s: _t(rng.standard_normal(s).astype(np.float32), dev)
    t = [r(n_users, c), r(n_items, c), r(n_users, c), r(n_items, c)]
    w = [r(c, c) * 0.2, r(c) * 0.1, r(c, c) * 0.2, r(c) * 0.1, r(2 * c, c) * 0.15, r(c) * 0.1, r(c, c) * 0.2, r(c) * 0.1,
         r(c) * 0.2, _t(np.array([0.02], np.float32), dev)]
    return t, w


@pytest.mark.parametrize("n_users", [4001, 5999, 9001])
def test_hybrid_scorer_excludes_bit_exactly(dev, n_users):
    """n_users where the dispatch of cbrs_score_hybrid_topk_bf16 considers 16, 24 and 32 users per CTA (k = 1 and 10 run
    at 24 for 5,999 users; wider widths need more shared memory than two CTAs per SM leave at any k)"""
    from deep_cbrs_amar_renaissance_b200 import ops
    n_items = 299
    t, w = _hybrid_tables(dev, n_users, n_items, n_users)
    _check_exact(lambda k, ex: ops.score_hybrid_topk_bf16(*t, *w, k, exclude=ex), n_users, n_items, dev)


def _basic_model(n_users, n_items, seed=12):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic
    set_seed(42)
    adj = random_bipartite(n_users, n_items, 30 * n_users, seed=seed)
    model = basic.BasicGCN(adj, embedding_dim=16, n_hiddens=[16, 16], n_layers=2, final_node="concatenation",
                           dense_units=[48, 48], clf_units=[64, 64], activation="relu", dropout_rate=0.0)
    model((np.array([0]), np.array([n_users])))
    rng = np.random.RandomState(seed)
    model.set_weights([w if w.ndim > 1 and w.shape[0] > 512 else (w + rng.standard_normal(w.shape).astype(np.float32) * 0.1)
                       for w in model.get_weights()])
    model.cache_propagation = True
    return model, adj


def _item_lists(rowptr, items, n_items):
    from deep_cbrs_amar_renaissance_b200.scoring import ItemLists
    return ItemLists(rowptr, items, n_items)


def test_generic_path_excludes_bit_exactly_across_item_blocks(dev, monkeypatch):
    """fused=False: score blocks of 100 items (lists cross the block borders), cbrs_exclude_cols, top-k and the merge"""
    from deep_cbrs_amar_renaissance_b200 import scoring
    n_users, n_items = 47, 301
    model, _ = _basic_model(n_users, n_items)
    monkeypatch.setattr(scoring._blocks, "__defaults__", (None, 100))
    _check_exact(lambda k, ex: model.recommend_top_k(n_users, n_items, k, fused=False,
                                                     exclude=None if ex is None else _item_lists(*ex, n_items)),
                 n_users, n_items, dev)


def _oracle_excluded(scores, lists):
    """excluded entries replaced by distinct finite values below every sigmoid output (no -inf into gap arithmetic)"""
    s = np.array(scores, np.float64)
    for u, lst in enumerate(lists):
        lst = [i for i in lst if 0 <= i < s.shape[1]]
        s[u, lst] = -1.0 - np.asarray(lst, np.float64)
    return s


def _random_lists(n_users, n_items, seed, max_len):
    rng = np.random.RandomState(seed)
    return [sorted(rng.choice(n_items, rng.randint(0, max_len), replace=False).tolist()) for _ in range(n_users)]


def test_basic_gcn_against_float64_oracle(dev):
    from deep_cbrs_amar_renaissance_b200.scoring import catalog_scores
    n_users, n_items, k = 203, 333, 10
    model, adj = _basic_model(n_users, n_items, seed=3)
    lists = _random_lists(n_users, n_items, 4, 200)
    ex = _item_lists(*(_t(a, dev) for a in _csr(lists)), n_items)
    w = export_weights(model)
    emb = ol.propagate("gcn", w["embeddings"], og.gcn_filter(adj), w["layers"])
    uu, ii = np.repeat(np.arange(n_users), n_items), np.tile(np.arange(n_items), n_users) + n_users
    oracle = _oracle_excluded(ol.basic_rs(emb, uu, ii, w["unet"], w["inet"], w["clf"]).reshape(n_users, n_items), lists)
    for kw in (dict(), dict(precision="fp32-ffma"), dict(fused=False)):
        ids, vals = model.recommend_top_k(n_users, n_items, k, exclude=ex, **kw)
        assert assert_topk_equivalent(ids.cpu().numpy(), vals.cpu().numpy(), oracle, k) > 0.95, kw
    # the generic path against a stable sort of its own score matrix, listed items dropped
    dense = _oracle_excluded(catalog_scores(model, model.propagate(), n_users, n_items).cpu().numpy(), lists)
    ids, vals = model.recommend_top_k(n_users, n_items, k, fused=False, exclude=ex)
    order = np.argsort(-dense, axis=1, kind="stable")[:, :k]
    assert np.array_equal(ids.cpu().numpy(), order)
    assert np.array_equal(vals.cpu().numpy(), np.take_along_axis(dense, order, 1).astype(np.float32))


def test_feature_based_hybrid_against_float64_oracle(dev):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import hybrid
    n_users, n_items, dim, k = 90, 260, 768, 10
    set_seed(42)
    adj = random_bipartite(n_users, n_items, 4000, seed=18)
    bert = (np.random.RandomState(5).standard_normal((n_users + n_items, dim)) * 0.5).astype(np.float32)
    model = hybrid.HybridBertGCN(adj, embedding_dim=16, n_hiddens=[16, 16], n_layers=2, final_node="concatenation",
                                 dense_units=[[48, 48], [256, 64], [64, 64]], clf_units=[64, 64], activation="relu",
                                 dropout_rate=0.0, feature_based=True, fusion_method="concatenate", residual=False)
    model.set_content_table(bert)
    model((np.array([0]), np.array([n_users])))
    rng = np.random.RandomState(9)
    model.set_weights([w if w.ndim > 1 and w.shape[0] > 512 else (w + rng.standard_normal(w.shape).astype(np.float32) * 0.1)
                       for w in model.get_weights()])
    model.cache_propagation = True
    lists = _random_lists(n_users, n_items, 6, 150)
    ex = _item_lists(*(_t(a, dev) for a in _csr(lists)), n_items)
    w = export_weights(model)
    emb = ol.propagate("gcn", w["embeddings"], og.gcn_filter(adj), w["layers"])
    uu, ii = np.repeat(np.arange(n_users), n_items), np.tile(np.arange(n_items), n_users) + n_users
    oracle = _oracle_excluded(ol.hybrid_cbrs(emb, uu, ii, bert[uu], bert[ii], w, feature_based=True)
                              .reshape(n_users, n_items), lists)
    ids, vals = model.recommend_top_k(n_users, n_items, k, exclude=ex)            # fp32: the generic path
    assert assert_topk_equivalent(ids.cpu().numpy(), vals.cpu().numpy(), oracle, k, tol=2e-5) > 0.5
    ids, vals = model.recommend_top_k(n_users, n_items, k, exclude=ex, precision="bf16")   # the chained bf16 kernel
    ids = ids.cpu().numpy()
    assert (ids >= 0).all() and not any(int(i) in set(lists[u]) for u in range(n_users) for i in ids[u])
    got = np.take_along_axis(oracle, ids.astype(np.int64), 1)
    ref = -np.sort(-oracle, axis=1)[:, :k]
    assert np.abs(got - ref).max() < 3e-2     # the bf16 distance of tests/test_gpu_hybrid_catalog.py


@pytest.mark.parametrize("kw", [dict(), dict(precision="fp32-ffma"), dict(precision="bf16"), dict(fused=False)])
def test_user_subsets_and_empty_lists(dev, kw):
    n_users, n_items, k = 70, 250, 10
    model, _ = _basic_model(n_users, n_items, seed=8)
    lists = _random_lists(n_users, n_items, 9, 120)
    ex = _item_lists(*(_t(a, dev) for a in _csr(lists)), n_items)
    full_i, full_v = model.recommend_top_k(n_users, n_items, k, exclude=ex, **kw)
    none_i, none_v = model.recommend_top_k(n_users, n_items, k, **kw)
    empty = _item_lists(torch.zeros(n_users + 1, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int32, device=dev),
                        n_items)
    e_i, e_v = model.recommend_top_k(n_users, n_items, k, exclude=empty, **kw)
    assert torch.equal(e_i, none_i) and torch.equal(e_v.view(torch.int32), none_v.view(torch.int32))
    for u in range(n_users):
        assert not set(full_i[u].tolist()) & set(lists[u])
    for sub in ([33, 5, 69, 5, 0, 17], list(range(21, 38))):   # unsorted with a repeat; contiguous (a rowptr slice)
        users = torch.tensor(sub, device=dev)
        si, sv = model.recommend_top_k(n_users, n_items, k, users=users, exclude=ex, **kw)
        assert torch.equal(si, full_i[users]) and torch.equal(sv.view(torch.int32), full_v[users].view(torch.int32))


# ------------------------------------------------------------------ guard bands around lists, ids and scores
SENT = -7.25e30
GUARD = 2048


class _Arena:
    def __init__(self, dev, floats):
        self.buf = torch.full((floats,), SENT, device=dev, dtype=torch.float32)
        self.used = torch.zeros(floats, dtype=torch.bool, device=dev)
        self.off = GUARD

    def block(self, rows, cols, ld):
        """float32 [rows, cols] view with leading dimension ld, 32-byte aligned, guard bands around it"""
        self.off = (self.off + 7) // 8 * 8
        view = self.buf[self.off:self.off + rows * ld].view(rows, ld)[:, :cols]
        self.used[self.off:self.off + rows * ld].view(rows, ld)[:, :cols] = True
        self.off += rows * ld + GUARD
        assert self.off + GUARD <= self.buf.numel()
        return view

    def take(self, n, dtype=torch.float32):
        """n contiguous elements of `dtype`"""
        words = max(1, n * torch.empty(0, dtype=dtype).element_size() // 4)
        return self.block(1, words, words).reshape(-1).view(dtype)

    def check(self, what):
        sent = torch.tensor([SENT], dtype=torch.float32).view(torch.int32).item()
        bad = (~self.used) & (self.buf.view(torch.int32) != sent)
        assert not bool(bad.any()), "%s wrote outside its output: %d stray words" % (what, int(bad.sum()))


def _guarded_lists(arena, n_users, n_items, dev):
    """lists with unsorted rows and long neighbours, each in its own guarded slice"""
    rng = np.random.RandomState(1)
    lists = []
    for u in range(n_users):
        if u % 4 == 0:
            lists.append(rng.permutation(n_items)[:40].tolist())          # unsorted
        elif u % 4 == 1:
            lists.append(sorted(rng.randint(0, n_items, 900).tolist()))    # long
        else:
            lists.append(sorted(rng.choice(n_items, 7, replace=False).tolist()))
    rowptr, items = _csr(lists)
    rp = arena.take(len(rowptr), torch.int64)
    it = arena.take(len(items), torch.int32)
    rp.copy_(_t(rowptr, dev))
    it.copy_(_t(items, dev))
    return rp, it, lists


def test_ex_entry_points_stay_inside_their_buffers(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ops._stream()
    n_users, n_items, k = 37, 203, 11
    rng = np.random.RandomState(2)
    for name, c1, c2 in (("ffma", 64, 96), ("tf32x3", 64, 64), ("bf16", 64, 64), ("bf16", 64, 128), ("bf16", 128, 64),
                         ("hybrid", 64, 64)):
        a = _Arena(dev, 40 * GUARD + 2 * n_users * k + 2 * 30000)
        rp, it, _ = _guarded_lists(a, n_users, n_items, dev)
        ids = a.take(n_users * k, torch.int32)
        vals = a.take(n_users * k)
        if name == "hybrid":
            t, w = _hybrid_tables(dev, n_users, n_items, 3)
            ws = torch.empty(lib.cbrs_score_hybrid_topk_bf16_workspace_bytes(), dtype=torch.uint8, device=dev)
            rc = lib.cbrs_score_hybrid_topk_bf16_ex(*[vp(x) for x in t], n_users, n_items, 64, *[vp(x) for x in w], k, vp(ids),
                                                    vp(vals), vp(rp), vp(it), vp(ws), ws.numel(), st)
        else:
            P, Q = (_t(rng.standard_normal((n, c1)).astype(np.float32), dev) for n in (n_users, n_items))
            w2, b2 = _t(glorot(rng, (c1, c2)), dev), _t(rng.standard_normal(c2).astype(np.float32) * 0.1, dev)
            w3, b3 = _t(glorot(rng, (c2, 1)).reshape(-1), dev), _t(np.array([0.05], np.float32), dev)
            args = [vp(P), c1, vp(Q), c1, n_users, n_items, c1, vp(w2), vp(b2), c2, vp(w3), vp(b3), k, vp(ids), vp(vals),
                    vp(rp), vp(it)]
            if name == "ffma":
                rc = lib.cbrs_score_catalog_topk_ex(*args, st)
            elif name == "tf32x3":
                ws = torch.empty(lib.cbrs_score_catalog_topk_tf32x3_workspace_bytes(c1, c2), dtype=torch.uint8, device=dev)
                rc = lib.cbrs_score_catalog_topk_tf32x3_ex(*args, vp(ws), ws.numel(), st)
            else:
                ws = torch.empty(lib.cbrs_score_catalog_topk_bf16_workspace_bytes(n_items, c1, c2), dtype=torch.uint8,
                                 device=dev)
                rc = lib.cbrs_score_catalog_topk_bf16_ex(*args, vp(ws), ws.numel(), st)
        _lib.check(rc, name)
        torch.cuda.synchronize()
        a.check("%s (%d, %d)" % (name, c1, c2))
        assert (ids.view(n_users, k) >= -1).all() and (ids.view(n_users, k) < n_items).all()
    # cbrs_exclude_cols on a strided block: only the block's own columns may change
    a = _Arena(dev, 40 * GUARD + 30000 + n_users * 120)
    rp, it, lists = _guarded_lists(a, n_users, n_items, dev)
    block = a.block(n_users, 90, 120)
    block.fill_(0.5)
    ops.exclude_cols(block, 100, (rp, it))
    torch.cuda.synchronize()
    a.check("exclude_cols")
    got = block.cpu().numpy()
    for u, lst in enumerate(lists):
        want = np.full(90, 0.5, np.float32)
        if u % 4 != 0:     # sorted rows: exactly the listed items inside [100, 190)
            want[[i - 100 for i in lst if 100 <= i < 190]] = -np.inf
            assert np.array_equal(got[u], want), u
        else:              # unsorted rows: a subset of their own items
            assert set(np.nonzero(np.isneginf(got[u]))[0] + 100) <= set(lst)


def test_one_null_list_pointer_is_invalid(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    st = ops._stream()
    f = torch.zeros(64 * 64, device=dev)
    ids = torch.zeros(16, dtype=torch.int32, device=dev)
    rp = torch.zeros(2, dtype=torch.int64, device=dev)
    it = torch.zeros(1, dtype=torch.int32, device=dev)
    ws = torch.empty(1 << 20, dtype=torch.uint8, device=dev)
    for rpp, itp, missing in ((vp(rp), None, "excl_items"), (None, vp(it), "excl_rowptr")):
        common = [vp(f), 64, vp(f), 64, 1, 8, 64, vp(f), vp(f), 64, vp(f), vp(f), 4, vp(ids), vp(f), rpp, itp]
        for rc in (lib.cbrs_score_catalog_topk_ex(*common, st),
                   lib.cbrs_score_catalog_topk_tf32x3_ex(*common, vp(ws), ws.numel(), st),
                   lib.cbrs_score_catalog_topk_bf16_ex(*common, vp(ws), ws.numel(), st),
                   lib.cbrs_score_hybrid_topk_bf16_ex(*[vp(f)] * 4, 1, 8, 64, *[vp(f)] * 10, 4, vp(ids), vp(f), rpp, itp,
                                                      vp(ws), ws.numel(), st),
                   lib.cbrs_exclude_cols(vp(f), 64, 1, 8, 0, rpp, itp, st)):
            assert rc == -1   # CBRS_E_INVALID
            assert (missing + " is null").encode() in lib.cbrs_last_error()


# ------------------------------------------------------------------ metrics and the experiment driver
def _rival(test, top_ids, users, items, k):
    """numpy restatement of RiVal 0.2 P/R/F1@k on full-catalog lists top_ids [U, >= k] (catalog indices)"""
    rel = {}
    for u, i, r in test:
        if r >= 1:
            rel.setdefault(u, set()).add(i)
    index = {u: r for r, u in enumerate(users)}
    ps, rs = [], []
    for u, its in rel.items():
        rec = [items[i] for i in top_ids[index[u], :k] if i >= 0] if u in index else []
        tp = len(set(rec) & its)
        ps.append(tp / k)
        rs.append(tp / len(its))
    p, r = float(np.mean(ps)), float(np.mean(rs))
    return p, r, (2 * p * r / (p + r) if p + r > 0 else 0.0)


def test_catalog_metrics_match_a_numpy_restatement(dev):
    from deep_cbrs_amar_renaissance_b200.scoring import ItemLists
    from deep_cbrs_amar_renaissance_b200.utilities.metrics import catalog_predictions, precision_recall_f1_at_k
    n_users, n_items = 80, 120
    model, adj = _basic_model(n_users, n_items, seed=21)
    rng = np.random.RandomState(3)
    coo = adj.tocoo() if hasattr(adj, "tocoo") else adj.coo
    mask = (coo.row < n_users) & (coo.col >= n_users)
    train = np.stack([coo.row[mask], coo.col[mask], rng.randint(0, 2, mask.sum())], 1)
    test = np.stack([rng.randint(0, n_users, 600), rng.randint(0, n_items, 600), rng.randint(0, 2, 600)], 1)
    users, items = np.arange(1000, 1000 + n_users), np.arange(5000, 5000 + n_items)
    seen = ItemLists.from_ratings(train, n_users, n_items, device=dev)
    ids, vals = model.recommend_top_k(n_users, n_items, 10, exclude=seen)
    w = export_weights(model)
    emb = ol.propagate("gcn", w["embeddings"], og.gcn_filter(adj), w["layers"])
    uu, ii = np.repeat(np.arange(n_users), n_items), np.tile(np.arange(n_items), n_users) + n_users
    lists = [sorted(set(train[train[:, 0] == u, 1] - n_users)) for u in range(n_users)]
    oracle = _oracle_excluded(ol.basic_rs(emb, uu, ii, w["unet"], w["inet"], w["clf"]).reshape(n_users, n_items), lists)
    order = np.argsort(-oracle, axis=1, kind="stable")[:, :10]
    assert np.array_equal(ids.cpu().numpy(), order)    # no near-ties at this size
    frame = catalog_predictions(ids, vals, users, items)
    assert len(frame) == n_users * 10 and frame["users"].tolist() == np.repeat(users, 10).tolist()
    test_orig = np.stack([users[test[:, 0]], items[test[:, 1]], test[:, 2]], 1)
    for k in (5, 10):
        got = precision_recall_f1_at_k(test_orig, frame.to_numpy(), k)
        want = _rival(test_orig, order, users, items, k)
        assert np.allclose([got["precision"], got["recall"], got["f1"]], want, rtol=0, atol=1e-12), (k, got, want)


BASE_KEYS = {"trainable_params", "non_trainable_params", "batch_time", "training_time", "history", "test_loss",
             "test_accuracy"} | {"%s_at_%d" % (m, k) for m in ("precision", "recall", "f1") for k in (5, 10)}
CATALOG_KEYS = {"catalog_%s_at_%d" % (m, k) for m in ("precision", "recall", "f1") for k in (5, 10)}


def test_driver_catalog_metrics_is_opt_in(dev, tmp_path):
    import yaml

    from deep_cbrs_amar_renaissance_b200 import experiment as ex
    from tests.test_zz_gpu_experiment import write_inputs
    cfg, _, paths = write_inputs(tmp_path / "data")
    graph = {"load_function_name": "load_user_item_graph"}
    bert = {"load_function_name": "load_user_item_graph_bert_embeddings"}
    hyb = {"name": "hybrid.HybridBertGCN", "dense_units": [[16, 16], [16, 8], [16, 16]]}
    exps = os.path.join(str(tmp_path), "exps.yaml")
    with open(exps, "w") as fp:
        yaml.safe_dump({"linear": {
            "plain": {"model": {"name": "basic.BasicGCN"}, "dataset": graph},
            "catalog": {"model": {"name": "basic.BasicGCN"}, "dataset": graph, "catalog_metrics": True},
            "catalog-hybrid": {"model": hyb, "dataset": bert, "catalog_metrics": True},
        }}, fp)
    res = ex.main(["-c", cfg, "-e", exps, "--out", str(tmp_path / "runs"), "--exp_name", "catalog"])
    assert set(res["plain"]) == BASE_KEYS
    for name in ("catalog", "catalog-hybrid"):
        assert set(res[name]) == BASE_KEYS | CATALOG_KEYS, name
        for key in CATALOG_KEYS:
            assert 0.0 <= res[name][key] <= 1.0
    # the scorers over pre-computed embedding rows have no full-catalog top-k: refused before training
    config = ex.load_yaml(cfg)
    config["catalog_metrics"] = True
    with pytest.raises(ValueError, match="catalog_metrics"):
        ex.Experimenter(config, str(tmp_path / "refused"))
