"""Full-catalog top-k at every k up to 128 (the largest the API takes) on every scorer path, against an independent
oracle: the fused BasicRS kernels (FFMA, 3xTF32, bf16 v1 / v2 / v3), both chained hybrid kernels, cbrs_topk_rows with
cbrs_exclude_cols, and the generic item-blocked path of scoring.catalog_top_k.

What changes with k lives in the kernels' candidate lists (capacity 2k + 32, compacted when more than 2k are filled),
in the k rounds of the compaction and of cbrs_topk_rows, in the final write loop (a lane writes several slots once
k > 32), in the shared-memory size and in the users per CTA.  So the k grid sits on the warp and list borders, the
catalogs on the 32-item tile borders and around k, the user counts around the 16-user CTA; the weights of the
adversarial orders make every item beat the threshold (rising), none after the first k (falling), or tie.

Oracles: the float64 chains of tests/helpers.py (the bf16-rounding ones for the bf16 kernels), with the tolerances of
the kernels' own parity tests.  Tolerance-free on top: the list at k is the bit-identical prefix of the list at 128,
and a user's list does not depend on which users share its CTA.  Equal returned scores come in ascending id order
where the ranking key is the returned score (the FFMA kernel, cbrs_topk_rows, the generic path); the tensor-core
kernels rank on the logit and return its sigmoid, which can round two logits to one score, so there the id order is
checked on exact duplicate items (equal logits) only."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import graph as og
from oracle import layers as ol
from tests.helpers import (HYBRID_WEIGHTS, assert_topk_equivalent, basic_chain, bf16_basic_chain, export_weights, glorot,
                           hybrid_bf16_scores, hybrid_chain_scores, hybrid_tables, random_bipartite)

pytestmark = pytest.mark.gpu

KS = (1, 2, 31, 32, 33, 63, 64, 65, 78, 79, 96, 127, 128)

# kernel -> (family, precision, c1, c2, oracle tolerance on the scores)
KERNELS = {
    "ffma-c2<=64": ("basic", "fp32-ffma", 64, 48, 2e-6),
    "ffma-c2>64": ("basic", "fp32-ffma", 32, 96, 2e-6),
    "tf32x3-c1=32": ("basic", "fp32", 32, 64, 2e-6),
    "tf32x3-c1=64": ("basic", "fp32", 64, 64, 2e-6),
    "bf16-v3": ("basic", "bf16", 64, 64, 1e-4),
    "bf16-v2": ("basic", "bf16", 64, 128, 2e-5),
    "bf16-v1-qreg": ("basic", "bf16", 64, 192, 2e-5),
    "bf16-v1": ("basic", "bf16", 128, 64, 2e-5),
    "hybrid-bf16": ("hybrid", "bf16", 64, 64, 2e-3),
    "hybrid-tf32x3": ("hybrid", "fp32", 64, 64, 1e-5),
}
HYBRID = [name for name, spec in KERNELS.items() if spec[0] == "hybrid"]
SCORE_RANKED = {name for name, spec in KERNELS.items() if spec[1] == "fp32-ffma"}   # the others rank on the logit


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _inputs(kind, n_users, n_items, seed):
    """numpy operands of a kernel: basic (P, Q, w2, b2, w3, b3), hybrid ((P1, Q1, P2, Q2), weights by name)"""
    family, _, c1, c2, _ = KERNELS[kind]
    if family == "hybrid":
        return hybrid_tables(n_users, n_items, seed)
    rng = np.random.RandomState(seed)
    P = rng.standard_normal((n_users, c1)).astype(np.float32)
    Q = rng.standard_normal((n_items, c1)).astype(np.float32)
    w2, b2 = glorot(rng, (c1, c2)), (rng.standard_normal(c2) * 0.1).astype(np.float32)
    w3, b3 = glorot(rng, (c2, 1)).reshape(-1), np.array([0.05], np.float32)
    return [P, Q, w2, b2, w3, b3]


def _users(kind, x, rows):
    """the same operands with only the user rows `rows` (an index array or slice)"""
    if KERNELS[kind][0] == "hybrid":
        (P1, Q1, P2, Q2), w = x
        return (P1[rows], Q1, P2[rows], Q2), w
    return [x[0][rows]] + list(x[1:])


def _items(kind, x, fn):
    """the same operands with fn applied to every item table"""
    if KERNELS[kind][0] == "hybrid":
        (P1, Q1, P2, Q2), w = x
        return (P1, fn(Q1), P2, fn(Q2)), w
    return [x[0], fn(x[1])] + list(x[2:])


def _run(kind, x, k, dev):
    """(ids, vals) numpy [U, k] of the kernel on the operands x"""
    from deep_cbrs_amar_renaissance_b200 import ops
    family, precision = KERNELS[kind][:2]
    if family == "basic":
        ids, vals = ops.score_catalog_topk(*(_t(a, dev) for a in x), k, precision)
    else:
        fn = ops.score_hybrid_topk_bf16 if precision == "bf16" else ops.score_hybrid_topk_tf32x3
        tabs, w = x
        ids, vals = fn(*(_t(a, dev) for a in tabs), *(_t(w[n], dev) for n in HYBRID_WEIGHTS), k)
    return ids.cpu().numpy(), vals.cpu().numpy()


def _oracle(kind, x):
    family, precision = KERNELS[kind][:2]
    if family == "basic":
        return bf16_basic_chain(*x) if precision == "bf16" else basic_chain(*x)
    tabs, w = x
    return hybrid_bf16_scores(*tabs, w) if precision == "bf16" else hybrid_chain_scores(tabs, w)


def _check_structure(ids, vals, n_items, k, what="", ties=True):
    """ids distinct and in range, scores finite and descending, exactly max(0, k - n_items) trailing -1 / -inf slots;
    ties: equal scores in ascending id order"""
    kk = min(k, n_items)
    assert ids.shape == vals.shape and ids.shape[1] == k, what
    head_i, head_v = ids[:, :kk], vals[:, :kk]
    assert (head_i >= 0).all() and (head_i < n_items).all(), "%s: ids out of range: %s" % (what, head_i[(head_i < 0) |
                                                                                                    (head_i >= n_items)][:8])
    assert all(len(set(row)) == kk for row in head_i.tolist()), "%s: an item twice in a list" % what
    assert np.isfinite(head_v).all(), what
    step = np.diff(head_v, axis=1)
    assert (step <= 0).all(), "%s: scores not descending" % what
    assert not ties or (np.diff(head_i, axis=1)[step == 0] > 0).all(), "%s: tied scores not in ascending id order" % what
    assert (ids[:, kk:] == -1).all() and np.isneginf(vals[:, kk:]).all(), \
        "%s: tail slots %s / %s" % (what, ids[:, kk:][:2], vals[:, kk:][:2])


def _same(a, b, what):
    """bit-identical (ids, vals) pairs"""
    assert np.array_equal(a[0], b[0]), "%s: ids differ in rows %s" % (what, np.nonzero((a[0] != b[0]).any(1))[0][:8])
    assert np.array_equal(a[1].view(np.uint32), b[1].view(np.uint32)), "%s: scores differ" % what


# ------------------------------------------------------------------ 1. every k border on every fused kernel
@pytest.mark.parametrize("kind", list(KERNELS))
def test_every_k_against_the_oracle(dev, kind):
    """37 users (the last CTA part-filled) x a catalog that is no multiple of the 32-item tile: every k of KS against
    the oracle, and each list the bit-identical prefix of the k = 128 list"""
    n_users, n_items = (37, 1500) if KERNELS[kind][0] == "basic" else (37, 700)
    tol = KERNELS[kind][4]
    x = _inputs(kind, n_users, n_items, 11)
    oracle = _oracle(kind, x)
    full = _run(kind, x, 128, dev)
    for k in KS:
        ids, vals = _run(kind, x, k, dev) if k != 128 else full
        _check_structure(ids, vals, n_items, k, "%s k=%d" % (kind, k), kind in SCORE_RANKED)
        assert_topk_equivalent(ids, vals, oracle, k, tol=tol)
        _same((ids, vals), (full[0][:, :k], full[1][:, :k]), "%s: k=%d vs the prefix of k=128" % (kind, k))


# ------------------------------------------------------------------ 2. catalog edges
EDGE_ITEMS = (1, 31, 32, 33, 63, 64, 65, 127, 128, 129)   # tile borders; k - 1, k, k + 1 of k = 64 and 128


def _twins(Q):
    """rows 32 and 128 copies of rows 31 and 127: exact duplicates straddling a tile border"""
    Q = Q.copy()
    for a in (31, 127):
        if len(Q) > a + 1:
            Q[a + 1] = Q[a]
    return Q


def _hybrid_refuses(kind, x, k, dev):
    """k > n_items: CBRS_E_INVALID from the C ABI, before anything is written"""
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda a: ctypes.c_void_p(a.data_ptr())
    (P1, Q1, P2, Q2), w = x
    tabs = [_t(a, dev) for a in (P1, Q1, P2, Q2)]
    wts = [_t(w[n], dev) for n in HYBRID_WEIGHTS]
    ids = torch.full((len(P1) * k,), -5, dtype=torch.int32, device=dev)
    vals = torch.full((len(P1) * k,), 3.0, device=dev)
    if KERNELS[kind][1] == "bf16":
        ws = torch.empty(lib.cbrs_score_hybrid_topk_bf16_workspace_bytes(), dtype=torch.uint8, device=dev)
        fn = lib.cbrs_score_hybrid_topk_bf16_ex
    else:
        ws = torch.empty(lib.cbrs_score_hybrid_topk_tf32x3_workspace_bytes(), dtype=torch.uint8, device=dev)
        fn = lib.cbrs_score_hybrid_topk_tf32x3
    rc = fn(*[vp(a) for a in tabs], len(P1), len(Q1), 64, *[vp(a) for a in wts], k, vp(ids), vp(vals), None, None, vp(ws),
            ws.numel(), ops._stream())
    torch.cuda.synchronize()
    assert rc == -1, (kind, k, rc)   # CBRS_E_INVALID
    assert (ids == -5).all() and (vals == 3.0).all()


@pytest.mark.parametrize("n_items", EDGE_ITEMS)
@pytest.mark.parametrize("kind", list(KERNELS))
def test_catalog_edges(dev, kind, n_items):
    n_users = 17
    x = _items(kind, _inputs(kind, n_users, n_items, n_items), _twins)
    oracle = _oracle(kind, x)
    tol = KERNELS[kind][4]
    full = None
    for k in (128, 64, 1):
        if kind in HYBRID and k > n_items:
            _hybrid_refuses(kind, x, k, dev)
            continue
        ids, vals = _run(kind, x, k, dev)
        what = "%s n_items=%d k=%d" % (kind, n_items, k)
        _check_structure(ids, vals, n_items, k, what, kind in SCORE_RANKED)
        kk = min(k, n_items)
        assert_topk_equivalent(ids[:, :kk], vals[:, :kk], oracle, kk, tol=tol)
        if full is None:
            full = ids, vals
        else:
            _same((ids, vals), (full[0][:, :k], full[1][:, :k]), what + " vs the prefix of the longest list")
        for a in (31, 127):   # twins: the same score, the lower id first
            if n_items > a + 1:
                for u in range(n_users):
                    pos = {int(i): r for r, i in enumerate(ids[u, :kk])}
                    assert not (a + 1 in pos and a not in pos), (what, u, a)
                    if a + 1 in pos:
                        assert pos[a] < pos[a + 1] and vals[u, pos[a]] == vals[u, pos[a + 1]], (what, u, a)


@pytest.mark.parametrize("kind", list(KERNELS))
def test_duplicates_across_the_catalog(dev, kind):
    """300 items made of 7 distinct rows (item i is a copy of item i % 7): every score is repeated ~43 times, bit for
    bit, so a list is whole groups, each group's items in ascending order, and the groups ranked as the oracle ranks
    them"""
    n_users, n_items = 17, 300
    x = _items(kind, _inputs(kind, n_users, n_items, 5), lambda Q: Q[np.arange(n_items) % 7])
    oracle = _oracle(kind, x)
    for k in (1, 64, 128):
        ids, vals = _run(kind, x, k, dev)
        _check_structure(ids, vals, n_items, k, "%s k=%d" % (kind, k), kind in SCORE_RANKED)
        assert_topk_equivalent(ids, vals, oracle, k, tol=KERNELS[kind][4])
        for u in range(n_users):
            groups = list(dict.fromkeys((ids[u] % 7).tolist()))   # in list order
            want = np.concatenate([np.arange(g, n_items, 7) for g in groups])[:k]
            assert np.array_equal(ids[u], want), (kind, k, u, ids[u][:12], want[:12])
            for g in groups:   # one score per group
                assert len(set(vals[u][ids[u] % 7 == g].view(np.uint32).tolist())) == 1, (kind, k, u, g)


# ------------------------------------------------------------------ 3. user-count edges
@pytest.mark.parametrize("kind", list(KERNELS))
def test_user_count_edges(dev, kind):
    """33 users (CTAs of 16 + 16 + 1) against the oracle; the same users scored as 1, 15, 16 and 17 users, and alone,
    give the same lists bit for bit, at k = 64 and 128 (the 3xTF32 hybrid chain runs 16 users per CTA at 64, 8 at 128)"""
    n_users, n_items = 33, 300
    x = _inputs(kind, n_users, n_items, 3)
    oracle = _oracle(kind, x)
    for k in (64, 128):
        full = _run(kind, x, k, dev)
        _check_structure(*full, n_items, k, kind, kind in SCORE_RANKED)
        assert_topk_equivalent(*full, oracle, k, tol=KERNELS[kind][4])
        for n in (1, 15, 16, 17):
            part = _run(kind, _users(kind, x, slice(0, n)), k, dev)
            _same(part, (full[0][:n], full[1][:n]), "%s: the first %d users of 33, k=%d" % (kind, n, k))
        for u in (0, 15, 16, 17, 31, 32):
            alone = _run(kind, _users(kind, x, slice(u, u + 1)), k, dev)
            _same(alone, (full[0][u:u + 1], full[1][u:u + 1]), "%s: user %d alone, k=%d" % (kind, u, k))


def test_hybrid_bf16_users_per_cta(dev):
    """4,800 users: the bf16 chain runs 24 users per CTA at k = 10 (one wave of two CTAs per SM) and 16 at k = 128;
    both lists agree with each other, with the oracle on the first and last 48 users, and with those users scored as
    a batch of 48 (16 users per CTA)"""
    kind, n_users, n_items = "hybrid-bf16", 4800, 130
    x = _inputs(kind, n_users, n_items, 48)
    lists = {k: _run(kind, x, k, dev) for k in (10, 128)}
    _same(lists[10], (lists[128][0][:, :10], lists[128][1][:, :10]), "k=10 vs the prefix of k=128")
    for rows in (slice(0, 48), slice(n_users - 48, n_users)):
        sub = _users(kind, x, rows)
        oracle = _oracle(kind, sub)
        for k, (ids, vals) in lists.items():
            _check_structure(ids[rows], vals[rows], n_items, k, "k=%d" % k, ties=False)
            assert_topk_equivalent(ids[rows], vals[rows], oracle, k, tol=KERNELS[kind][4])
            _same(_run(kind, sub, k, dev), (ids[rows], vals[rows]), "48 users vs 4,800, k=%d" % k)


# ------------------------------------------------------------------ 4. adversarial score orders
N_ADV = 600
# consecutive bf16 values from 1.0: every product below stays exact in bf16 / tf32 / fp32 (the weights are powers of
# two), so the logit a * t + b is strictly monotonic in t on every kernel
T_ADV = ((np.arange(N_ADV, dtype=np.uint32) + 0x3F80) << 16).view(np.float32)


def _adversarial(kind, t, n_users=17):
    """operands whose score is sigmoid(a * t[i] + b), the same for every user, with logits in [-4, 4]"""
    family, _, c1, c2, _ = KERNELS[kind]
    a = np.float32(8.0 / (T_ADV[-1] - T_ADV[0]))
    b = np.array([-4.0 - a * T_ADV[0]], np.float32)
    if family == "hybrid":
        c = 64
        P = np.zeros((n_users, c), np.float32)
        Q = np.repeat(t[:, None], c, axis=1).astype(np.float32)
        w = dict(w3a2=np.full((c, c), 2.0 ** -6, np.float32), w3b2=np.full((c, c), 2.0 ** -6, np.float32),
                 wc1=np.full((2 * c, c), 2.0 ** -7, np.float32), wc2=np.full((c, c), 2.0 ** -6, np.float32),
                 wc3=np.full(c, a / c, np.float32), bc3=b)
        for name in ("b3a2", "b3b2", "bc1", "bc2"):
            w[name] = np.zeros(c, np.float32)
        return (P, Q, P, Q), w
    P = np.zeros((n_users, c1), np.float32)
    Q = np.repeat(t[:, None], c1, axis=1).astype(np.float32)
    w2 = np.full((c1, c2), 2.0 ** -8, np.float32)               # h2 = t * c1 / 256 in every column
    w3 = np.full(c2, a * 256.0 / (c1 * c2), np.float32)
    return [P, Q, w2, np.zeros(c2, np.float32), w3, b]


ORDERS = {
    "rising": (lambda: T_ADV, lambda k: np.arange(N_ADV - 1, N_ADV - 1 - k, -1)),
    "falling": (lambda: T_ADV[::-1].copy(), lambda k: np.arange(k)),
    "tied": (lambda: np.full(N_ADV, T_ADV[N_ADV // 2], np.float32), lambda k: np.arange(k)),
    "outlier": (lambda: np.concatenate([np.full(N_ADV - 1, T_ADV[0], np.float32), T_ADV[-1:]]),
                lambda k: np.concatenate([[N_ADV - 1], np.arange(k - 1)])),
}


@pytest.mark.parametrize("order", list(ORDERS))
@pytest.mark.parametrize("kind", list(KERNELS))
def test_adversarial_orders(dev, kind, order):
    """rising: every item beats the threshold, a list is compacted every few tiles; falling: only the first k items
    ever enter; tied: ids 0..k-1; outlier: the single best item is the last one"""
    t, expect = ORDERS[order]
    x = _adversarial(kind, t())
    oracle = _oracle(kind, _users(kind, x, slice(0, 1)))
    for k in (1, 64, 128):
        ids, vals = _run(kind, x, k, dev)
        what = "%s %s k=%d" % (kind, order, k)
        _check_structure(ids, vals, N_ADV, k, what)   # the logits are strictly ordered or exactly tied
        want = expect(k)
        assert (ids == want[None, :]).all(), "%s: %s, want %s" % (what, ids[0][:8], want[:8])
        assert (vals.view(np.uint32) == vals[:1].view(np.uint32)).all(), what   # every user alike
        ref = oracle[0][want]
        assert np.abs(vals[0] - ref).max() <= KERNELS[kind][4], (what, np.abs(vals[0] - ref).max())
        if order == "tied":
            assert (vals == vals[0, 0]).all(), what


# ------------------------------------------------------------------ 5. cbrs_topk_rows and cbrs_exclude_cols
def _stable_top(s, k):
    """numpy's stable descending order: the first k (ids, scores), padded with -1 / -inf past the row"""
    order = np.argsort(-s, axis=1, kind="stable")[:, :k]
    ids = np.full((len(s), k), -1, np.int32)
    vals = np.full((len(s), k), -np.inf, np.float32)
    ids[:, :order.shape[1]] = order
    vals[:, :order.shape[1]] = np.take_along_axis(s, order, 1)
    return ids, vals


def _tie_heavy(rng, n_rows, n_cols):
    s = np.round(rng.random_sample((n_rows, n_cols)), 2).astype(np.float32)   # ~100 distinct values: long tie runs
    s[0] = 0.5                                                                 # all tied
    if n_rows > 1:
        s[1, ::7] = np.inf
        s[1, 3::11] = -np.inf
    if n_rows > 2:
        s[2] = -np.inf                                                         # nothing but -inf
    if n_rows > 3:
        s[3] = (np.arange(n_cols) % 2).astype(np.float32)                      # two values
    return s


@pytest.mark.parametrize("n_rows,n_items,k", [(9, 1000, 128), (9, 1000, 97), (6, 100, 128), (5, 1, 128), (5, 1, 1),
                                              (4, 128, 128), (4, 129, 128), (300, 257, 65)])
def test_topk_rows_against_a_stable_sort(dev, n_rows, n_items, k):
    from deep_cbrs_amar_renaissance_b200 import ops
    s = _tie_heavy(np.random.RandomState(n_items + k), n_rows, n_items)
    ids, vals = ops.topk_rows(_t(s, dev), k)
    _same((ids.cpu().numpy(), vals.cpu().numpy()), _stable_top(s, k), "topk_rows %d x %d, k=%d" % (n_rows, n_items, k))


@pytest.mark.parametrize("k", [1, 33, 128])
def test_topk_rows_on_a_strided_view_and_exclude_cols(dev, k):
    """a [9, 200] block at column 7 of [9, 300] rows (ld = 300); then cbrs_exclude_cols on it as the catalog's items
    100..299 (a block that does not start at item 0) and the top-k of what is left"""
    from deep_cbrs_amar_renaissance_b200 import ops
    rng = np.random.RandomState(k)
    buf = _tie_heavy(rng, 9, 300)
    dbuf = _t(buf, dev)
    view = dbuf[:, 7:207]
    ids, vals = ops.topk_rows(view, k)
    _same((ids.cpu().numpy(), vals.cpu().numpy()), _stable_top(buf[:, 7:207], k), "strided view")
    lists = [sorted(rng.choice(400, rng.randint(0, 150), replace=False).tolist()) for _ in range(9)]
    lists[4] = list(range(400))                                       # every item of the block
    rowptr = np.zeros(10, np.int64)
    rowptr[1:] = np.cumsum([len(x) for x in lists])
    items = np.concatenate([np.asarray(x, np.int32) for x in lists])
    ops.exclude_cols(view, 100, (_t(rowptr, dev), _t(items, dev)))
    want = buf[:, 7:207].copy()
    for r, lst in enumerate(lists):
        cols = [i - 100 for i in lst if 100 <= i < 300]
        want[r, cols] = -np.inf
    got = dbuf.cpu().numpy()
    assert np.array_equal(got[:, 7:207], want) and np.array_equal(got[:, :7], buf[:, :7]) \
        and np.array_equal(got[:, 207:], buf[:, 207:])
    ids, vals = ops.topk_rows(view, k)
    _same((ids.cpu().numpy(), vals.cpu().numpy()), _stable_top(want, k), "after exclude_cols")


# ------------------------------------------------------------------ 6. the generic path and its item-block merge
def _basic_gcn(n_users, n_items, clf_units=(64, 64), seed=12):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import basic
    set_seed(42)
    adj = random_bipartite(n_users, n_items, 20 * n_users, seed=seed)
    model = basic.BasicGCN(adj, embedding_dim=16, n_hiddens=[16, 16], n_layers=2, final_node="concatenation",
                           dense_units=[48, 48], clf_units=list(clf_units), activation="relu", dropout_rate=0.0)
    model((np.array([0]), np.array([n_users])))
    rng = np.random.RandomState(seed)
    model.set_weights([w if w.ndim > 1 and w.shape[0] > 512 else (w + rng.standard_normal(w.shape).astype(np.float32) * 0.1)
                       for w in model.get_weights()])
    model.cache_propagation = True
    return model, adj


def _basic_oracle(model, adj, n_users, n_items):
    w = export_weights(model)
    emb = ol.propagate("gcn", w["embeddings"], og.gcn_filter(adj), w["layers"])
    uu, ii = np.repeat(np.arange(n_users), n_items), np.tile(np.arange(n_items), n_users) + n_users
    return ol.basic_rs(emb, uu, ii, w["unet"], w["inet"], w["clf"]).reshape(n_users, n_items)


@pytest.mark.parametrize("n_items", [301, 100])
def test_generic_path_across_item_blocks(dev, monkeypatch, n_items):
    """fused=False with blocks of 50 items: at k = 128 the merge runs over 7 blocks (the last one 1 item) of a 301-item
    catalog, or 2 of a 100-item one (k > n_items: the 28 slots past the catalog hold -1 / -inf)"""
    from deep_cbrs_amar_renaissance_b200 import scoring
    n_users = 21
    model, adj = _basic_gcn(n_users, n_items)
    oracle = _basic_oracle(model, adj, n_users, n_items)
    monkeypatch.setattr(scoring._blocks, "__defaults__", (None, 50))
    full = None
    for k in (128, 65, 64, 33, 1):
        ids, vals = (a.cpu().numpy() for a in model.recommend_top_k(n_users, n_items, k, fused=False))
        what = "generic n_items=%d k=%d" % (n_items, k)
        _check_structure(ids, vals, n_items, k, what)
        kk = min(k, n_items)
        assert_topk_equivalent(ids[:, :kk], vals[:, :kk], oracle, kk)
        if full is None:
            full = ids, vals
        else:
            _same((ids, vals), (full[0][:, :k], full[1][:, :k]), what + " vs the prefix of k=128")
    # the fused kernels write the same tail
    ids, vals = (a.cpu().numpy() for a in model.recommend_top_k(n_users, n_items, 128, precision="fp32-ffma"))
    _check_structure(ids, vals, n_items, 128, "fused n_items=%d" % n_items)   # the FFMA kernel


def _hybrid_model(n_users, n_items):
    from deep_cbrs_amar_renaissance_b200.keras_like import set_seed
    from deep_cbrs_amar_renaissance_b200.models import hybrid
    set_seed(42)
    adj = random_bipartite(n_users, n_items, 2000, seed=18)
    bert = (np.random.RandomState(5).standard_normal((n_users + n_items, 768)) * 0.5).astype(np.float32)
    model = hybrid.HybridBertGCN(adj, embedding_dim=16, n_hiddens=[16, 16], n_layers=2, final_node="concatenation",
                                 dense_units=[[48, 48], [256, 64], [64, 64]], clf_units=[64, 64], activation="relu",
                                 dropout_rate=0.0, feature_based=True, fusion_method="concatenate", residual=False)
    model.set_content_table(bert)
    model((np.array([0]), np.array([n_users])))
    rng = np.random.RandomState(9)
    model.set_weights([w if w.ndim > 1 and w.shape[0] > 512 else (w + rng.standard_normal(w.shape).astype(np.float32) * 0.1)
                       for w in model.get_weights()])
    model.cache_propagation = True
    w = export_weights(model)
    emb = ol.propagate("gcn", w["embeddings"], og.gcn_filter(adj), w["layers"])
    uu, ii = np.repeat(np.arange(n_users), n_items), np.tile(np.arange(n_items), n_users) + n_users
    oracle = ol.hybrid_cbrs(emb, uu, ii, bert[uu], bert[ii], w, feature_based=True).reshape(n_users, n_items)
    return model, oracle


@pytest.mark.parametrize("n_items", [100, 160])
def test_hybrid_model_at_k_128(dev, monkeypatch, n_items):
    """A feature-based hybrid at k = 128: with 160 items both chained kernels take it; with 100 (k > n_items) neither
    does and both precisions run the generic path, whose lists end in 28 slots of -1 / -inf"""
    from deep_cbrs_amar_renaissance_b200 import ops, scoring
    calls = []
    for name in ("score_hybrid_topk_bf16", "score_hybrid_topk_tf32x3"):
        real = getattr(ops, name)
        monkeypatch.setattr(ops, name, lambda *a, _real=real, _name=name, **kw: calls.append(_name) or _real(*a, **kw))
    monkeypatch.setattr(scoring._blocks, "__defaults__", (None, 50))
    n_users, k = 19, 128
    model, oracle = _hybrid_model(n_users, n_items)
    kk = min(k, n_items)
    for precision, tol in (("fp32", 2e-5), ("bf16", None)):
        ids, vals = (a.cpu().numpy() for a in model.recommend_top_k(n_users, n_items, k, precision=precision))
        _check_structure(ids, vals, n_items, k, "hybrid %s n_items=%d" % (precision, n_items), ties=n_items < k)
        if tol is not None:
            assert_topk_equivalent(ids[:, :kk], vals[:, :kk], oracle, kk, tol=tol)
        else:   # the bf16 distance of tests/test_gpu_hybrid_catalog.py
            got = np.take_along_axis(oracle, ids[:, :kk].astype(np.int64), 1)
            assert np.abs(got - vals[:, :kk]).max() < 3e-2
    assert calls == ([] if n_items < k else ["score_hybrid_topk_tf32x3", "score_hybrid_topk_bf16"])


# ------------------------------------------------------------------ 7. routing x k
# (c1, c2) corners of what _fused_basic sends to a fused kernel: c1 a multiple of 8 up to 256, c2 up to 128
ROUTED = [(c1, c2) for c1 in (8, 32, 64, 72, 128, 224, 232, 256) for c2 in (1, 16, 64, 65, 128)]


@pytest.mark.parametrize("precision", ["fp32", "fp32-ffma", "bf16"])
def test_every_routed_shape_takes_k_128(dev, precision):
    """No routed classifier shape may refuse k = 128 for its shared memory (the FFMA kernel at c1 >= 232, c2 > 64 once
    did); the widest shapes' lists are checked against the oracle"""
    from deep_cbrs_amar_renaissance_b200 import ops
    n_users, n_items, k = 17, 200, 128
    for c1, c2 in ROUTED:
        rng = np.random.RandomState(c1 * 1000 + c2)
        x = [rng.standard_normal((n_users, c1)).astype(np.float32), rng.standard_normal((n_items, c1)).astype(np.float32),
             glorot(rng, (c1, c2)), (rng.standard_normal(c2) * 0.1).astype(np.float32), glorot(rng, (c2, 1)).reshape(-1),
             np.array([0.05], np.float32)]
        ids, vals = ops.score_catalog_topk(*(_t(a, dev) for a in x), k, precision)
        ids, vals = ids.cpu().numpy(), vals.cpu().numpy()
        _check_structure(ids, vals, n_items, k, "%s c1=%d c2=%d" % (precision, c1, c2), ties=precision == "fp32-ffma")
        if c1 >= 232 and c2 > 64:
            if precision == "bf16":
                assert_topk_equivalent(ids, vals, bf16_basic_chain(*x), k, tol=2e-5)
            else:
                assert_topk_equivalent(ids, vals, basic_chain(*x), k)


def test_widest_basic_classifier_at_k_128(dev):
    """BasicGCN with a 256 -> 128 classifier: recommend_top_k(k = 128) at the default precision takes the FFMA kernel"""
    n_users, n_items = 20, 300
    model, adj = _basic_gcn(n_users, n_items, clf_units=(256, 128), seed=4)
    ids, vals = (a.cpu().numpy() for a in model.recommend_top_k(n_users, n_items, 128))
    _check_structure(ids, vals, n_items, 128, "BasicGCN 256 -> 128")
    assert_topk_equivalent(ids, vals, _basic_oracle(model, adj, n_users, n_items), 128)
