"""GPU tests of the fp32-accurate chained catalog scorer of the feature-based hybrid model (cbrs_score_hybrid_topk_tf32x3:
the five 64 x 64 products of the reference's src/models/hybrid.py:72-89 as 3xTF32 on the tensor cores).

Oracle: the chain in float64.  The stated fp32 tolerance of the catalog scorers is 1e-5 on the (sigmoid) scores, ids
compared where the oracle's gaps exceed it.  A single-TF32 evaluation of the same chain must miss that tolerance, so the
tests fail if a correction term of the split is dropped."""
import ctypes

import numpy as np
import pytest
import torch

from tests.helpers import (HYBRID_WEIGHTS, assert_topk_equivalent, hybrid_chain, hybrid_chain_scores, hybrid_tables,
                           random_bipartite)
from tests.test_gpu_catalog_exclusion import (GUARD, _Arena, _check_exact, _csr, _guarded_lists, _hybrid_tables,
                                              _item_lists, _random_lists, _rival)

pytestmark = pytest.mark.gpu
TOL = 1e-5


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    torch.cuda.set_device(0)
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def _run(tabs, w, k, dev, exclude=None):
    from deep_cbrs_amar_renaissance_b200 import ops
    return ops.score_hybrid_topk_tf32x3(*[_t(x, dev) for x in tabs], *[_t(w[n], dev) for n in HYBRID_WEIGHTS], k,
                                        exclude=exclude)


@pytest.mark.parametrize("n_users,n_items,k", [(37, 1000, 10), (5, 7, 5), (130, 333, 20), (16, 32, 3), (1, 2049, 10),
                                               (4800, 40, 5), (300, 5000, 64), (64, 300, 128)])
def test_against_float64_chain(dev, n_users, n_items, k):
    tabs, w = hybrid_tables(n_users, n_items, n_users + n_items)
    ids, vals = (x.cpu().numpy() for x in _run(tabs, w, k, dev))
    assert (ids >= 0).all() and (ids < n_items).all()
    assert all(len(set(row)) == k for row in ids)                       # no item twice
    assert (np.diff(vals, axis=1) <= 0).all()                           # descending
    oracle = hybrid_chain_scores(tabs, w)
    assert_topk_equivalent(ids, vals, oracle, k, tol=TOL)
    uu = np.repeat(np.arange(n_users), k)
    got = np.take_along_axis(oracle, ids.astype(np.int64), 1)
    assert np.abs(got - vals).max() <= TOL
    # a single-TF32 evaluation of the same pairs misses the tolerance: the kernel's accuracy comes from the split
    single = hybrid_chain(*tabs, w, uu, ids.reshape(-1).astype(np.int64), rounded=True).reshape(n_users, k)
    assert np.abs(single - got).max() > TOL


@pytest.mark.parametrize("k", [12, 128])
def test_exact_ties_go_to_the_lower_item(dev, k):
    from deep_cbrs_amar_renaissance_b200 import ops
    n_users, n_items, c = 20, 300, 64
    z = lambda *s: torch.zeros(*s, device=dev)
    ids, vals = ops.score_hybrid_topk_tf32x3(z(n_users, c), z(n_items, c), z(n_users, c), z(n_items, c), z(c, c), z(c),
                                             z(c, c), z(c), z(2 * c, c), z(c), z(c, c), z(c), z(c), z(1), k)
    assert (ids.cpu().numpy() == np.arange(k)[None, :]).all() and (vals == 0.5).all()


@pytest.mark.parametrize("n_users", [53, 1203])
def test_exclusion_bit_exactly(dev, n_users):
    """k = 1, 10, 64 run at 16 users per CTA, the k = 128 reference at 8; neither user count fills its last CTA"""
    from deep_cbrs_amar_renaissance_b200 import ops
    n_items = 299
    t, w = _hybrid_tables(dev, n_users, n_items, n_users)
    _check_exact(lambda k, ex: ops.score_hybrid_topk_tf32x3(*t, *w, k, exclude=ex), n_users, n_items, dev)


@pytest.mark.parametrize("k", [10, 128])
def test_position_invariance_and_determinism(dev, k):
    from deep_cbrs_amar_renaissance_b200 import ops
    n_users, n_items = 90, 517
    t, w = _hybrid_tables(dev, n_users, n_items, 7)
    a_i, a_v = ops.score_hybrid_topk_tf32x3(*t, *w, k)
    b_i, b_v = ops.score_hybrid_topk_tf32x3(*t, *w, k)
    assert torch.equal(a_i, b_i) and torch.equal(a_v.view(torch.int32), b_v.view(torch.int32))
    sub = torch.tensor([33, 5, 89, 5, 0, 17, 64, 63, 16, 15], device=dev)
    s_i, s_v = ops.score_hybrid_topk_tf32x3(t[0][sub], t[1], t[2][sub], t[3], *w, k)
    assert torch.equal(s_i, a_i[sub]) and torch.equal(s_v.view(torch.int32), a_v[sub].view(torch.int32))


def test_c_abi_status_codes(dev):
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda x: ctypes.c_void_p(x.data_ptr())
    st = ops._stream()
    n_users, n_items, k = 5, 40, 4
    t, w = _hybrid_tables(dev, n_users, n_items, 3)
    ids = torch.full((n_users * k,), -5, dtype=torch.int32, device=dev)
    vals = torch.full((n_users * k,), 3.0, device=dev)
    need = lib.cbrs_score_hybrid_topk_tf32x3_workspace_bytes()
    assert need == 5 * 32768
    ws = torch.empty(need + 64, dtype=torch.uint8, device=dev)
    rp = torch.zeros(n_users + 1, dtype=torch.int64, device=dev)
    it = torch.zeros(1, dtype=torch.int32, device=dev)

    def call(tabs=None, nu=n_users, ni=n_items, c=64, kk=k, lists=(None, None), wsp=None, wsb=need, wts=None, out=None):
        tabs = [vp(x) for x in t] if tabs is None else tabs
        wts = [vp(x) for x in w] if wts is None else wts
        o = (vp(ids), vp(vals)) if out is None else out
        return lib.cbrs_score_hybrid_topk_tf32x3(*tabs, nu, ni, c, *wts, kk, *o, *lists,
                                                 vp(ws) if wsp is None else wsp, wsb, st)

    assert call() == 0
    torch.cuda.synchronize()
    assert (ids >= 0).all()
    for i in range(4):   # null tables
        tabs = [vp(x) for x in t]
        tabs[i] = None
        assert call(tabs=tabs) == -1
    for i in range(10):  # null weights / biases
        wts = [vp(x) for x in w]
        wts[i] = None
        assert call(wts=wts) == -1
    assert call(out=(None, vp(vals))) == -1 and call(out=(vp(ids), None)) == -1
    assert call(wsp=ctypes.c_void_p(0)) == -1
    for lists, missing in (((vp(rp), None), "excl_items"), ((None, vp(it)), "excl_rowptr")):
        assert call(lists=lists) == -1
        assert (missing + " is null").encode() in lib.cbrs_last_error()
    assert call(c=32) == -4                                   # CBRS_E_UNSUPPORTED
    for kk, ni in ((0, n_items), (-1, n_items), (129, 300), (41, n_items)):
        assert call(kk=kk, ni=ni) == -1, (kk, ni)
    assert call(nu=-1) == -1
    assert call(wsb=need - 1) == -2                           # CBRS_E_WORKSPACE
    assert call(wsp=ctypes.c_void_p(ws.data_ptr() + 8)) == -2
    ids.fill_(-5)
    vals.fill_(3.0)
    assert call(nu=0) == 0
    torch.cuda.synchronize()
    assert (ids == -5).all() and (vals == 3.0).all()          # n_users == 0 writes nothing
    big_i = torch.empty(n_users * n_items, dtype=torch.int32, device=dev)
    big_v = torch.empty(n_users * n_items, device=dev)
    assert call(kk=n_items, out=(vp(big_i), vp(big_v))) == 0    # k = n_items is valid
    torch.cuda.synchronize()
    assert (torch.sort(big_i.view(n_users, n_items), 1).values == torch.arange(n_items, device=dev)).all()


@pytest.mark.parametrize("k", [11, 128])
def test_stays_inside_its_buffers(dev, k):
    from deep_cbrs_amar_renaissance_b200 import _lib, ops
    lib = _lib.load()
    vp = lambda x: ctypes.c_void_p(x.data_ptr())
    n_users, n_items = 37, 203
    need = lib.cbrs_score_hybrid_topk_tf32x3_workspace_bytes()
    a = _Arena(dev, 40 * GUARD + 2 * n_users * k + 2 * 30000 + need // 4)
    rp, it, lists = _guarded_lists(a, n_users, n_items, dev)
    ids = a.take(n_users * k, torch.int32)
    vals = a.take(n_users * k)
    ws = a.take(need // 4)
    t, w = _hybrid_tables(dev, n_users, n_items, 3)
    for lp in ((vp(rp), vp(it)), (None, None)):
        rc = lib.cbrs_score_hybrid_topk_tf32x3(*[vp(x) for x in t], n_users, n_items, 64, *[vp(x) for x in w], k, vp(ids),
                                               vp(vals), *lp, vp(ws), need, ops._stream())
        _lib.check(rc, "tf32x3 hybrid")
        torch.cuda.synchronize()
        a.check("cbrs_score_hybrid_topk_tf32x3 (k = %d)" % k)
        got = ids.view(n_users, k).cpu().numpy()
        assert (got >= -1).all() and (got < n_items).all()
        if lp[0] is not None:   # sorted rows: none of their items may appear
            for u in range(n_users):
                if u % 4:
                    assert not set(got[u].tolist()) & set(lists[u])


# ------------------------------------------------------------------ model level
GRID = (16, [16, 16], [[48, 48], [256, 64], [64, 64]], [64, 64])   # econfigs/hybrid-gnn.yaml shapes


def _hybrid_model(n_users, n_items, grid=GRID, **extra):
    from tests.test_gpu_models import _build, _randomise
    adj = random_bipartite(n_users, n_items, 5000, seed=28)
    bert = (np.random.RandomState(5).standard_normal((n_users + n_items, 768)) * 0.5).astype(np.float32)
    kw = dict(feature_based=True, fusion_method="concatenate", residual=False)
    kw.update(extra)
    model = _build("HybridBertGCN", adj, grid, module="hybrid", **kw)
    model.set_content_table(bert)
    model((np.array([0]), np.array([n_users])))
    _randomise(model, 3)
    model.cache_propagation = True
    return model


@pytest.fixture
def spy(monkeypatch):
    from deep_cbrs_amar_renaissance_b200 import ops
    calls = []
    real = ops.score_hybrid_topk_tf32x3

    def wrapped(*a, **kw):
        calls.append(a[-1])
        return real(*a, **kw)
    monkeypatch.setattr(ops, "score_hybrid_topk_tf32x3", wrapped)
    return calls


def test_model_fp32_takes_the_kernel_and_matches_the_generic_path(dev, spy):
    n_users, n_items, k = 70, 400, 10
    model = _hybrid_model(n_users, n_items)
    ids, vals = model.recommend_top_k(n_users, n_items, k, precision="fp32")
    assert len(spy) == 1
    gi, gv = model.recommend_top_k(n_users, n_items, k + 1, fused=False)
    assert len(spy) == 1
    ids, vals, gi, gv = ids.cpu().numpy(), vals.cpu().numpy(), gi.cpu().numpy(), gv.cpu().numpy()
    assert np.abs(vals - gv[:, :k]).max() <= TOL
    gaps = gv[:, :-1] - gv[:, 1:]
    prev = np.concatenate([np.full((n_users, 1), np.inf), gaps[:, :-1]], 1)
    clear = (gaps > 2e-5) & (prev > 2e-5)
    assert clear.mean() > 0.5 and (ids[clear] == gi[:, :k][clear]).all()


def test_model_exclusion_and_user_subsets(dev, spy):
    n_users, n_items, k = 70, 400, 10
    model = _hybrid_model(n_users, n_items)
    lists = _random_lists(n_users, n_items, 9, 150)
    ex = _item_lists(*(_t(x, dev) for x in _csr(lists)), n_items)
    full_i, full_v = model.recommend_top_k(n_users, n_items, k, exclude=ex)
    for u in range(n_users):
        assert not set(full_i[u].tolist()) & set(lists[u])
    for sub in ([33, 5, 69, 5, 0, 17], list(range(21, 38))):   # unsorted with a repeat; contiguous (a rowptr slice)
        users = torch.tensor(sub, device=dev)
        si, sv = model.recommend_top_k(n_users, n_items, k, users=users, exclude=ex)
        assert torch.equal(si, full_i[users]) and torch.equal(sv.view(torch.int32), full_v[users].view(torch.int32))
        si, sv = model.recommend_top_k(n_users, n_items, k, users=users)
        ni, nv = model.recommend_top_k(n_users, n_items, k)
        assert torch.equal(si, ni[users]) and torch.equal(sv.view(torch.int32), nv[users].view(torch.int32))
    assert len(spy) == 7


@pytest.mark.parametrize("case", ["fp32-ffma", "c16", "attention", "residual"])
def test_other_routes_do_not_take_the_kernel(dev, spy, case):
    n_users, n_items, k = 40, 150, 5
    if case == "fp32-ffma":
        model, precision = _hybrid_model(n_users, n_items), "fp32-ffma"
    elif case == "c16":
        model, precision = _hybrid_model(n_users, n_items, (16, [16, 16], [[48, 48], [256, 64], [16, 16]], [64, 64])), "fp32"
    elif case == "attention":
        model, precision = _hybrid_model(n_users, n_items, fusion_method="attention"), "fp32"
    else:
        model, precision = _hybrid_model(n_users, n_items, residual=True), "fp32"
    ids, vals = model.recommend_top_k(n_users, n_items, k, precision=precision)
    assert spy == []
    gi, gv = model.recommend_top_k(n_users, n_items, k, fused=False)
    assert torch.equal(ids, gi) and torch.equal(vals.view(torch.int32), gv.view(torch.int32))


def test_driver_catalog_metrics_use_the_kernel(dev, tmp_path, spy):
    from deep_cbrs_amar_renaissance_b200 import experiment as ex
    from deep_cbrs_amar_renaissance_b200.scoring import ItemLists
    from tests.test_zz_gpu_experiment import write_inputs
    cfg, _, paths = write_inputs(tmp_path / "data")
    config = ex.load_yaml(cfg)
    config["model"].update(name="hybrid.HybridBertGCN", dense_units=[[16, 16], [16, 8], [64, 64]], clf_units=[64, 64])
    config["dataset"]["load_function_name"] = "load_user_item_graph_bert_embeddings"
    config["catalog_metrics"] = True
    e = ex.Experimenter(config, str(tmp_path / "runs"))
    e.run()
    assert len(spy) == 1
    users, items = e.trainset.users, e.trainset.items
    seen = ItemLists.from_ratings(e.trainset.ratings, len(users), len(items), device="cuda")
    ids, _ = e.model.recommend_top_k(len(users), len(items), 10, precision="fp32", exclude=seen)
    ids = ids.cpu().numpy()
    test = np.loadtxt(paths["test_ratings_filepath"], dtype=np.int64, delimiter="\t")[:, :3]   # original ids
    for k in (5, 10):
        want = _rival(test, ids, np.asarray(users), np.asarray(items), k)
        got = [e.metrics["catalog_%s_at_%d" % (m, k)] for m in ("precision", "recall", "f1")]
        assert np.allclose(got, want, rtol=0, atol=1e-12), (k, got, want)
