"""GPU parity for the chained tensor-core catalog scorer of the feature-based hybrid model
(cbrs_score_hybrid_topk_bf16; /root/reference/src/models/hybrid.py:72-89 applied to every (user, item) pair).

Oracle: the same network in numpy with every MMA operand rounded to bf16 where the kernel rounds it (h1, h2, x1, x2, g and
all weight matrices) and float64 sums.  The kernel's fp32 accumulation order inside an MMA is unspecified and an
activation that lands within an fp32 ulp of a bf16 rounding boundary may round the other way, which moves a score by up
to one bf16 ulp of an intermediate: tolerance 2e-3 on the (sigmoid) scores, ids compared where the oracle's gaps exceed
it; and the result must stay within 3e-2 of the exact fp32 scorer."""
import numpy as np
import pytest
import torch

from oracle import graph as og
from oracle import layers as ol
from tests.helpers import assert_topk_equivalent, export_weights, hybrid_bf16_scores, hybrid_tables, random_bipartite

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def dev():
    from deep_cbrs_amar_renaissance_b200 import ops
    ops.check_device()
    return torch.device("cuda", 0)


def _t(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


@pytest.mark.parametrize("n_users,n_items,k", [(37, 1000, 10), (5, 7, 5), (130, 333, 20), (16, 32, 3), (1, 2049, 10),
                                               (4800, 40, 5)])   # 4800 users: 24 users per CTA (one wave of 2 CTAs per SM)
def test_chained_hybrid_scorer_matches_bf16_oracle(dev, n_users, n_items, k):
    from deep_cbrs_amar_renaissance_b200 import ops
    (P1, Q1, P2, Q2), w = hybrid_tables(n_users, n_items, n_users + n_items)
    ids, vals = ops.score_hybrid_topk_bf16(_t(P1, dev), _t(Q1, dev), _t(P2, dev), _t(Q2, dev), _t(w["w3a2"], dev),
                                           _t(w["b3a2"], dev), _t(w["w3b2"], dev), _t(w["b3b2"], dev), _t(w["wc1"], dev),
                                           _t(w["bc1"], dev), _t(w["wc2"], dev), _t(w["bc2"], dev), _t(w["wc3"], dev),
                                           _t(w["bc3"], dev), k)
    ids_np, vals_np = ids.cpu().numpy(), vals.cpu().numpy()
    kk = min(k, n_items)
    assert (ids_np >= 0).all() and (ids_np < n_items).all()
    assert all(len(set(row)) == kk for row in ids_np[:, :kk])          # no item twice
    assert (np.diff(vals_np[:, :kk], axis=1) <= 0).all()                 # descending
    assert_topk_equivalent(ids_np[:, :kk], vals_np[:, :kk], hybrid_bf16_scores(P1, Q1, P2, Q2, w), kk, tol=2e-3)
    exact = hybrid_bf16_scores(P1, Q1, P2, Q2, w, rounded=False)
    got_exact = np.take_along_axis(exact, ids_np[:, :kk].astype(np.int64), axis=1)
    assert np.abs(got_exact - vals_np[:, :kk]).max() < 3e-2


def test_exact_ties_go_to_the_lower_item(dev):
    from deep_cbrs_amar_renaissance_b200 import ops
    n_users, n_items, c, k = 20, 300, 64, 12
    z = lambda *s: torch.zeros(*s, device=dev)
    ids, vals = ops.score_hybrid_topk_bf16(z(n_users, c), z(n_items, c), z(n_users, c), z(n_items, c), z(c, c), z(c), z(c, c),
                                           z(c), z(2 * c, c), z(c), z(c, c), z(c), z(c), z(1), k)
    assert (ids.cpu().numpy() == np.arange(k)[None, :]).all() and (vals == 0.5).all()


def test_hybrid_model_catalog_top_k_on_the_tensor_cores():
    """HybridBertGCN, feature-based, econfigs/hybrid-gnn.yaml grid2 shapes: recommend_top_k(precision='bf16') takes the
    chained kernel; against the fp32 oracle of the whole model (hybrid.py:72-89) within the bf16 distance, and against
    the blocked pair pipeline running the same layers through cbrs_dense_tc."""
    from deep_cbrs_amar_renaissance_b200 import scoring
    from tests.test_gpu_models import _build, _randomise
    n_users, n_items, dim, k = 70, 400, 768, 10
    adj = random_bipartite(n_users, n_items, 5000, seed=28)
    bert = (np.random.RandomState(5).standard_normal((n_users + n_items, dim)) * 0.5).astype(np.float32)
    grid = (16, [16, 16], [[48, 48], [256, 64], [64, 64]], [64, 64])
    model = _build("HybridBertGCN", adj, grid, module="hybrid", feature_based=True, fusion_method="concatenate", residual=False)
    model.set_content_table(bert)
    model((np.array([0]), np.array([n_users])))
    _randomise(model, 3)
    model.cache_propagation = True
    emb_dev = model.propagate()
    users = torch.arange(n_users, device="cuda")
    items = torch.arange(n_users, n_users + n_items, device="cuda")
    assert scoring._fused_hybrid_feature(model, emb_dev, users, items, k) is not None
    ids, vals = model.recommend_top_k(n_users, n_items, k, precision="bf16")
    w = export_weights(model)
    emb = ol.propagate("gcn", w["embeddings"], og.gcn_filter(adj), w["layers"])
    uu = np.repeat(np.arange(n_users), n_items)
    ii = np.tile(np.arange(n_items), n_users) + n_users
    exact = ol.hybrid_cbrs(emb, uu, ii, bert[uu], bert[ii], w, feature_based=True).reshape(n_users, n_items)
    ids_np, vals_np = ids.cpu().numpy(), vals.cpu().numpy()
    got_exact = np.take_along_axis(exact, ids_np.astype(np.int64), axis=1)
    assert np.abs(got_exact - vals_np).max() < 3e-2
    # the k-th best exact score is not far below what the kernel returned at rank k (a wrong list would be)
    kth = -np.sort(-exact, axis=1)[:, k - 1]
    assert (got_exact.min(axis=1) >= kth - 3e-2).all()
    model.set_scorer_precision("bf16")
    ids_g, vals_g = model.recommend_top_k(n_users, n_items, k, fused=False)
    assert np.abs(np.sort(vals_g.cpu().numpy(), axis=1) - np.sort(vals_np, axis=1)).max() < 2e-2
    # fp32 precision keeps the fp32 path (no silent downgrade)
    model.set_scorer_precision("fp32")
    ids32, vals32 = model.recommend_top_k(n_users, n_items, k, precision="fp32")
    assert assert_topk_equivalent(ids32.cpu().numpy(), vals32.cpu().numpy(), exact, k, tol=2e-5) > 0.5
