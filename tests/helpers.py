"""Shared test inputs: seeded graphs, weights, and tolerant comparisons."""
import numpy as np
from scipy import sparse

from oracle import layers as ol

RTOL = 1e-5  # north star: embeddings and scores within 1e-5 relative (fp32)


def random_bipartite(n_users, n_items, n_pos, seed=0, n_props=0, n_links=0, dup_links=0):
    """Symmetrised COO adjacency in the reference's entry order (+ optional property links with duplicates)."""
    rng = np.random.RandomState(seed)
    keys = np.unique(rng.randint(0, n_users * n_items, size=n_pos))
    rng.shuffle(keys)
    r, c = keys // n_items, keys % n_items + n_users
    n = n_users + n_items + n_props
    if n_props:
        ii = rng.randint(0, n_items, size=n_links) + n_users
        pp = rng.randint(0, n_props, size=n_links) + n_users + n_items
        pick = rng.randint(0, n_links, size=dup_links)
        r = np.concatenate([r, ii, ii[pick]])
        c = np.concatenate([c, pp, pp[pick]])
    rows = np.concatenate([r, c]).astype(np.int32)
    cols = np.concatenate([c, r]).astype(np.int32)
    return sparse.coo_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=(n, n), dtype=np.float32)


def glorot(rng, shape):
    lim = np.sqrt(6.0 / (shape[-2] + shape[-1])) if len(shape) > 1 else np.sqrt(3.0 / shape[0])
    return rng.uniform(-lim, lim, size=shape).astype(np.float32)


def assert_close(got, want, rtol=RTOL, atol=None, what=""):
    """max |got-want| <= rtol * max|want| (relative to the tensor scale) unless atol is given."""
    got = np.asarray(got, dtype=np.float64)
    want = np.asarray(want, dtype=np.float64)
    assert got.shape == want.shape, "{}: shape {} vs {}".format(what, got.shape, want.shape)
    scale = max(np.abs(want).max(), 1e-30) if want.size else 1.0
    tol = atol if atol is not None else rtol * scale
    err = np.abs(got - want).max() if want.size else 0.0
    assert err <= tol, "{}: max abs err {:.3e} > {:.3e} (scale {:.3e})".format(what, err, tol, scale)


def assert_topk_equivalent(ids, vals, oracle_scores, k, tol=2e-6):
    """ids must be bit-identical to the oracle's stable top-k wherever the oracle's score gaps
    exceed `tol`; inside a near-tie (fp32 exp differs by an ulp between CPU and GPU) the returned
    item must still carry an oracle score within tol of the oracle's item at that rank."""
    s = np.asarray(oracle_scores, np.float64)
    order = np.argsort(-s, axis=1, kind="stable")[:, :k]
    ref_vals = np.take_along_axis(s, order, axis=1)
    ids = np.asarray(ids)
    got_vals = np.take_along_axis(s, ids.astype(np.int64), axis=1)
    assert np.abs(got_vals - ref_vals).max() <= tol, "top-k scores differ beyond tolerance"
    assert np.abs(np.asarray(vals, np.float64) - got_vals).max() <= max(tol, 1e-5), "returned scores differ from the oracle's"
    sorted_s = -np.sort(-s, axis=1)[:, :k + 1]
    if sorted_s.shape[1] < k + 1:  # k == catalog size: nothing ranks below the last slot
        sorted_s = np.concatenate([sorted_s, np.full((len(s), 1), -np.inf)], axis=1)
    gaps = sorted_s[:, :-1] - sorted_s[:, 1:]
    prev_gap = np.concatenate([np.full((len(s), 1), np.inf), gaps[:, :-1]], axis=1)
    clear = (gaps > tol) & (prev_gap > tol)
    assert (ids[clear] == order[clear]).all(), "top-k ids differ where the ranking is unambiguous"
    return float(clear.mean()) if clear.size else 1.0


# ------------------------------------------------------------------ catalog scorer oracles
def bf16_round(x):
    """round-to-nearest-even fp32 -> bf16 -> fp32 (numpy)"""
    u = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) & 0xFFFF0000
    return u.astype(np.uint32).view(np.float32)


def tf32_round(x):
    """round to the nearest tf32 (10 explicit mantissa bits), ties away from zero as cvt.rna"""
    b = np.asarray(x, np.float32).view(np.uint32).astype(np.uint64)
    return ((b + 0x1000) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def _user_blocks(n_users, n_items, pairs=1 << 17):
    step = max(1, pairs // max(n_items, 1))
    return [(u0, min(u0 + step, n_users)) for u0 in range(0, n_users, step)]


def basic_chain(P, Q, w2, b2, w3, b3):
    """The fused BasicRS scorer (cbrs_score_catalog_topk*) in float64: sigmoid(relu(relu(P[u] + Q[i]) W2 + b2) w3 + b3)
    for every (user, item) -> [U, I]"""
    f8 = np.float64
    out = np.empty((len(P), len(Q)))
    for u0, u1 in _user_blocks(len(P), len(Q)):
        h1 = np.maximum(P[u0:u1, None, :].astype(f8) + Q[None, :, :], 0)
        h2 = np.maximum(h1 @ w2.astype(f8) + b2, 0)
        out[u0:u1] = 1.0 / (1.0 + np.exp(-(h2 @ w3.astype(f8) + f8(b3[0]))))
    return out


def bf16_basic_chain(P, Q, w2, b2, w3, b3):
    """The bf16 catalog scorer (cbrs_score_catalog_topk_bf16) with its operands rounded where each kernel variant rounds
    them, sums in float64 -> [U, I].  Tolerances of the kernels against it: 1e-4 for v3 (c1 <= 64, c2 <= 64: an
    activation within an fp32 ulp of a bf16 rounding boundary may round the other way before the output product),
    2e-5 for v2 / v1 (fp32 summation order inside the MMA is unspecified)."""
    c1, c2 = w2.shape
    f8 = np.float64
    out = np.empty((len(P), len(Q)), np.float32)
    for u0, u1 in _user_blocks(len(P), len(Q)):
        nu = u1 - u0
        if c1 <= 64 and c2 <= 128:  # v2 / v3: P and Q rounded first, bf16 add (exact sum rounded once), relu
            h1 = bf16_round(bf16_round(P[u0:u1])[:, None, :] + bf16_round(Q)[None, :, :])
            h1 = np.maximum(h1, 0).reshape(-1, c1)
        else:                       # v1
            h1 = bf16_round(np.maximum(P[u0:u1, None, :] + Q[None, :, :], 0).reshape(-1, c1))
        if c1 <= 64 and c2 <= 64:
            # v3 (every product on the tensor core): the bias is a row of the bf16 image of W2, relu(h1 W2 + b2) is
            # rounded to bf16 and the output layer is a second product against bf16(w3)
            acc = h1.astype(f8) @ bf16_round(w2).astype(f8) + bf16_round(b2).astype(f8)
            h2 = bf16_round(np.maximum(acc, 0).astype(np.float32))
            s = ol.sigmoid((h2.astype(f8) @ bf16_round(w3).astype(f8)).astype(np.float32) + b3)
        else:
            h2 = np.maximum(h1.astype(f8) @ bf16_round(w2).astype(f8) + b2, 0).astype(np.float32)
            s = ol.sigmoid((h2.astype(f8) @ w3.astype(f8)).astype(np.float32) + b3)
        out[u0:u1] = s.reshape(nu, len(Q))
    return out


HYBRID_WEIGHTS = ("w3a2", "b3a2", "w3b2", "b3b2", "wc1", "bc1", "wc2", "bc2", "wc3", "bc3")   # argument order


def hybrid_tables(n_users, n_items, seed):
    """Seeded operands of the chained hybrid scorers: tables (P1, Q1, P2, Q2) [*, 64] and the weights by name"""
    rng = np.random.RandomState(seed)
    c = 64
    P1, P2 = (rng.standard_normal((n_users, c)).astype(np.float32) for _ in range(2))
    Q1, Q2 = (rng.standard_normal((n_items, c)).astype(np.float32) for _ in range(2))
    w = dict(w3a2=glorot(rng, (c, c)), w3b2=glorot(rng, (c, c)), wc1=glorot(rng, (2 * c, c)), wc2=glorot(rng, (c, c)),
             wc3=glorot(rng, (c, 1)).reshape(-1), bc3=np.array([0.05], np.float32))
    for b in ("b3a2", "b3b2", "bc1", "bc2"):
        w[b] = (rng.standard_normal(c) * 0.1).astype(np.float32)
    return (P1, Q1, P2, Q2), w


def hybrid_chain(P1, Q1, P2, Q2, w, uu, ii, rounded=False):
    """The chained hybrid scorer in float64: sigmoid scores of the pairs (uu[j], ii[j]); rounded: every product operand
    rounded to tf32 (a single-TF32 evaluation)"""
    f8 = np.float64
    r = (lambda x: tf32_round(x).astype(f8)) if rounded else (lambda x: np.asarray(x, f8))
    relu = lambda x: np.maximum(x, 0)
    h1 = relu(P1[uu].astype(f8) + Q1[ii])
    h2 = relu(P2[uu].astype(f8) + Q2[ii])
    x1 = relu(r(h1) @ r(w["w3a2"]) + w["b3a2"])
    x2 = relu(r(h2) @ r(w["w3b2"]) + w["b3b2"])
    g = relu(r(x1) @ r(w["wc1"][:64]) + r(x2) @ r(w["wc1"][64:]) + w["bc1"])
    h = relu(r(g) @ r(w["wc2"]) + w["bc2"])
    return 1.0 / (1.0 + np.exp(-(h @ w["wc3"].astype(f8) + f8(w["bc3"][0]))))


def hybrid_chain_scores(tabs, w):
    """hybrid_chain over every (user, item) -> [U, I] float64"""
    n_users, n_items = len(tabs[0]), len(tabs[1])
    out = np.empty((n_users, n_items))
    for u0, u1 in _user_blocks(n_users, n_items):
        uu, ii = np.repeat(np.arange(u0, u1), n_items), np.tile(np.arange(n_items), u1 - u0)
        out[u0:u1] = hybrid_chain(*tabs, w, uu, ii).reshape(u1 - u0, n_items)
    return out


def hybrid_bf16_scores(P1, Q1, P2, Q2, w, rounded=True):
    """The chained bf16 hybrid scorer (cbrs_score_hybrid_topk_bf16): every MMA operand rounded to bf16 where the kernel
    rounds it (h1, h2, x1, x2, g and all weight matrices), float64 sums -> [U, I].  rounded=False: the exact fp32 chain."""
    r = bf16_round if rounded else (lambda x: np.asarray(x, np.float32))
    f8 = np.float64
    out = np.empty((len(P1), len(Q1)), np.float32)

    def layer(x, k, b):
        return np.maximum(r(x).astype(f8) @ r(k).astype(f8) + b, 0).astype(np.float32)

    for u0, u1 in _user_blocks(len(P1), len(Q1)):
        pairs = lambda P, Q: np.maximum(P[u0:u1, None, :] + Q[None, :, :], 0).reshape(-1, P.shape[1]).astype(np.float32)
        x1 = layer(pairs(P1, Q1), w["w3a2"], w["b3a2"])
        x2 = layer(pairs(P2, Q2), w["w3b2"], w["b3b2"])
        g = layer(np.concatenate([x1, x2], 1), w["wc1"], w["bc1"])
        h = layer(g, w["wc2"], w["bc2"])
        logit = (h.astype(f8) @ w["wc3"].astype(f8) + w["bc3"]).astype(np.float32)
        out[u0:u1] = ol.sigmoid(logit).reshape(u1 - u0, len(Q1))
    return out


def weights_struct(w, proj_first=None):
    """{product weight path: array} -> the numpy structures the oracle takes (Keras layouts: kernel [in,out]).
    proj_first: {fusion layer name: bool} for attention fusions that project."""
    w = dict(w)

    def stack(prefix):
        ks = sorted({int(n[len(prefix):].split("/")[0]) for n in w if n.startswith(prefix)})
        return [(w["%s%d/kernel" % (prefix, k)], w["%s%d/bias" % (prefix, k)]) for k in ks]

    out = dict(embeddings=w["gnn/gnn_layers/embeddings"], layers=[])
    k = 0
    while any(n.startswith("gnn/gnn_layers/seq_layers.%d/" % k) for n in w):
        pre = "gnn/gnn_layers/seq_layers.%d/" % k
        lw = {n[len(pre):]: v for n, v in w.items() if n.startswith(pre)}
        if "kernel" in lw and lw["kernel"].ndim == 3:  # GATConv stores [F,1,H]
            lw["kernel"] = lw["kernel"].reshape(lw["kernel"].shape[0], -1)
        if "attn_kernel_self" in lw:
            lw["attn_self"] = lw.pop("attn_kernel_self").reshape(-1)
            lw["attn_neigh"] = lw.pop("attn_kernel_neigh").reshape(-1)
        out["layers"].append(lw)
        k += 1
    if any(n.startswith("rs/unet/") or n.startswith("rs/inet/") for n in w) or not any(n.startswith("rs/dense1a/") for n in w):
        out.update(unet=stack("rs/unet/layers."), inet=stack("rs/inet/layers."), clf=stack("rs/clf/layers."))
    else:
        for name in ("dense1a", "dense1b", "dense2a", "dense2b", "dense3a", "dense3b", "clf"):
            out[name] = stack("rs/%s/layers." % name)
        if any(n.startswith("rs/residual/") for n in w):
            out["residual"] = stack("rs/residual/layers.")
        for name in ("fuse1a", "fuse1b", "fuse2"):
            if "rs/%s/att_weight" % name in w:
                out[name] = dict(att_weight=w["rs/%s/att_weight" % name], proj_weight=w.get("rs/%s/proj_weight" % name),
                                 proj_first=(proj_first or {}).get(name))
    return out


def export_weights(model):
    """Model weights as the numpy structures the oracle takes."""
    named = {n: w.detach().cpu().numpy() for n, w in model.named_weights()}
    pf = {name: getattr(model.rs, name).proj_first for name in ("fuse1a", "fuse1b", "fuse2")
          if hasattr(model.rs, name) and getattr(getattr(model.rs, name), "proj_first", None) is not None}
    out = weights_struct(named, pf)
    n_layers = len(model.gnn.gnn_layers.seq_layers)
    out["layers"] += [{} for _ in range(n_layers - len(out["layers"]))]  # weight-free LightGCN layers
    return out


def kg_graphs(n_users=40, n_items=30, n_props=25, n_pos=420, n_links=150, dup_links=12):
    """Seeded (user-item [U+I], item-property [I+P]) adjacencies in the layout of type_adjacency='unary-kg'
    (preprocess.py:113-145): both symmetrised, the second with `dup_links` repeated (item, property) links - the
    same pair under two predicates - which GCN-type layers sum and GraphSage / GAT keep as separate edges."""
    ui = random_bipartite(n_users, n_items, n_pos, seed=13)
    ip = random_bipartite(n_items, n_props, n_links, seed=5)
    half = ip.nnz // 2
    pick = np.random.RandomState(9).randint(0, half, size=dup_links)
    r = np.concatenate([ip.row[:half], ip.row[pick]])
    c = np.concatenate([ip.col[:half], ip.col[pick]])
    rows, cols = np.concatenate([r, c]).astype(np.int32), np.concatenate([c, r]).astype(np.int32)
    ip = sparse.coo_matrix((np.ones(len(rows), np.float32), (rows, cols)), shape=ip.shape, dtype=np.float32)
    return ui, ip


KG_GRAPHS = {"default": dict(), "sparse": dict(n_pos=120, n_links=40, dup_links=4)}  # tests/golden/make_golden_models_kg.py


KG_COMMON = dict(n_layers=2, embedding_dim=8, l2_regularizer=1e-4, aggregate="mean", dropout_rate=0.0,
                 final_node="concatenation", activation="relu")


def kg_model(case, graphs, n_users, n_items):
    """the constructor call of tests/golden/make_golden_models_kg.py on the product's classes"""
    from deep_cbrs_amar_renaissance_b200.models import basic, hybrid
    name = case.split("-")[0]
    kw = dict(KG_COMMON, n_hiddens=[8, 8])
    if name.startswith("Hybrid"):
        kw.update(dense_units=[[12, 12], [14, 6], [16, 16]], clf_units=[16, 16], feature_based=True)
    else:
        kw.update(dense_units=[12, 12], clf_units=[16, 16])
    if case.endswith("-itemconcat"):
        kw["item_node"] = "concatenation"
    if case.endswith("-uiconcat"):
        kw["user_item_node"] = "concatenation"
    if case.endswith("-mean"):
        kw.update(final_node="mean", aggregate="sum")
    adjs = graphs if "TW" in name else graphs[:2]
    return getattr(hybrid if name.startswith("Hybrid") else basic, name)(n_users, n_items, adjs, **kw), kw


def relation_blocks(a_hat, first_rel1_node):
    """The normalised adjacency split into the two relations of SURVEY row R by node range: an entry belongs to
    relation 1 when it touches a node >= first_rel1_node (item <-> property links), else to relation 0; self loops ride
    on relation 0 (the device build's self_rel).  Returns [A_0, A_1] as scipy CSR."""
    coo = a_hat.tocoo()
    is_r1 = (coo.row >= first_rel1_node) | (coo.col >= first_rel1_node)
    is_r1 = np.where(coo.row == coo.col, False, is_r1)
    return [sparse.csr_matrix((coo.data[pick], (coo.row[pick], coo.col[pick])), shape=coo.shape) for pick in (~is_r1, is_r1)]
