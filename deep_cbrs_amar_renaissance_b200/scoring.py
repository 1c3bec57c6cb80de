"""Full-catalog scoring + per-user top-k (scope row T, catalog form).

The reference only ranks the test pairs (/root/reference/src/experiment.py:197-207);
scoring every (user, item) is the new capability the north star asks for.  Work that
depends on one entity only (the towers of BasicRS / HybridCBRS, src/models/basic.py:33-34,
src/models/hybrid.py:74-77) is hoisted and computed once per user / item; the pairwise
part runs over blocks of users x all items, the tower rows being gathered inside the
first pairwise Dense kernel, and each block's [UB, I] scores go through cbrs_topk_rows.
Users are independent => sharded across ranks with no collective (SURVEY 8e).

Every path takes per-user exclusion lists (ItemLists, typically the items a user rated in training): they are kept out
of that user's top-k, inside the fused kernels or on the generic path's score blocks (cbrs_exclude_cols).
"""
import numpy as np
import torch

from . import ops

_PAIR_BUDGET = 1 << 18  # pairs per block: keeps a block's 64-wide activations L2-resident


class ItemLists:
    """Per-user lists of catalog items, CSR over GLOBAL user ids: user u's items are items[rowptr[u]:rowptr[u + 1]],
    sorted ascending, as catalog indices in [0, n_items) (item node id - n_users).  Passed as `exclude=` to
    catalog_top_k / recommend_top_k, which keep those items out of the user's top-k."""

    def __init__(self, rowptr, items, n_items):
        if not (torch.is_tensor(rowptr) and rowptr.dim() == 1 and rowptr.dtype == torch.int64 and rowptr.numel() >= 1):
            raise ValueError("ItemLists: rowptr must be a 1-D int64 tensor of n_users + 1 offsets")
        if not (torch.is_tensor(items) and items.dim() == 1 and items.dtype == torch.int32):
            raise ValueError("ItemLists: items must be a 1-D int32 tensor")
        if int(rowptr[0]) != 0 or int(rowptr[-1]) != items.numel():
            raise ValueError("ItemLists: rowptr must run from 0 to len(items) = {}, got {} .. {}".format(
                items.numel(), int(rowptr[0]), int(rowptr[-1])))
        self.rowptr, self.items, self.n_items = rowptr.contiguous(), items.contiguous(), int(n_items)

    @property
    def n_users(self):
        return self.rowptr.numel() - 1

    @classmethod
    def from_ratings(cls, ratings, n_users, n_items, device=None, min_rating=None, distinct=False):
        """Items per user from the [R, >= 2] ratings format of a dataset (`trainset.ratings`, `testset.ratings`): column
        0 the user index, column 1 the item index offset by n_users, column 2 the rating.  Built on `device` (default:
        the tensor's own device, or CUDA for a numpy array when one is present).
        Defaults (the seen items of a training set): every row counts, whatever its rating: a rated item is a seen
        item; a pair rated twice is listed twice.
        min_rating: keep only the rows whose rating is >= min_rating (needs column 2).  distinct: one entry per
        (user, item).  `min_rating=1, distinct=True` on test ratings gives the relevance sets of
        utilities.metrics.precision_recall_f1_at_k, the input of catalog_ranking_metrics."""
        arr = None if torch.is_tensor(ratings) else np.asarray(ratings)
        r = ratings if arr is None else torch.as_tensor(arr[:, :2].astype(np.int64))
        if device is None:
            device = r.device if arr is None else ("cuda" if torch.cuda.is_available() else "cpu")
        if r.dim() != 2 or r.shape[1] < 2:
            raise ValueError("ItemLists.from_ratings: expected a [R, >= 2] ratings array")
        if min_rating is not None:
            if (ratings if arr is None else arr).shape[1] < 3:
                raise ValueError("ItemLists.from_ratings: min_rating needs a rating column (column 2)")
            rating = ratings[:, 2] if arr is None else torch.as_tensor(arr[:, 2].astype(np.float64))
            r = r[rating >= min_rating]
        r = r[:, :2].to(device=device, dtype=torch.int64)
        user, item = r[:, 0], r[:, 1] - n_users
        if r.shape[0] and (bool((user < 0).any()) or bool((user >= n_users).any()) or bool((item < 0).any())
                           or bool((item >= n_items).any())):
            raise ValueError("ItemLists.from_ratings: user ids must lie in [0, {}) and item ids in [{}, {})".format(
                n_users, n_users, n_users + n_items))
        key = torch.unique(user * n_items + item) if distinct else torch.sort(user * n_items + item).values
        counts = torch.bincount(key // n_items, minlength=n_users)
        rowptr = torch.zeros(n_users + 1, dtype=torch.int64, device=device)
        torch.cumsum(counts, 0, out=rowptr[1:])
        return cls(rowptr, (key % n_items).to(torch.int32), n_items)


def _exclusion_rows(exclude, n_users, n_items, users, all_users):
    """(rowptr, items) whose row r is the list of the r-th scored user, or None.  The whole user range uses the lists
    as they are, a contiguous range a view of rowptr (offsets are absolute), any other subset gathers its sub-lists."""
    if exclude is None:
        return None
    if not isinstance(exclude, ItemLists):
        raise TypeError("exclude must be an ItemLists")
    if exclude.n_users != n_users or exclude.n_items != n_items:
        raise ValueError("exclude holds lists for {} users x {} items, the catalog is {} x {}".format(
            exclude.n_users, exclude.n_items, n_users, n_items))
    rowptr, items = exclude.rowptr.to(users.device), exclude.items.to(users.device)
    n = users.numel()
    if all_users or n == 0:
        return rowptr, items
    if bool((users < 0).any()) or bool((users >= n_users).any()):
        raise ValueError("users must lie in [0, {})".format(n_users))
    u0 = int(users[0])
    if bool(torch.equal(users, torch.arange(u0, u0 + n, device=users.device))):
        return rowptr[u0:u0 + n + 1], items
    begin, counts = rowptr[users], rowptr[users + 1] - rowptr[users]
    sub = torch.zeros(n + 1, dtype=torch.int64, device=users.device)
    torch.cumsum(counts, 0, out=sub[1:])
    pos = torch.arange(int(sub[-1]), device=users.device) - torch.repeat_interleave(sub[:-1] - begin, counts)
    return sub, items[pos]


def _blocks(n_users, n_items, user_block=None, budget=_PAIR_BUDGET):
    """(users per block, items per block): a block never exceeds `budget` pairs.  Catalogs wider than the budget are
    cut along the ITEM axis too (the per-user top-k is then merged across item blocks), so no path degenerates into
    one user per Python iteration however large the catalog is."""
    ib = min(n_items, budget)
    ub = user_block or max(1, budget // ib)
    return min(ub, max(n_users, 1)), ib


def _block_indices(cache, ub, n_items, device):
    key = (ub, n_items)
    if key not in cache:
        pu = torch.arange(ub, device=device, dtype=torch.int64).repeat_interleave(n_items)
        pi = torch.arange(n_items, device=device, dtype=torch.int64).repeat(ub)
        cache[key] = (pu, pi)
    return cache[key]


def _pair_scorer(model, emb, user_nodes, item_nodes):
    """Returns f(pu, pi) -> scores [len(pu), 1]; pu / pi index the hoisted per-entity tables."""
    rs = model.rs
    if hasattr(rs, "unet"):  # BasicRS
        if rs.unet.layers:
            ut = rs.unet.call_sources([(emb, user_nodes)])
            it = rs.inet.call_sources([(emb, item_nodes)])
            return lambda pu, pi: rs.clf.call_sources([(ut, pu), (it, pi)])
        return lambda pu, pi: rs.clf.call_sources([(emb, user_nodes[pu]), (emb, item_nodes[pi])])
    # HybridCBRS
    table = model.content_table
    if table is None:
        raise ValueError("catalog scoring of a hybrid model needs set_content_table(...)")
    ug = rs.dense1a.call_sources([(emb, user_nodes)])
    ig = rs.dense1b.call_sources([(emb, item_nodes)])
    ub = rs.dense2a.call_sources([(table, user_nodes)])
    ib = rs.dense2b.call_sources([(table, item_nodes)])
    plain = rs.residual is None and all(f.method == 'concatenate' for f in (rs.fuse1a, rs.fuse1b, rs.fuse2))
    if rs.feature_based or not plain:
        return lambda pu, pi: rs.tail((ug, pu), (ig, pi), (ub, pu), (ib, pi))
    # entity-based, plain: dense3a / dense3b depend on one entity each and are hoisted too
    x1 = rs.dense3a.call_sources([(ug, None), (ub, None)])
    x2 = rs.dense3b.call_sources([(ig, None), (ib, None)])
    return lambda pu, pi: rs.clf.call_sources([(x1, pu), (x2, pi)])


def catalog_scores(model, emb, n_users, n_items, users=None):
    """Dense [U, n_items] score matrix (tests / small catalogs only)."""
    dev = emb.device
    users = torch.arange(n_users, device=dev, dtype=torch.int64) if users is None else users.to(dev, torch.int64)
    items = torch.arange(n_users, n_users + n_items, device=dev, dtype=torch.int64)
    score = _pair_scorer(model, emb, users, items)
    cache = {}
    ub, ib = _blocks(users.numel(), n_items)
    out = torch.empty(users.numel(), n_items, dtype=torch.float32, device=dev)
    for u0 in range(0, users.numel(), ub):
        nb = min(ub, users.numel() - u0)
        for i0 in range(0, n_items, ib):
            ni = min(ib, n_items - i0)
            pu, pi = _block_indices(cache, nb, ni, dev)
            out[u0:u0 + nb, i0:i0 + ni] = score(pu + u0, pi + i0).reshape(nb, ni)
    return out


def _hoisted_sources(model, emb, users, items):
    """(user source, item source, classifier) when the scorer is `clf([f(user) || g(item)])` with f, g depending on one
    entity each - BasicRS (src/models/basic.py:31-37) and the entity-based HybridCBRS with plain concatenation
    (src/models/hybrid.py:83-89: dense3a sees the user's two embeddings only, dense3b the item's) - else None."""
    rs = model.rs
    if hasattr(rs, "unet"):  # BasicRS
        if rs.unet.layers:
            return (rs.unet.call_sources([(emb, users)]), None), (rs.inet.call_sources([(emb, items)]), None), rs.clf
        return (emb, users), (emb, items), rs.clf
    plain = rs.residual is None and all(f.method == 'concatenate' for f in (rs.fuse1a, rs.fuse1b, rs.fuse2))
    if rs.feature_based or not plain or model.content_table is None:
        return None
    table = model.content_table
    ug = rs.dense1a.call_sources([(emb, users)])
    ig = rs.dense1b.call_sources([(emb, items)])
    ub = rs.dense2a.call_sources([(table, users)])
    ib = rs.dense2b.call_sources([(table, items)])
    x1 = rs.dense3a.call_sources([(ug, None), (ub, None)])
    x2 = rs.dense3b.call_sources([(ig, None), (ib, None)])
    return (x1, None), (x2, None), rs.clf


def _fused_basic(model, emb, users, items, k, precision="fp32", exclude=None):
    """Scorers of the form clf([f(user) || g(item)]) with two hidden classifier layers -> the fused kernel
    (cbrs_score_catalog_topk: hoisted first layer, second layer, output, sigmoid and running top-k in one pass)."""
    clf = model.rs.clf
    if len(clf.layers) != 3 or k > 128:
        return None
    l1, l2, l3 = clf.layers
    if l1.activation != "relu" or l2.activation != "relu" or l3.units != 1:
        return None
    if l1.units % 8 or l1.units > 256 or l2.units > 128:
        return None
    src = _hoisted_sources(model, emb, users, items)
    if src is None:
        return None
    u_src, i_src, _ = src
    du = u_src[0].shape[1]
    l1.build_for(du + i_src[0].shape[1])
    l2.build_for(l1.units)
    l3.build_for(l2.units)
    P = ops.dense(u_src[0], l1.kernel[:du], l1.bias, None, idx1=u_src[1])   # bias folded into the user half
    Q = ops.dense(i_src[0], l1.kernel[du:], None, None, idx1=i_src[1])
    return ops.score_catalog_topk(P, Q, l2.kernel, l2.bias, l3.kernel.reshape(-1), l3.bias, k, precision, exclude)


def _fused_hybrid_feature(model, emb, users, items, k, exclude=None, precision="bf16"):
    """Feature-based HybridCBRS with the shapes of every hybrid grid of the reference (dense3a / dense3b = two 64-wide
    layers, classifier 64 -> 64 -> 1, relu, plain concatenation) -> a chained tensor-core kernel: precision 'bf16'
    cbrs_score_hybrid_topk_bf16 (bf16 operands), 'fp32' cbrs_score_hybrid_topk_tf32x3 (3xTF32, fp32 accuracy).  None
    when the scorer has another shape, the precision has no such kernel or k exceeds the catalog."""
    rs = model.rs
    if hasattr(rs, "unet") or not rs.feature_based or rs.residual is not None or model.content_table is None or k > 128:
        return None
    if precision not in ("bf16", "fp32") or k > items.numel():   # both chained kernels refuse k > n_items
        return None
    if any(f.method != 'concatenate' for f in (rs.fuse1a, rs.fuse1b, rs.fuse2)):
        return None
    d3a, d3b, clf = rs.dense3a.layers, rs.dense3b.layers, rs.clf.layers
    if len(d3a) != 2 or len(d3b) != 2 or len(clf) != 3 or clf[2].units != 1:
        return None
    if any(ly.units != 64 or ly.activation != "relu" for ly in (*d3a, *d3b, clf[0], clf[1])):
        return None
    table = model.content_table
    ug = rs.dense1a.call_sources([(emb, users)])
    ig = rs.dense1b.call_sources([(emb, items)])
    ub = rs.dense2a.call_sources([(table, users)])
    ib = rs.dense2b.call_sources([(table, items)])
    g, c = ug.shape[1], ub.shape[1]
    d3a[0].build_for(g + ig.shape[1]); d3a[1].build_for(64)
    d3b[0].build_for(c + ib.shape[1]); d3b[1].build_for(64)
    clf[0].build_for(128); clf[1].build_for(64); clf[2].build_for(64)
    P1 = ops.dense(ug, d3a[0].kernel[:g], d3a[0].bias, None)     # bias folded into the user half
    Q1 = ops.dense(ig, d3a[0].kernel[g:], None, None)
    P2 = ops.dense(ub, d3b[0].kernel[:c], d3b[0].bias, None)
    Q2 = ops.dense(ib, d3b[0].kernel[c:], None, None)
    kernel = ops.score_hybrid_topk_bf16 if precision == "bf16" else ops.score_hybrid_topk_tf32x3
    return kernel(P1, Q1, P2, Q2, d3a[1].kernel, d3a[1].bias, d3b[1].kernel, d3b[1].bias, clf[0].kernel, clf[0].bias,
                  clf[1].kernel, clf[1].bias, clf[2].kernel.reshape(-1), clf[2].bias, k, exclude)


def catalog_top_k(model, emb, n_users, n_items, k=10, users=None, user_block=None, fused=True, precision="fp32",
                  exclude=None):
    """exclude: an ItemLists over all n_users; each user's listed items are kept out of its top-k (slots past the number
    of eligible items hold -1 / -inf)."""
    dev = emb.device
    all_users = users is None
    users = torch.arange(n_users, device=dev, dtype=torch.int64) if users is None else users.to(dev, torch.int64)
    items = torch.arange(n_users, n_users + n_items, device=dev, dtype=torch.int64)
    excl = _exclusion_rows(exclude, n_users, n_items, users, all_users)
    if fused:
        out = _fused_basic(model, emb, users, items, k, precision, excl)
        if out is None and precision in ("bf16", "fp32"):   # 'fp32-ffma' keeps the generic path for hybrids
            out = _fused_hybrid_feature(model, emb, users, items, k, excl, precision)
        if out is not None:
            return out
    score = _pair_scorer(model, emb, users, items)
    cache = {}
    ub, ib = _blocks(users.numel(), n_items, user_block)
    # slots past the catalog (k > n_items) keep -1 / -inf, as the fused kernels write them
    ids = torch.full((users.numel(), k), -1, dtype=torch.int32, device=dev)
    vals = torch.full((users.numel(), k), -float("inf"), dtype=torch.float32, device=dev)
    for u0 in range(0, users.numel(), ub):
        nb = min(ub, users.numel() - u0)
        best_i = best_v = None
        for i0 in range(0, n_items, ib):
            ni = min(ib, n_items - i0)
            pu, pi = _block_indices(cache, nb, ni, dev)
            s = score(pu + u0, pi + i0).reshape(nb, ni)
            if excl is not None:   # scores are sigmoid outputs: -inf marks an excluded item and nothing else
                ops.exclude_cols(s, i0, (excl[0][u0:], excl[1]))
            bi, bv = ops.topk_rows(s, min(k, ni))
            bi = bi + i0
            if best_i is None:
                best_i, best_v = bi, bv
                continue
            # merge with the best of the earlier (lower-id) item blocks: candidates stay ordered by (score desc, id asc)
            # inside each part and the earlier part comes first, so cbrs_topk_rows' rule "ties go to the lower column"
            # is still "ties go to the lower item id"
            cand_v = torch.cat([best_v, bv], dim=1).contiguous()
            cand_i = torch.cat([best_i, bi], dim=1)
            sel, best_v = ops.topk_rows(cand_v, min(k, cand_v.shape[1]))
            best_i = torch.gather(cand_i, 1, sel.long())
        if excl is not None:
            best_i = torch.where(torch.isneginf(best_v), torch.full_like(best_i, -1), best_i)
        ids[u0:u0 + nb, :best_i.shape[1]], vals[u0:u0 + nb, :best_v.shape[1]] = best_i, best_v
    return ids, vals
