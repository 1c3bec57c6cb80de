"""Per-user top-k of an explicit pair list (mirror of
/root/reference/src/utilities/metrics.py:11-34).

The reference sorts a pandas frame by (users asc, scores desc) - a stable sort - and
keeps head(k) per user with an O(U) filter loop; here one stable device radix sort of
(user, ~score) keys does both.

`top_k_metrics` in the reference shells out to binaries/mimir.jar (Java; RiVal 0.2 Precision and
Recall at a cutoff, F1 from their means).  There is no JRE in this image, so the jar cannot run and
its numbers cannot be pinned; `precision_recall_f1_at_k` restates RiVal 0.2's published definitions
([3P], scope row (f)-2) and `top_k_metrics` walks the same directory layout and writes the same
results.tsv with it."""
import os

import numpy as np
import pandas as pd
import torch

from .. import ops


def top_k_predictions(predictions, users, items, k=5):
    """predictions [n,3] = (user idx, item idx offset by len(users), score).
    Returns a DataFrame(users, items, scores) with ORIGINAL ids, users ascending,
    scores descending, ties in input order."""
    predictions = np.asarray(predictions)
    dev = torch.device("cuda", torch.cuda.current_device())
    u = torch.from_numpy(np.ascontiguousarray(predictions[:, 0].astype(np.int64))).to(dev)
    s = torch.from_numpy(np.ascontiguousarray(predictions[:, 2].astype(np.float32))).to(dev)
    keep = ops.topk_pairs(u, s, len(users), k).cpu().numpy()
    df = pd.DataFrame()
    df['users'] = np.asarray(users)[predictions[keep, 0].astype(np.int64)]
    df['items'] = np.asarray(items)[predictions[keep, 1].astype(np.int64) - len(users)]
    df['scores'] = predictions[keep, 2]
    return df


def catalog_predictions(ids, vals, users, items):
    """Full-catalog top-k (recommend_top_k's ids / scores [U, k]) as the DataFrame(users, items, scores) frame
    top_k_predictions returns: ORIGINAL ids (row r is users[r], catalog index i is items[i]), rows in input order,
    each row's items by score descending.  Slots holding -1 (fewer eligible items than k) are dropped."""
    ids = ids.cpu().numpy() if torch.is_tensor(ids) else np.asarray(ids)
    vals = vals.cpu().numpy() if torch.is_tensor(vals) else np.asarray(vals)
    rows, cols = np.nonzero(ids >= 0)
    df = pd.DataFrame()
    df['users'] = np.asarray(users)[rows]
    df['items'] = np.asarray(items)[ids[rows, cols].astype(np.int64)]
    df['scores'] = vals[rows, cols]
    return df


def precision_recall_f1_at_k(test_ratings, predictions, k, relevance_threshold=1):
    """Precision@k, Recall@k and F1@k in the sense of RiVal 0.2 (the library inside mimir.jar):

    * a test item is relevant for a user when its rating >= relevance_threshold;
    * per user, the recommended list is the predictions sorted by score descending (ties in file order);
      tp = relevant items among the first k;  precision_u = tp / k  (RiVal divides by the cutoff even when
      fewer than k items were recommended);  recall_u = tp / #relevant(u);
    * users without a relevant test item are skipped (no ground truth), users without predictions count 0;
    * Precision and Recall are the means over the remaining users; F1 = 2PR / (P + R) of the means.

    test_ratings, predictions: arrays / frames with columns (user, item, rating | score), original ids.
    Returns dict(precision=, recall=, f1=, users=)."""
    t = np.asarray(test_ratings)
    p = np.asarray(predictions)
    rel = {}
    for u, i, r in zip(t[:, 0], t[:, 1], t[:, 2]):
        if r >= relevance_threshold:
            rel.setdefault(u, set()).add(i)
    order = np.lexsort((np.arange(len(p)), -p[:, 2].astype(np.float64), p[:, 0]))
    recs = {}
    for row in order:
        recs.setdefault(p[row, 0], []).append(p[row, 1])
    ps, rs = [], []
    for u, items in rel.items():
        top = recs.get(u, [])[:k]
        tp = sum(1 for i in top if i in items)
        ps.append(tp / float(k))
        rs.append(tp / float(len(items)))
    prec = float(np.mean(ps)) if ps else 0.0
    rec = float(np.mean(rs)) if rs else 0.0
    f1 = 2 * prec * rec / (prec + rec) if prec + rec > 0 else 0.0
    return dict(precision=prec, recall=rec, f1=f1, users=len(ps))


RANKING_METRICS = ("precision", "recall", "f1", "ndcg", "map", "hit_rate", "mrr")


def catalog_ranking_metrics(ids, relevant, users=None, cutoffs=(5, 10), metrics=RANKING_METRICS, per_user=False):
    """Full-ranking metrics of top-k lists at each cutoff, computed on the device (cbrs_rank_metrics): only the sums
    come back to the host.

    ids: CUDA int32 [n_rows, k], the lists of recommend_top_k (catalog indices, best first, -1 = empty slot); row r is
    user users[r] (users: int64 [n_rows], distinct), or user r when users is None.
    relevant: scoring.ItemLists over all users, e.g. ItemLists.from_ratings(testset.ratings, ..., min_rating=1,
    distinct=True).  Binary relevance; the definitions are those above cbrs_rank_metrics in include/cbrs_b200.h.

    As in precision_recall_f1_at_k (RiVal 0.2): every mean is over ALL users with at least one relevant item, those
    that were not scored counting 0; F1 = 2PR / (P + R) of the means.
    Returns {"<metric>_at_<c>": float} for each metric of `metrics` (names in RANKING_METRICS) and cutoff, "users": the
    number of users with a relevant item, and with per_user=True "per_user": fp64 [n_rows, n_cutoffs, 6] of the columns
    ops.RANK_METRICS per scored row (NaN for a row without relevant items) for paired comparisons."""
    from ..scoring import ItemLists
    metrics = tuple(metrics)
    unknown = [m for m in metrics if m not in RANKING_METRICS]
    if unknown:
        raise ValueError("unknown ranking metrics {}; known: {}".format(unknown, RANKING_METRICS))
    if not isinstance(relevant, ItemLists):
        raise TypeError("relevant must be an ItemLists")
    cutoffs = ops.rank_metrics_cutoffs(ids, cutoffs)
    rowptr, items = relevant.rowptr.to(ids.device), relevant.items.to(ids.device)
    sums, pu = ops.rank_metrics(ids, (rowptr, items), users, cutoffs, per_user=per_user, n_items=relevant.n_items)
    n_rel = int((rowptr[1:] > rowptr[:-1]).sum())
    sums = sums.cpu().numpy()
    out = {}
    for ci, c in enumerate(cutoffs):
        mean = {m: float(sums[ci, j]) / n_rel if n_rel else 0.0 for j, m in enumerate(ops.RANK_METRICS)}
        p, r = mean["precision"], mean["recall"]
        mean["f1"] = 2 * p * r / (p + r) if p + r > 0 else 0.0
        out.update({"{}_at_{}".format(m, c): mean[m] for m in metrics})
    out["users"] = n_rel
    if per_user:
        out["per_user"] = pu
    return out


def top_k_metrics(test_filepath, predictions_path, relevance_threshold=1, sep='\t'):
    """Same directory walk as the reference (metrics.py:37-80): every `top_<k>` directory holding
    predictions*.tsv gets a results.tsv with Precision / Recall / F1 at that cutoff (averaged over the
    prediction files when there are several folds).  Computed here instead of by the Java jar."""
    if not os.path.isdir(predictions_path):
        raise RuntimeError("Invalid predictions path specified. Unable to run evaluator.")
    test = pd.read_csv(test_filepath, sep=sep, header=None).to_numpy()
    out = {}
    for root, dirs, files in os.walk(predictions_path):
        preds = sorted(f for f in files if f.startswith("predictions"))
        if not preds:
            continue
        cutoff = int(str(root)[root.rfind(os.sep):].split("_")[1])
        rows = [precision_recall_f1_at_k(test, pd.read_csv(os.path.join(root, f), sep=sep, header=None).to_numpy(),
                                         cutoff, relevance_threshold) for f in preds]
        res = {m: float(np.mean([r[m] for r in rows])) for m in ("precision", "recall", "f1")}
        with open(os.path.join(root, "results.tsv"), "w") as fp:
            # one headerless row (label, precision, recall, f1): what the reference's caller reads back with
            # read_csv(header=None).drop(0, axis=1).squeeze() -> [P, R, F1]  (experiment.py:211-213)
            fp.write("top_%d\t%.6f\t%.6f\t%.6f\n" % (cutoff, res["precision"], res["recall"], res["f1"]))
        out[cutoff] = res
    return out
