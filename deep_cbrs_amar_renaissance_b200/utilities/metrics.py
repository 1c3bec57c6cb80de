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
