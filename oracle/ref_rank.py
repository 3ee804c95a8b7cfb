"""CPU oracle of the ranking evaluation (test infrastructure only: imported by tests/, never by the
product path). It restates DESIGN.md section 2, row f-5 by brute force on top of `full_predictions`
(model.py:82-84), the way `ref_topk.topk` does: per row, the candidates (every column unless `seen`
excludes it) in the order score descending, ties by ascending column (`np.lexsort`).

`targets` is a per-row list of (cols, vals): the row's target ratings in entry order. A repeated column
counts once with its last value (last writer). A target is relevant when its value is >= `min_value`
(None: all) and its column is a candidate."""
import numpy as np


def _order(scores_row, seen_cols):
    """(candidate columns in rank order, boolean candidate mask)."""
    s = np.asarray(scores_row, dtype=np.float32)
    cand = np.ones(s.size, dtype=bool)
    if seen_cols is not None:
        cand[np.asarray(seen_cols, dtype=np.int64)] = False
    cols = np.nonzero(cand)[0]
    order = np.lexsort((cols, -s[cols].astype(np.float64)))
    return cols[order], cand


def _relevant(target, cand, min_value):
    cols, vals = target
    last = {}
    for c, v in zip(np.asarray(cols).tolist(), np.asarray(vals, dtype=np.float32).tolist()):
        last[int(c)] = v
    keep = [c for c, v in last.items() if (min_value is None or v >= np.float32(min_value)) and cand[c]]
    return np.array(sorted(keep), dtype=np.int64)


def ranks(scores, targets, seen=None, min_value=None):
    """Returns (row_ptr int64 [B + 1], cols int64, ranks int64, n_cand int64 [B]): the relevant targets of
    every row in CSR form, columns ascending inside a row, with their 1-based rank among the candidates."""
    scores = np.asarray(scores)
    B = scores.shape[0]
    row_ptr = [0]
    out_c, out_r, n_cand = [], [], []
    for b in range(B):
        order, cand = _order(scores[b], None if seen is None else seen[b])
        rel = _relevant(targets[b], cand, min_value)
        place = np.empty(scores.shape[1], dtype=np.int64)
        place[order] = np.arange(1, order.size + 1)
        out_c.append(rel)
        out_r.append(place[rel])
        n_cand.append(order.size)
        row_ptr.append(row_ptr[-1] + rel.size)
    cat = lambda xs: np.concatenate(xs).astype(np.int64) if xs else np.zeros(0, dtype=np.int64)
    return np.array(row_ptr, dtype=np.int64), cat(out_c), cat(out_r), np.array(n_cand, dtype=np.int64)


def metrics(scores, targets, seen=None, ks=(10,), min_value=None):
    """The metrics of DESIGN.md section 2, row f-5, read off each row's sorted candidate list directly (no
    ranks): the mean over rows with a relevant target (AUC: and a negative), with the row counts."""
    scores = np.asarray(scores)
    sums = {"MRR": 0.0, "AUC": 0.0}
    for k in ks:
        for name in ("HR@%d", "precision@%d", "recall@%d", "NDCG@%d"):
            sums[name % k] = 0.0
    rows = auc_rows = 0
    for b in range(scores.shape[0]):
        order, cand = _order(scores[b], None if seen is None else seen[b])
        rel_cols = _relevant(targets[b], cand, min_value)
        if rel_cols.size == 0:
            continue
        rows += 1
        is_rel = np.isin(order, rel_cols)            # relevance along the ranked list
        n_rel = int(is_rel.sum())
        n_neg = order.size - n_rel
        sums["MRR"] += 1.0 / (np.argmax(is_rel) + 1)
        if n_neg >= 1:
            auc_rows += 1
            negs_ahead = np.cumsum(~is_rel)[is_rel]      # negatives ranked above each relevant target
            sums["AUC"] += 1.0 - float(negs_ahead.sum()) / (n_rel * n_neg)
        for k in ks:
            top = is_rel[:k]
            hits = int(top.sum())
            dcg = float(np.sum(top / np.log2(2.0 + np.arange(top.size))))
            idcg = float(np.sum(1.0 / np.log2(2.0 + np.arange(min(k, n_rel)))))
            sums["HR@%d" % k] += float(hits > 0)
            sums["precision@%d" % k] += hits / k
            sums["recall@%d" % k] += hits / n_rel
            sums["NDCG@%d" % k] += dcg / idcg
    out = {"rows": rows, "AUC_rows": auc_rows}
    for name, v in sums.items():
        n = auc_rows if name == "AUC" else rows
        out[name] = v / n if n else float("nan")
    return out
