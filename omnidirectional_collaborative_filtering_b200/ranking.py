"""Ranking metrics from exact ranks (host side of `OmniNet.evaluate_ranking`; DESIGN.md section 2, row f-5).

The device (`ocf_rank_targets`) gives every relevant target of a batch row its 1-based rank among the row's
candidate columns, in the order `recommend` uses (score descending, ties by ascending column). This module
turns ranks into metrics, in float64:

  for a row with n_rel >= 1 relevant targets and n_neg = n_cand - n_rel other candidates,
    hits@k       = #{t : rank(t) <= k}
    HR@k         = [hits@k > 0]
    precision@k  = hits@k / k
    recall@k     = hits@k / n_rel
    NDCG@k       = sum_{rank(t) <= k} 1 / log2(1 + rank(t))  /  sum_{i = 1}^{min(k, n_rel)} 1 / log2(1 + i)
    MRR          = 1 / min_t rank(t)
    AUC          = 1 - sum_t (rank(t) - pos(t)) / (n_rel * n_neg)      (pos(t): t's place among the row's
                   targets sorted by rank; only for rows with n_neg >= 1)

Each metric is the mean over the rows that have a relevant target (AUC: and a negative). `metrics_from_ranks`
returns sums and row counts so that batches accumulate; `finalize` turns them into means.
"""
from __future__ import annotations

import numpy as np


def _k_names(k):
    return ("HR@%d" % k, "precision@%d" % k, "recall@%d" % k, "NDCG@%d" % k)


def empty_sums(ks):
    """Sums of zero rows (the start of an accumulation over batches)."""
    out = {"rows": 0, "AUC_rows": 0, "MRR": 0.0, "AUC": 0.0}
    for k in ks:
        for name in _k_names(int(k)):
            out[name] = 0.0
    return out


def metrics_from_ranks(row_ptr, ranks, n_cand, ks):
    """Per-metric sums over the rows of one batch.

    row_ptr [rows + 1]: row r's relevant targets are ranks[row_ptr[r]:row_ptr[r + 1]] (any order);
    ranks: 1-based ranks among the row's candidates; n_cand [rows]: candidates of each row.
    Returns a dict: "rows" (rows with a relevant target), "AUC_rows" (of those, rows with a negative),
    and the sums of "MRR", "AUC" and, for every k in `ks`, "HR@k", "precision@k", "recall@k", "NDCG@k"."""
    row_ptr = np.asarray(row_ptr, dtype=np.int64)
    ranks = np.asarray(ranks, dtype=np.int64)
    n_cand = np.asarray(n_cand, dtype=np.int64)
    n_rows = row_ptr.size - 1
    out = empty_sums(ks)
    n_rel = np.diff(row_ptr)
    if ranks.size == 0:
        return out
    if ranks.min() < 1:
        raise ValueError("ranks are 1-based")
    row = np.repeat(np.arange(n_rows, dtype=np.int64), n_rel)
    order = np.lexsort((ranks, row))                  # by row, then by rank
    ranks = ranks[order]
    pos = np.arange(ranks.size, dtype=np.int64) - np.repeat(row_ptr[:-1], n_rel) + 1
    has = n_rel > 0
    out["rows"] = int(has.sum())
    rel = n_rel[has].astype(np.float64)
    first = ranks[row_ptr[:-1][has]]                  # each row's best rank
    out["MRR"] = float(np.sum(1.0 / first.astype(np.float64)))
    n_neg = n_cand - n_rel
    if np.any(n_neg[has] < 0):
        raise ValueError("a row has more relevant targets than candidates")
    gap = np.bincount(row, weights=(ranks - pos).astype(np.float64), minlength=n_rows)
    auc_ok = has & (n_neg >= 1)
    out["AUC_rows"] = int(auc_ok.sum())
    out["AUC"] = float(np.sum(1.0 - gap[auc_ok] / (n_rel[auc_ok].astype(np.float64) * n_neg[auc_ok])))
    gain = 1.0 / np.log2(1.0 + ranks.astype(np.float64))
    for k in ks:
        k = int(k)
        if k < 1:
            raise ValueError("k must be >= 1")
        inside = ranks <= k
        hits = np.bincount(row, weights=inside.astype(np.float64), minlength=n_rows)[has]
        dcg = np.bincount(row, weights=np.where(inside, gain, 0.0), minlength=n_rows)[has]
        ideal = np.cumsum(1.0 / np.log2(2.0 + np.arange(k, dtype=np.float64)))
        idcg = ideal[np.minimum(n_rel[has], k) - 1]
        hr, prec, recall, ndcg = _k_names(k)
        out[hr] = float(np.sum(hits > 0))
        out[prec] = float(np.sum(hits / k))
        out[recall] = float(np.sum(hits / rel))
        out[ndcg] = float(np.sum(dcg / idcg))
    return out


def accumulate(total, part):
    """Adds the sums of `part` into `total` (same ks) and returns `total`."""
    for name, v in part.items():
        total[name] = total[name] + v
    return total


def finalize(sums):
    """Means from accumulated sums: every metric over "rows" (AUC over "AUC_rows"); NaN over zero rows.
    The two row counts are kept."""
    out = {"rows": int(sums["rows"]), "AUC_rows": int(sums["AUC_rows"])}
    for name, v in sums.items():
        if name in ("rows", "AUC_rows"):
            continue
        n = sums["AUC_rows"] if name == "AUC" else sums["rows"]
        out[name] = float(v) / n if n else float("nan")
    return out
