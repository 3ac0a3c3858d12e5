"""Numpy restatement of what GAUC reads and computes in the reference (test infrastructure only):
  evaluator/collector.py   the rec.meanrank branch (sort every masked score row, _average_rank, argmin) and
                           _average_rank itself
  evaluator/metrics.py     GAUC.metric_info
Used by the GAUC tests to check the fused path (hopwise_b200.recommender.full_sort_meanrank,
hopwise_b200.evaluator.gauc_sums) against the same formulas on dense rows."""

from __future__ import annotations

import numpy as np


def average_rank(sorted_scores: np.ndarray) -> np.ndarray:
    """The collector's _average_rank: for rows that are already ordered, the 1-based position of every entry, runs
    of equal values sharing the mean of the positions they occupy."""
    srt = np.asarray(sorted_scores)
    n, m = srt.shape
    out = np.zeros((n, m), dtype=np.float64)
    pos = np.arange(1, m + 1, dtype=np.float64)
    for r in range(n):
        run = np.cumsum(np.concatenate([[True], srt[r, 1:] != srt[r, :-1]])) - 1   # run id of every position
        out[r] = (np.bincount(run, weights=pos) / np.bincount(run))[run]
    return out


def meanrank(masked_scores: np.ndarray, pos_u, pos_i) -> np.ndarray:
    """float32 [n, 3] rows (pos_rank_sum, user_len, pos_len) of rec.meanrank from masked score rows: the average
    ranks of the row's positives summed (a duplicate pair counts once), the argmin of the sorted row and the number
    of positives."""
    s = np.asarray(masked_scores)
    n, m = s.shape
    pos = np.zeros((n, m), dtype=bool)
    pos[np.asarray(pos_u, dtype=np.int64), np.asarray(pos_i, dtype=np.int64)] = True
    order = np.argsort(-s, axis=1, kind="stable")
    srt = np.take_along_axis(s, order, axis=1)
    ranks = average_rank(srt)
    pos_sorted = np.take_along_axis(pos, order, axis=1)
    rank_sum = (ranks * pos_sorted).sum(axis=1)
    user_len = np.argmin(srt, axis=1)
    return np.stack([rank_sum, user_len, pos.sum(axis=1)], axis=1).astype(np.float32)


def gauc(meanrank_rows: np.ndarray) -> float:
    """GAUC.metric_info: users without positives or without negatives dropped, auc_u = pair_num / (neg_len pos_len),
    pair_num = (user_len + 1) pos_len - pos_len (pos_len + 1) / 2 - pos_rank_sum, weighted by pos_len."""
    mr = np.asarray(meanrank_rows, dtype=np.float64)
    rank_sum, user_len, pos_len = mr[:, 0], mr[:, 1], mr[:, 2]
    neg_len = user_len - pos_len
    keep = (pos_len != 0) & (neg_len != 0)
    rank_sum, user_len, pos_len, neg_len = rank_sum[keep], user_len[keep], pos_len[keep], neg_len[keep]
    pair_num = (user_len + 1) * pos_len - pos_len * (pos_len + 1) / 2 - rank_sum
    return float((pair_num / (neg_len * pos_len) * pos_len).sum() / pos_len.sum())
