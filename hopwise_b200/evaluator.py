"""Fused full-sort evaluation: scores -> mask -> top-k -> hit matrix -> ranking metrics.

Host-side mirror of (paths under /root/reference/hopwise/):
  trainer/trainer.py:716-735      _full_sort_batch_eval (scores[:,0] = -inf, history -> -inf)
  evaluator/collector.py:152-206  Collector.eval_batch_collect ("rec.topk" = pos_idx | pos_len)
  evaluator/collector.py:234-249  get_data_struct
  evaluator/base_metric.py:75-99  used_info / topk_result (mean over users, value at k-1, rounding)
  evaluator/metrics.py:44-232     Hit, MRR, Recall, NDCG, Precision
  evaluator/collector.py          the "rec.meanrank" branch and _average_rank
  evaluator/metrics.py            GAUC.metric_info
  evaluator/evaluator.py:27-41    Evaluator.evaluate -> OrderedDict

The dense [n_users, n_items] score matrix of the reference never exists here: the kernel keeps
the per-user top-k on chip, and GAUC's ranks are counted during the same kind of sweep
(kge_full_sort_rank_counts).  Tie order is (score desc, item id asc).

Sampled evaluation (eval_args.mode uniN / popN: trainer.py's _neg_sample_batch_eval scatters the candidate scores
into -inf rows of n_items columns) goes through collect_sampled: the loader's batches are concatenated on the device
and every block of users takes one kge_candidate_select call over its candidate lists.
"""

from __future__ import annotations

import ctypes as C
from collections import OrderedDict

import numpy as np
import torch

from . import _abi

METRIC_ORDER = ("recall", "mrr", "ndcg", "hit", "precision")  # row order of kge_topk_metric_sums


def csr_from_pairs(rows, cols, n_rows: int, device):
    """(offsets[n_rows+1], cols sorted per row) from COO pairs such as the loader's
    (history_row, history_col) / (positive_u, positive_i) (general_dataloader.py:253-267)."""
    rows = torch.as_tensor(rows, dtype=torch.int64).to(device)
    cols = torch.as_tensor(cols, dtype=torch.int64).to(device)
    if rows.numel():
        span = int(cols.max().item()) + 1
        packed, _ = torch.sort(rows * span + cols)
        r2 = torch.div(packed, span, rounding_mode="floor")
        c2 = packed - r2 * span
        counts = torch.bincount(r2, minlength=n_rows)
    else:
        c2 = torch.zeros(0, dtype=torch.int64, device=device)
        counts = torch.zeros(n_rows, dtype=torch.int64, device=device)
    off = torch.zeros(n_rows + 1, dtype=torch.int64, device=device)
    torch.cumsum(counts, 0, out=off[1:])
    return off, c2.contiguous()


def topk_hits(ids: torch.Tensor, pos_off: torch.Tensor, pos_items: torch.Tensor) -> torch.Tensor:
    """int32 [n, k+1]: hit flags of the top-k ids then pos_len (collector.py:178-183)."""
    n, k = ids.shape
    out = torch.empty(n, k + 1, dtype=torch.int32, device=ids.device)
    _abi.check(
        _abi.lib().kge_topk_hits(ids.data_ptr(), n, k, pos_off.data_ptr(), pos_items.data_ptr(), out.data_ptr(),
                                 _abi.stream_ptr()),
        "kge_topk_hits",
    )
    return out


def topk_metric_sums(rec_topk: torch.Tensor) -> torch.Tensor:
    """float64 [5, k] sums over users of recall, mrr, ndcg, hit, precision at every cutoff."""
    n, k1 = rec_topk.shape
    k = k1 - 1
    sums = torch.zeros(5, k, dtype=torch.float64, device=rec_topk.device)
    rec_topk = rec_topk.contiguous()
    _abi.check(
        _abi.lib().kge_topk_metric_sums(rec_topk.data_ptr(), n, k, sums.data_ptr(), _abi.stream_ptr()),
        "kge_topk_metric_sums",
    )
    return sums


def metrics_from_sums(sums: torch.Tensor, n_users: int, topk, metrics=("recall", "mrr", "ndcg", "hit", "precision"),
                      decimals: int | None = 4) -> OrderedDict:
    """The Evaluator.evaluate() dictionary: {'recall@10': ..} (base_metric.py:86-99)."""
    host = sums.cpu().numpy() / float(n_users)
    out = OrderedDict()
    for name in metrics:
        row = host[METRIC_ORDER.index(name.lower())]
        for k in topk:
            v = float(row[k - 1])
            out[f"{name.lower()}@{k}"] = round(v, decimals) if decimals is not None else v
    return out


def gauc_sums(meanrank: torch.Tensor) -> torch.Tensor:
    """float64 [2] = (sum of auc_u * pos_len, sum of pos_len) over the users GAUC keeps, from rec.meanrank rows
    (pos_rank_sum, user_len, pos_len) (GAUC.metric_info): users without positives or without negatives are dropped,
    auc_u = ((user_len + 1) pos_len - pos_len (pos_len + 1) / 2 - pos_rank_sum) / (neg_len pos_len).  Sums of
    user blocks or ranks add up; GAUC = sums[0] / sums[1]."""
    rank_sum, user_len, pos_len = meanrank.to(torch.float64).unbind(1)
    neg_len = user_len - pos_len
    keep = (pos_len != 0) & (neg_len != 0)
    pair_num = (user_len + 1) * pos_len - pos_len * (pos_len + 1) / 2 - rank_sum
    weighted = torch.where(keep, pair_num / torch.where(keep, neg_len * pos_len, 1.0), 0.0) * pos_len
    return torch.stack([weighted.sum(), torch.where(keep, pos_len, 0.0).sum()])


def gauc_from_sums(sums: torch.Tensor, decimals: int | None = 4) -> float:
    """GAUC = sum(auc_u * pos_len) / sum(pos_len), rounded like GAUC.calculate_metric."""
    host = sums.cpu()
    v = float(host[0] / host[1])
    return round(v, decimals) if decimals is not None else v


class FusedCollector:
    """Collector twin fed by the fused top-k instead of dense scores.

    ``eval_batch_collect(model, user_ids, history_index, positive_u, positive_i)`` takes the same
    per-batch tuple the reference loader yields; ``get_data_struct()`` returns
    ``{"rec.topk": int32 [n_users, max(topk)+1], "rec.items": ids, "topk": topk}``, plus
    ``"rec.meanrank"`` (float32 [n_users, 3], full_sort_meanrank) when the config's metrics include GAUC.
    """

    def __init__(self, config):
        self.topk = list(config["topk"])
        self.kmax = max(self.topk)
        try:
            metrics = config["metrics"]
        except (KeyError, TypeError):
            metrics = None
        self.meanrank = any(str(x).lower() == "gauc" for x in (metrics or ()))
        self._topk, self._items, self._meanrank = [], [], []

    def eval_batch_collect(self, model, user_ids, history_index, positive_u, positive_i):
        device = next(model.parameters()).device
        users = torch.as_tensor(user_ids).to(device)
        n = users.numel()
        hist_off = hist_items = None
        if history_index is not None:
            hist_off, hist_items = csr_from_pairs(history_index[0], history_index[1], n, device)
        ids, _ = model.full_sort_topk(users, self.kmax, hist_off, hist_items, mask_pad=True, return_scores=False)
        pos_off, pos_items = csr_from_pairs(positive_u, positive_i, n, device)
        self._topk.append(topk_hits(ids, pos_off, pos_items))
        self._items.append(ids)
        if self.meanrank:
            self._meanrank.append(model.full_sort_meanrank(users, pos_off, pos_items, hist_off, hist_items, mask_pad=True))
        return ids

    def get_data_struct(self):
        rec = torch.cat(self._topk) if self._topk else torch.zeros(0, self.kmax + 1, dtype=torch.int32)
        items = torch.cat(self._items) if self._items else torch.zeros(0, self.kmax, dtype=torch.int64)
        struct = {"rec.topk": rec, "rec.items": items, "topk": self.topk}
        if self.meanrank:
            struct["rec.meanrank"] = torch.cat(self._meanrank) if self._meanrank else torch.zeros(0, 3)
        self._topk, self._items, self._meanrank = [], [], []
        return struct


def evaluate_full_sort(model, user_ids, hist_off, hist_items, pos_off, pos_items, topk=(10,), decimals=4,
                       user_block: int | None = None, return_struct: bool = False, gauc: bool = False):
    """Whole-split evaluation with device-resident CSR inputs; returns the metric dictionary (with ``gauc=True``
    it also holds ``"gauc"``, from full_sort_meanrank)."""
    device = next(model.parameters()).device
    users = torch.as_tensor(user_ids).to(device)
    n = users.numel()
    kmax = max(topk)
    block = user_block or n
    sums = torch.zeros(5, kmax, dtype=torch.float64, device=device)
    g_sums = torch.zeros(2, dtype=torch.float64, device=device)
    recs = []
    for s in range(0, n, block):
        e = min(n, s + block)
        ho = hi = None
        if hist_off is not None:
            base = hist_off[s]
            ho = (hist_off[s : e + 1] - base).contiguous()
            hi = hist_items[int(base.item()) : int(hist_off[e].item())] if block < n else hist_items
        ids, _ = model.full_sort_topk(users[s:e], kmax, ho, hi, mask_pad=True, return_scores=False)
        pbase = pos_off[s]
        po = (pos_off[s : e + 1] - pbase).contiguous()
        pi = pos_items[int(pbase.item()) : int(pos_off[e].item())] if block < n else pos_items
        rec = topk_hits(ids, po, pi)
        sums += topk_metric_sums(rec)
        if gauc:
            g_sums += gauc_sums(model.full_sort_meanrank(users[s:e], po, pi, ho, hi, mask_pad=True))
        if return_struct:
            recs.append(rec)
    result = metrics_from_sums(sums, n, topk, decimals=decimals)
    if gauc:
        result["gauc"] = gauc_from_sums(g_sums, decimals)
    if return_struct:
        return result, torch.cat(recs)
    return result


def collect_sampled(model, batches, k: int, meanrank: bool = False, user_block: int | None = None):
    """The collector's data of a sampled evaluation, without the [batch_users, n_items] score rows.

    ``batches`` yields what hopwise's sampled loader yields and ``_neg_sample_batch_eval`` receives:
    ``(interaction, row_idx, positive_u, positive_i)``, with the candidate rows of each batch user contiguous in
    ``interaction`` and ``row_idx`` naming their batch-local user; the batch has ``positive_u[-1] + 1`` users.  It is
    iterated exactly once (the loader draws fresh negatives on every pass).  Returns ``(struct, n_batches)``: struct
    holds ``"rec.topk"`` (int32 [n, k+1]), ``"rec.items"`` (int64 [n, k]), ``"rec.users"`` (the interactions' user
    column) and, with ``meanrank``, ``"rec.meanrank"`` (float32 [n, 3]); the rows are the batches' users in order.
    Every block of ``user_block`` users (default: all) takes one kge_candidate_select call."""
    device = next(model.parameters()).device
    users, items, counts, pos_rows, pos_items = [], [], [], [], []
    n = n_batches = 0
    for interaction, row_idx, positive_u, positive_i in batches:
        n_batches += 1
        pu = torch.as_tensor(positive_u, dtype=torch.int64).cpu()
        rows = torch.as_tensor(row_idx, dtype=torch.int64).cpu()
        n_b = int(pu[-1]) + 1 if pu.numel() else 0   # trainer.py: batch_user_num = positive_u[-1] + 1
        if rows.numel() and (bool((rows.diff() < 0).any()) or int(rows[-1]) >= n_b or int(rows[0]) < 0):
            raise ValueError("the candidate rows of a batch must be grouped by user, in order, inside the batch's users")
        counts.append(torch.bincount(rows, minlength=n_b))
        users.append(torch.as_tensor(interaction[model.USER_ID]).to(device, non_blocking=True))
        items.append(torch.as_tensor(interaction[model.ITEM_ID]).to(device, non_blocking=True))
        pos_rows.append(pu + n)
        pos_items.append(torch.as_tensor(positive_i, dtype=torch.int64).cpu())
        n += n_b
    cand_off = torch.zeros(n + 1, dtype=torch.int64)
    if n:
        torch.cumsum(torch.cat(counts), 0, out=cand_off[1:])
    user_col = torch.cat(users) if users else torch.zeros(0, dtype=torch.int64, device=device)
    item_col = torch.cat(items) if items else torch.zeros(0, dtype=torch.int64, device=device)
    # the positives CSR, each (user, item) once: pos_matrix[positive_u, positive_i] = 1 (collector.py)
    pr = torch.cat(pos_rows).numpy() if pos_rows else np.zeros(0, np.int64)
    pi = torch.cat(pos_items).numpy() if pos_items else np.zeros(0, np.int64)
    span = int(max(model.n_items, pi.max() + 1 if pi.size else 1))
    packed = np.unique(pr * span + pi)
    prow = packed // span
    pos_off = np.zeros(n + 1, dtype=np.int64)
    np.cumsum(np.bincount(prow, minlength=n), out=pos_off[1:])
    pos_items_d = torch.from_numpy(packed - prow * span).to(device)
    pos_off_d = torch.from_numpy(pos_off).to(device)
    block = max(1, user_block or n)
    topk, ids_all, mr = [], [], []
    for s in range(0, n, block):
        e = min(n, s + block)
        c0, c1, p0, p1 = int(cand_off[s]), int(cand_off[e]), int(pos_off[s]), int(pos_off[e])
        po, pv = pos_off_d[s : e + 1] - p0, pos_items_d[p0:p1]
        ids, _, greater, equal, n_unmasked = model._candidate_select(
            user_col[c0:c1], item_col[c0:c1], cand_off[s : e + 1] - c0, k, True, False,
            po if meanrank else None, pv if meanrank else None)
        topk.append(topk_hits(ids, po, pv))
        ids_all.append(ids)
        if meanrank:
            mr.append(model._meanrank_rows(greater, equal, n_unmasked, po, pv))
    struct = {"rec.topk": torch.cat(topk) if topk else torch.zeros(0, k + 1, dtype=torch.int32, device=device),
              "rec.items": torch.cat(ids_all) if ids_all else torch.zeros(0, k, dtype=torch.int64, device=device),
              "rec.users": user_col}
    if meanrank:
        struct["rec.meanrank"] = torch.cat(mr) if mr else torch.zeros(0, 3, device=device)
    return struct, n_batches
