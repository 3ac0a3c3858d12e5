"""GAUC without a GPU: the numpy oracle of rec.meanrank / GAUC (collector.py's rec.meanrank branch and _average_rank,
metrics.py GAUC) against the reference's known answer and a brute-force pairwise AUC, and the library's gauc_sums
against the oracle."""

import numpy as np
import torch

import gauc_oracle as go
from oracle import fullsort as ofs


def test_average_rank_known_answer():
    """The example of the collector's _average_rank docstring."""
    got = go.average_rank(np.array([[1, 2, 2, 2, 3, 3, 6], [2, 2, 2, 2, 4, 5, 5]]))
    np.testing.assert_array_equal(got, [[1, 3, 3, 3, 5.5, 5.5, 7], [2.5, 2.5, 2.5, 2.5, 5, 6.5, 6.5]])


def _random_case(seed, n=40, m=60):
    """Scores with many ties (5 levels), 0-6 positives per user (so some users have none), some users whose
    positives are every unmasked item (no negatives), history masked."""
    rng = np.random.default_rng(seed)
    scores = rng.integers(0, 5, (n, m)).astype(np.float32)
    hist_u, hist_i, pos_u, pos_i = [], [], [], []
    for u in range(n):
        h = rng.choice(np.arange(1, m), int(rng.integers(0, 8)), replace=False)
        hist_u += [u] * len(h)
        hist_i += list(h)
        free = np.setdiff1d(np.arange(1, m), h)
        k = len(free) if u % 13 == 5 else int(rng.integers(0, 7))
        p = rng.choice(free, k, replace=False)
        pos_u += [u] * len(p)
        pos_i += list(p)
    return scores, np.array(hist_u), np.array(hist_i), np.array(pos_u), np.array(pos_i)


def _pairwise_auc(masked, pos_u, pos_i):
    """Per user: positives against the unmasked non-positives, ties counted 1/2, weighted by the positives."""
    pos = np.zeros(masked.shape, dtype=bool)
    pos[pos_u, pos_i] = True
    num = den = 0.0
    for u in range(masked.shape[0]):
        p = masked[u][pos[u]]
        q = masked[u][~pos[u] & np.isfinite(masked[u])]
        if len(p) == 0 or len(q) == 0:
            continue
        wins = (p[:, None] > q[None, :]).sum() + 0.5 * (p[:, None] == q[None, :]).sum()
        num += wins / (len(p) * len(q)) * len(p)
        den += len(p)
    return num / den


def test_gauc_equals_pairwise_auc():
    for seed in range(3):
        scores, hu, hi, pu, pi = _random_case(seed)
        masked = ofs.mask_scores(scores, hu, hi)
        mr = go.meanrank(masked, pu, pi)
        counts = np.bincount(pu, minlength=len(scores))
        assert (counts == 0).any() and (mr[:, 1] == mr[:, 2]).any()   # users GAUC drops are in the data
        np.testing.assert_array_equal(mr[:, 1], np.isfinite(masked).sum(axis=1))   # user_len = unmasked targets
        np.testing.assert_array_equal(mr[:, 2], counts)
        assert abs(go.gauc(mr) - _pairwise_auc(masked, pu, pi)) < 1e-12


def test_masked_positive_follows_the_reference_arithmetic():
    """A masked positive scores -inf: its average rank is U + (M + 1) / 2 (U unmasked targets above it, the M
    masked ones tied with it).  GAUC's formula then is not the pairwise AUC (neg_len = user_len - pos_len counts the
    masked positive among the unmasked targets): the oracle follows the formula, as the reference does."""
    scores = np.array([[0, 3, 1, 2, 2, 5, 4, 0]], dtype=np.float32)
    masked = ofs.mask_scores(scores, [0, 0], [3, 6])            # item 3 is a positive in the history
    pos_i = np.array([3, 4, 5])
    mr = go.meanrank(masked, np.zeros(3, dtype=np.int64), pos_i)
    U, M = 5, 3                                                  # unmasked: 1, 2, 4, 5, 7; masked: 0, 3, 6
    # finite scores descending: 5 (5), 3 (1), 2 (4), 1 (2), 0 (7) -> item 4 at 3, item 5 at 1
    want_sum = (U + (M + 1) / 2) + 3 + 1
    np.testing.assert_array_equal(mr, [[want_sum, U, 3]])
    pair_num = (U + 1) * 3 - 3 * 4 / 2 - want_sum
    assert go.gauc(mr) == pair_num / ((U - 3) * 3)
    # without the masked positive the same user is the pairwise AUC again
    mr2 = go.meanrank(masked, np.zeros(2, dtype=np.int64), pos_i[1:])
    assert go.gauc(mr2) == _pairwise_auc(masked, np.zeros(2, dtype=np.int64), pos_i[1:])


def test_gauc_sums_add_over_blocks():
    from hopwise_b200.evaluator import gauc_from_sums, gauc_sums

    scores, hu, hi, pu, pi = _random_case(7, n=90)
    mr = torch.from_numpy(go.meanrank(ofs.mask_scores(scores, hu, hi), pu, pi))
    whole = gauc_sums(mr)
    parts = sum(gauc_sums(mr[a:b]) for a, b in ((0, 13), (13, 14), (14, 60), (60, 90)))
    assert whole.dtype == torch.float64
    np.testing.assert_allclose(parts.numpy(), whole.numpy(), rtol=1e-14)
    assert abs(gauc_from_sums(whole, None) - go.gauc(mr.numpy())) < 1e-12
    assert gauc_from_sums(whole) == round(go.gauc(mr.numpy()), 4)
