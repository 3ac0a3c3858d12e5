"""The adversarial cases of tests/test_gpu_mma_filter.py reach the regime each is built for (no GPU needed).

A case that does not reach its regime tests nothing on the device, so every builder of tests/mma_filter_cases.py is
checked here with the numpy restatement of the filter (tests/test_filter_proof_cpu.py) laid out over the candidate
lists plan_mma gives the case:
  filter     no row is flagged, every exact top-k member is scored, and in some rows the fp16 order is wrong at the k-th
             place (an exact member's a^ below a non-member's): the filter and the exact rescore decided the answer
  overflow   exactly the rows built for it are flagged by a list that cannot be compacted
  survivors  the rescore gets more than 256 entries (its shared-memory radix), more groups than one fill holds (several
             fills) and more than RS_KEYS = 64 passing keys (the staged keys are folded into the sorted list)
  few / bad  the rows built for it are flagged by n_pass < k, or as rows the fp16 scaling cannot hold

The rescore's L2 pre-filter and the ranking.  For TransE / RotatE the rescore keeps a scored target when its fp32 chain
acc = sum (q_c - t_c)^2 satisfies acc <= hi_acc = (|q|^2 - 2 lo_a) 1.00001 + 4e-6 |q|^2, lo_a = (tau - 1.25 eps) / S.
A top-k member has S a >= tau - eps, so its exact |q - t|^2 sits at least 0.5 eps / S below |q|^2 - 2 lo_a; the chain
rounds it up by at most (P + 1) 2^-24 |q - t|^2 (P = parts * d columns, one rounding per column and two in the
difference).  When |q| << |t| the 2^-10 |q| tmax term of eps no longer covers that, but eps has a term that does not
shrink with |q|: K 2^-22 * 256 c (the fp32 accumulation of the norm columns), and c / S = 2^-e_w > max |t|^2 / 2^9, so
0.5 eps / S >= K 2^-24 max |t|^2 with K >= P + 3.  When |q| >> |t| the 1e-5 relative slack and 0.5 * 2^-10 |q| tmax
carry it up to |q| / tmax of a few hundred at K = 640, beyond which a chain rounded up at nearly every column could
exceed hi_acc.  Even then a member is not lost silently: the pre-filter and the ranking are monotone in the same fp32
value, so what fails the pre-filter is a tail of the exact ranking (up to keys whose fp32 scores tie, which the id
breaks); losing a member loses every key ranked below it, fewer than k keys pass and the row is flagged
(test_prefilter_is_a_tail_of_the_ranking restates this).
"""

import numpy as np
import pytest

import mma_filter_cases as mfc

CASES = mfc.all_cases()


def _flags(res):
    return [r["flag"] for r in res]


def _unflagged(res):
    return [r for r in res if r["flag"] is None]


@pytest.mark.parametrize("case_id", [c for c, v in CASES.items() if v.regime == "filter"])
def test_filter_cases_are_decided_by_the_filter(case_id):
    case = CASES[case_id]
    res, pl = mfc.simulate(case)
    assert _flags(res) == [None] * len(res), "a filter case must not send rows to the exact kernel"
    assert all(r["kept_all"] for r in res), "the filter dropped an exact top-k member"
    a = case.exact()
    if case.expect.get("tie_at_k"):
        for r in range(len(res)):
            row = np.where(case.masked(r), -np.inf, a[r])
            top = np.sort(row)[::-1]
            assert top[case.k - 1] == top[case.k], "the k-th place must be a tie"
    elif case.expect.get("last_in_topk"):
        last = len(case.T) - 1
        assert last % mfc.CH == len(case.T) % mfc.CH - 1 or len(case.T) % mfc.CH == 0
        for r in range(len(res)):
            assert last in np.argsort(-a[r], kind="stable")[: case.k]
    elif case.id.startswith("long_k"):
        # products of alternating sign: the best score is a small part of the sum of the products' magnitudes
        mag = np.abs(case.Q.astype(np.float64)) @ np.abs(case.T.astype(np.float64)).T
        best = np.argmax(a, axis=1)
        assert np.all(np.abs(case.Q.astype(np.float64) @ case.T.astype(np.float64).T)[np.arange(len(a)), best]
                      < 0.2 * mag[np.arange(len(a)), best])
    else:
        assert sum(r["wrong_order"] for r in res) >= 1, "the fp16 order is right everywhere: the filter decides nothing"


@pytest.mark.parametrize("cfg", ["", "f"])
@pytest.mark.parametrize("case_id", [c for c, v in CASES.items() if v.regime == "overflow"])
def test_overflow_cases_fill_their_lists(case_id, cfg):
    case = CASES[case_id]
    res, pl = mfc.simulate(case, cfg)
    n_zero = case.expect["flagged"]
    assert _flags(res) == ["overflow"] * n_zero + [None] * (len(res) - n_zero)
    # a list fills only when its slice holds more than TRIG chunks: the catalogue is sized for that under this plan
    assert min(len(lst) * len(lst[0]) for lst in mfc.lists_for(pl)) > mfc.CAND - 5
    if n_zero > 1024:
        assert pl["cfg"] in "af"   # (more flagged rows than FB_SPLIT_ROWS: the fallback's region B)


def test_the_same_rows_below_the_list_capacity_go_to_the_rescore():
    """A zero query over a catalogue whose lists hold fewer chunks than the compaction trigger is not flagged: its
    entries reach the rescore, far more than 256 of them."""
    case = mfc.overflow("DistMult", 10, 4, n_other=4, n_targets=12000)
    res, pl = mfc.simulate(case)
    assert max(len(lst) * len(lst[0]) for lst in mfc.lists_for(pl)) <= mfc.CAND - 5
    assert _flags(res) == [None] * 8
    assert res[0]["E"] == 12000 // mfc.CH + 1 and res[0]["n_pass"] == 12000 - 1


@pytest.mark.parametrize("cfg", ["", "f"])
@pytest.mark.parametrize("case_id", [c for c, v in CASES.items() if v.regime == "survivors"])
def test_survivor_cases_reach_the_large_rescore_branches(case_id, cfg):
    case = CASES[case_id]
    res, pl = mfc.simulate(case, cfg)
    assert _flags(res) == [None] * len(res)
    assert all(r["kept_all"] for r in res)
    assert min(r["E"] for r in res) > 256                       # shared-memory radix select of tau
    assert min(r["groups"] for r in res) > pl["nent"]           # several fills of the group-id buffer
    assert max(r["n_pass"] for r in res) > mfc.RS_KEYS           # the staged keys are folded into the sorted list


@pytest.mark.parametrize("case_id", [c for c in CASES if c.startswith("masking")])
def test_masking_cases(case_id):
    case = CASES[case_id]
    res, pl = mfc.simulate(case)
    e = case.expect
    assert [i for i, f in enumerate(_flags(res)) if f] == e["few_rows"]
    assert all(res[i]["flag"] == "few" for i in e["few_rows"])
    assert len(case.hist[e["long_hist_row"]]) > 256
    assert (~case.masked(e["exactly_k_row"])).sum() == case.k
    assert (~case.masked(e["few_rows"][0])).sum() == case.k - 1
    a = case.exact()
    kth = np.array([np.sort(np.where(case.masked(r), -np.inf, a[r]))[-case.k] for r in range(len(a))])
    assert np.mean(a[:, 0] > kth) > (0.0 if case.dist else 0.99), "target 0 ([PAD]) must outscore the exact top-k"
    assert all(r["kept_all"] for r in _unflagged(res))
    # history items outscore the k-th unmasked target: their chunks' maxima would lift tau above the true top-k if
    # unsafe chunks fed it
    for r in range(4, len(a)):
        assert a[r, case.hist[r]].max() > kth[r]


def test_magnitude_cases():
    def exps(case):
        q = np.abs(case.Q).max(1)
        e_i = 7 - np.floor(np.log2(q))
        tn2 = (case.T.astype(np.float32) ** 2).sum(1, dtype=np.float32)
        e_t = 7 - np.floor(np.log2(np.abs(case.T).max()))
        e_w = np.clip(7 - np.floor(np.log2(0.5 * tn2.max())), -60, 60)
        return e_i, np.clip(e_i, -60, 60) + e_t - e_w

    c = CASES["magnitudes-DistMult-rowscale-k32"]
    res, _ = mfc.simulate(c)
    e_i, _ = exps(c)
    assert e_i.max() > 60 and e_i.min() < -40                   # the E_CLAMP clamp is reached
    assert _flags(res) == [None] * len(res)
    c = CASES["magnitudes-TransE-rowscale-k10"]
    res, _ = mfc.simulate(c)
    _, e_c = exps(c)
    assert (e_c > 15).any()                                     # rows whose scale is lowered to keep c_i in fp16
    assert [f == "bad" for f in _flags(res)] == list(e_c < -14)  # e_c < -14: flagged, never dropped
    assert all(r["kept_all"] for r in _unflagged(res))
    c = CASES["magnitudes-DistMult-nonfinite-k10"]
    res, _ = mfc.simulate(c)
    assert [i for i, f in enumerate(_flags(res)) if f] == [5, 6] and {res[5]["flag"], res[6]["flag"]} == {"bad"}
    assert np.isfinite(c.Q[6]).all()                            # row 6: finite, but |q|^2 overflows fp32
    for cid in ("magnitudes-ComplEx-subnormal-k10", "magnitudes-RotatE-subnormal-k32"):
        c = CASES[cid]
        e_i, _ = exps(c)
        scaled = np.abs(np.ldexp(c.Q, e_i[:, None].astype(int)))
        assert ((scaled > 0) & (scaled < 2.0 ** -14)).any()     # fp16-subnormal after scaling
    # L2 tables at 1e12: max |t|^2 / 2 > 2^68 puts e_w at its clamp and the norm columns overflow fp16, so the sweep
    # cannot rank anything and every row goes to the exact kernel (slow, still exact)
    c = CASES["magnitudes-TransE-huge-k10"]
    res, _ = mfc.simulate(c)
    assert _flags(res) == ["few"] * len(res)


def test_sweep_shapes_change_the_lists():
    """Shape a: one list per target split; f and k: two column slices per split; c: 64-wide tiles."""
    for cfg, ncol, tn in (("a", 1, 128), ("f", 2, 128), ("c", 1, 64), ("k", 2, 128)):
        pl = mfc.plan("DistMult", 64, 256, 20000, cfg)
        assert (pl["cfg"], pl["ncol"], pl["tn"], pl["splits"]) == (cfg, ncol, tn, 4)
        chunks = sorted(c for lst in mfc.lists_for(pl) for tile in lst for c in tile)
        assert chunks == list(range(pl["n_tiles"] * tn // mfc.CH))
    assert mfc.plan("DistMult", 640, 128, 9000, "a")["cfg"] == "k"      # K = 640 only fits shape k
    assert mfc.plan("DistMult", 64, 1, 8192)["splits"] == mfc.MAX_SPLITS


def test_prefilter_is_a_tail_of_the_ranking():
    """The rescore's pre-filter (acc >= lo_a, or acc <= hi_acc for the L2 models) and the final order (score desc, id
    asc, score = acc or margin - sqrt(acc)) are monotone in the same fp32 value: the keys that fail it are a tail of the
    exact ranking of the scored targets, so a member can only be lost together with everything ranked below it, and
    then fewer than k keys pass and the row is flagged."""
    rng = np.random.default_rng(2)
    acc = np.sort(rng.random(2000).astype(np.float32))
    acc[100:110] = acc[100]                                      # ties
    for dist in (False, True):
        score = (np.float32(1.0) - np.sqrt(acc)).astype(np.float32) if dist else acc
        ids = rng.permutation(len(acc))
        order = np.lexsort((ids, -score))
        for cut in acc[::37]:
            passing = (acc <= cut) if dist else (acc >= cut)
            ranked = passing[order]
            assert not np.any(~ranked[:-1] & ranked[1:]), "a key ranked below a failed key passed"
