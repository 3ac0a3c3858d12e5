"""The tensor-core full-sort top-k on the adversarial cases of tests/mma_filter_cases.py, under every sweep shape.

Each case (its regime is asserted by tests/test_mma_filter_cases_cpu.py) checks
  (a) path="mma" gives the ids and scores of path="cuda" bit for bit;
  (b) the ids and scores are the canonical top-k (score desc, id asc) of the product's own dense scores after the
      trainer's masking, and the ids are the float64 top-k wherever the float64 gap at the k-th place is wider than
      the fp32 chain's rounding;
  (c) the rows sent to the exact kernel are exactly the rows the numpy restatement flags: none in a filter case (the
      answer came from the filter and the exact rescore), every row built to overflow in an overflow case;
  (d) the raw tensor-core scores satisfy |a^ - S a| <= eps per element, a in float64, S and eps from the restated
      sweep_operands / row_eps without the rescore's terms: the premise of the filter (tcgen05's fp32 accumulation
      included) on hardware.
"""

import numpy as np
import pytest
import torch

import mma_filter_cases as mfc
from kge_helpers import make_product_model
from oracle import fullsort as ofs
from test_filter_proof_cpu import sweep_operands

pytestmark = pytest.mark.gpu

CASES = mfc.all_cases()
SHAPES = "afck"
DENSE_MAX = 30_000_000     # scores per dense check; larger cases are checked on a subset of rows
BOUND_ROWS = 48


def _params():
    out = []
    for cid, c in CASES.items():
        for cfg in SHAPES:   # a shape the case's K does not fit falls back to the plan's pick: run that one once
            if mfc.plan(c.model, c.d, len(c.Q), len(c.T), cfg)["cfg"] == cfg:
                out.append(pytest.param(cid, cfg, id=f"{cid}-{cfg}"))
    return out


def _product_model(case):
    n, nt, d = len(case.Q), len(case.T), case.d
    m = make_product_model(case.model, n + 1, nt, nt, 3, d)
    parts = [(case.Q[:, p * d:(p + 1) * d], case.T[:, p * d:(p + 1) * d]) for p in range(mfc.PARTS[case.model])]
    with torch.no_grad():
        for (q, t), un, en in zip(parts, type(m).USER_TABLES, type(m).ENTITY_TABLES):
            getattr(m, un).weight[1:n + 1].copy_(torch.from_numpy(q))
            getattr(m, en).weight[:nt].copy_(torch.from_numpy(t))
        # identity relations: the query of a row is its head row, exactly (x * 1, x + 0, cos 0 = 1, sin 0 = 0)
        for p, rn in enumerate(type(m).RELATION_TABLES):
            getattr(m, rn).weight.fill_(1.0 if case.model in ("DistMult", "ComplEx") and p == 0 else 0.0)
    m.invalidate_target_image()
    return m


def _csr(case):
    if case.hist is None:
        return None, None
    off = np.concatenate([[0], np.cumsum([len(h) for h in case.hist])])
    items = np.concatenate(case.hist) if off[-1] else np.zeros(0, dtype=np.int64)
    return torch.from_numpy(off).cuda(), torch.from_numpy(items.astype(np.int64)).cuda()


@pytest.mark.parametrize("case_id,cfg", _params())
def test_mma_filter_case(monkeypatch, case_id, cfg):
    monkeypatch.setenv("KGE_MMA_CFG", cfg)
    case = CASES[case_id]
    n, nt, k = len(case.Q), len(case.T), case.k
    m = _product_model(case)
    off, items = _csr(case)
    if case.kg:
        heads = torch.from_numpy(case.heads).cuda()
        rels = torch.ones(n, dtype=torch.long).cuda()
        call = lambda **kw: m.full_sort_topk(heads, k, off, items, case.mask_pad, relation_ids=rels, **kw)  # noqa: E731
    else:
        users = torch.arange(1, n + 1).cuda()
        call = lambda **kw: m.full_sort_topk(users, k, off, items, case.mask_pad, **kw)  # noqa: E731
    ids_c, sc_c = call(path="cuda")
    if case.kg:   # the link-prediction entry point itself
        ids_m, sc_m = m.full_sort_topk_kg(heads, rels, k, off, items, case.mask_pad, path="mma")
    else:
        ids_m, sc_m = call(path="mma")
    flagged = m._mma_last_fallback_rows
    ids_c, sc_c, ids_m, sc_m = (x.cpu().numpy() for x in (ids_c, sc_c, ids_m, sc_m))

    # (c) the rows the exact kernel re-did are the rows the restated filter flags
    res, pl = mfc.simulate(case, cfg, torch.cuda.get_device_properties(0).multi_processor_count)
    assert pl["cfg"] == cfg
    assert flagged == sum(r["flag"] is not None for r in res), [r["flag"] for r in res if r["flag"]][:8]
    if case.regime in ("filter", "survivors"):
        assert flagged == 0
    if case.regime == "overflow":
        assert flagged == case.expect["flagged"]

    # (a) bit-identical to the CUDA-core kernel
    np.testing.assert_array_equal(ids_m, ids_c)
    np.testing.assert_array_equal(sc_m, sc_c)

    # (b) the canonical top-k of the product's dense scores, and the float64 top-k where its gap is resolvable
    rows = np.arange(n) if n * nt <= DENSE_MAX else np.unique(np.r_[np.linspace(0, n - 1, DENSE_MAX // nt).astype(int),
                                                                      np.arange(n - 40, n)])
    if case.kg:
        dense = m.full_sort_predict_kg({"head_id": heads[rows], "relation_id": rels[rows]}).cpu().numpy().reshape(len(rows), nt)
    else:
        dense = m.full_sort_predict({"user_id": users[rows]}).cpu().numpy()
    masked = np.stack([np.where(case.masked(r), -np.inf, dense[i]) for i, r in enumerate(rows)])
    want_ids, want_sc = ofs.topk_canonical(masked, k)
    np.testing.assert_array_equal(ids_m[rows], want_ids)
    np.testing.assert_array_equal(sc_m[rows], want_sc)
    Q = case.Q[rows]
    a64 = case.exact(Q)
    P = case.T.shape[1]
    tmax = np.sqrt((case.T.astype(np.float64) ** 2).sum(1).max())
    with np.errstate(over="ignore", invalid="ignore"):
        nq = np.sqrt((Q.astype(np.float64) ** 2).sum(1))
        tol = (P + 2) * 2.0 ** -23 * ((nq + tmax) ** 2 if case.dist else nq * tmax)
    checked = 0
    for i, r in enumerate(rows):
        if not np.isfinite(tol[i]) or res[r]["flag"] == "bad":
            continue
        row = np.where(case.masked(r), -np.inf, a64[i])
        top = np.argsort(-row, kind="stable")
        if (~case.masked(r)).sum() > k and row[top[k - 1]] - row[top[k]] > tol[i]:
            assert set(ids_m[r]) == set(top[:k]), f"row {r}: not the float64 top-k"
            checked += 1
    if case.regime == "overflow":
        assert checked >= 1

    # (d) the error bound of the raw tensor-core scores
    if case.expect.get("no_bound"):
        return
    sel = rows[np.linspace(0, len(rows) - 1, min(BOUND_ROWS, len(rows))).astype(int)]
    if case.kg:
        _, _, raw = m.full_sort_topk(heads, k, off, items, case.mask_pad, relation_ids=rels, path="mma", _debug_scores=True)
    else:
        _, _, raw = call(path="mma", _debug_scores=True)
    raw = raw[torch.from_numpy(sel).cuda(), :nt].cpu().numpy().astype(np.float64)
    _, S, eps = sweep_operands(case.Q[sel], case.T, case.dist, sweep_only=True)   # (the tcgen05 sweep's terms only)
    a = case.exact(case.Q[sel])
    for i in range(len(sel)):
        if not np.isfinite(eps[i]):
            continue                                           # a row the sweep does not rank (flagged)
        err = np.abs(raw[i] * S[i] - S[i] * a[i]).max()
        assert err <= eps[i], f"row {sel[i]}: |a^ - S a| = {err:.4g} > eps = {eps[i]:.4g}"
