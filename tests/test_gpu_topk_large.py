"""Fused full-sort top-k above k = 128 (the large-k epilogue of kge_full_sort_topk), its metric sums and the paths
that evaluate through it.

Every top-k is checked for exact equality, ids and scores, against the canonical top-k of the product's own dense
full_sort_predict / full_sort_predict_kg rows after the trainer's masking: the standard test_gpu_scoring.py applies
to k <= 128."""

import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch

from kge_helpers import make_product_model
import gauc_oracle as go
from oracle import fullsort as ofs

pytestmark = pytest.mark.gpu


def _random_history(rng, n, n_targets, hist_max=60, few_row=None):
    """COO (rows, ids) of a random history per row; row `few_row` masks all but 3 targets."""
    hu, hi = [], []
    for row in range(n):
        nh = n_targets - 1 - 3 if row == few_row else int(rng.integers(0, min(hist_max, n_targets - 1)))
        items = rng.choice(np.arange(1, n_targets), size=nh, replace=False)
        hu += [row] * len(items)
        hi += list(items)
    return np.array(hu, dtype=np.int64), np.array(hi, dtype=np.int64)


def _check(m, queries, k, hu=None, hi=None, rels=None, path="cuda", mask_pad=True, **kw):
    """full_sort_topk(_kg) == topk_canonical(mask_scores(dense)) exactly; returns (ids, scores) on the host."""
    from hopwise_b200 import evaluator as ev

    n = len(queries)
    q = torch.as_tensor(np.asarray(queries)).cuda()
    ho = hv = None
    if hu is not None:
        ho, hv = ev.csr_from_pairs(hu, hi, n, "cuda")
    if rels is None:
        ids, sc = m.full_sort_topk(q, k, ho, hv, mask_pad=mask_pad, path=path, **kw)
        dense = m.full_sort_predict({"user_id": q}).cpu().numpy()
    else:
        r = torch.as_tensor(np.asarray(rels)).cuda()
        ids, sc = m.full_sort_topk_kg(q, r, k, ho, hv, mask_pad=mask_pad, path=path, **kw)
        dense = m.full_sort_predict_kg({"head_id": q, "relation_id": r}).cpu().numpy().reshape(n, -1)
    if mask_pad:
        masked = ofs.mask_scores(dense, hu, hi)
    else:
        masked = np.array(dense)
        if hu is not None and len(hu):
            masked[hu, hi] = -np.inf
    want_ids, want_sc = ofs.topk_canonical(masked, k)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    np.testing.assert_array_equal(ids, want_ids)
    np.testing.assert_array_equal(sc, want_sc)
    return ids, sc


# ---- 1. every model, k just above the list epilogue and well above it ---------------------------------------------
@pytest.mark.parametrize("name,d,I", [("TransE", 30, 3001), ("DistMult", 64, 5000), ("RotatE", 32, 4000),
                                      ("ComplEx", 20, 3500), ("TorusE", 64, 6000), ("TransH", 64, 9000),
                                      ("TransD", 32, 3000)])
@pytest.mark.parametrize("k", [129, 500])
def test_every_model_matches_dense(name, d, I, k):
    U, E, R = 400, I + 300, 9
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(7)
    users = np.arange(1, 301)
    hu, hi = _random_history(rng, len(users), I, few_row=5)   # row 5: fewer unmasked targets than k
    ids, sc = _check(m, users, k, hu, hi)
    assert np.isneginf(sc[5, 3:]).all() and (ids[5, 3:] == np.sort(ids[5, 3:])).all()


# ---- 2. edges ----------------------------------------------------------------------------------------------------
def test_k129_extends_k128():
    m = make_product_model("DistMult", 200, 4000, 4000, 5, 48)
    users = torch.arange(1, 101).cuda()
    ids128, sc128 = m.full_sort_topk(users, 128)
    ids129, sc129 = m.full_sort_topk(users, 129)
    np.testing.assert_array_equal(ids129[:, :128].cpu().numpy(), ids128.cpu().numpy())
    np.testing.assert_array_equal(sc129[:, :128].cpu().numpy(), sc128.cpu().numpy())


@pytest.mark.parametrize("name,I", [("TransE", 700), ("ComplEx", 1500)])
def test_k_equals_n_targets_sorts_the_whole_row(name, I):
    m = make_product_model(name, 100, I, I + 10, 5, 24)
    rng = np.random.default_rng(8)
    users = np.arange(1, 41)
    hu, hi = _random_history(rng, len(users), I, hist_max=200)
    ids, sc = _check(m, users, I, hu, hi)
    for r in range(len(users)):   # every target once; the masked ones last, in id order
        assert sorted(ids[r]) == list(range(I))
        masked = np.isneginf(sc[r])
        assert masked.sum() == 1 + (hu == r).sum()
        assert (np.diff(ids[r, masked]) > 0).all()


def test_zero_one_rows_and_k_above_n_targets():
    from hopwise_b200 import _abi

    m = make_product_model("DistMult", 50, 600, 600, 5, 16)
    ids, sc = m.full_sort_topk(torch.zeros(0, dtype=torch.long).cuda(), 300)
    assert ids.shape == (0, 300) and sc.shape == (0, 300)
    _check(m, np.array([7]), 300)
    _check(m, np.array([7]), 599, mask_pad=False)
    with pytest.raises(_abi.KgeError, match="larger than the number of targets"):
        m.full_sort_topk(torch.arange(1, 4).cuda(), 601)


# ---- 3. compaction and tie-breaking ------------------------------------------------------------------------------
def _ordered_model(I, sign, d=4, U=20):
    """DistMult whose score of target j is sign * j * (user's first weight): every target is exactly representable."""
    m = make_product_model("DistMult", U, I, I, 3, d)
    with torch.no_grad():
        u = torch.zeros(U, d)
        u[:, 0] = torch.arange(1, U + 1, dtype=torch.float32)
        e = torch.zeros(I, d)
        e[:, 0] = sign * torch.arange(I, dtype=torch.float32)
        m.user_embedding.weight.copy_(u.cuda())
        m.relation_embedding.weight.fill_(1.0)
        m.entity_embedding.weight.copy_(e.cuda())
    m.invalidate_target_image()
    return m


@pytest.mark.parametrize("sign", [1.0, -1.0])
@pytest.mark.parametrize("k", [129, 1000])
def test_monotone_scores(sign, k):
    """Rising scores: every tile beats the threshold and forces a compaction.  Falling: the first tiles fill the
    buffers and nothing later passes."""
    I = 20000
    m = _ordered_model(I, sign)
    rng = np.random.default_rng(9)
    users = np.arange(1, 11)
    hu, hi = _random_history(rng, len(users), I, hist_max=300)
    ids, _ = _check(m, users, k, hu, hi)
    if sign > 0:
        assert (np.diff(ids, axis=1) < 0).all()
    _check(m, np.arange(1, 4), k)   # a few rows: many target splits


@pytest.mark.parametrize("k", [200, 2500])
def test_duplicated_entity_rows_tie_by_id(k):
    I, d, U = 6000, 12, 60
    m = make_product_model("DistMult", U, I, I, 3, d)
    rng = np.random.default_rng(10)
    base = torch.from_numpy(rng.normal(size=(7, d)).astype(np.float32))
    with torch.no_grad():
        m.entity_embedding.weight.copy_(base[torch.arange(I) % 7].cuda())
    m.invalidate_target_image()
    users = np.arange(1, 51)
    hu, hi = _random_history(rng, len(users), I)
    _check(m, users, k, hu, hi)


# ---- 4. target splits ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [3, 12000])
def test_few_rows_and_more_than_one_wave(n):
    """3 rows: the targets are cut into many splits that the merge combines.  12,000 rows: 375 CTAs, more than the
    GPU holds at once."""
    I = 3000
    m = make_product_model("TransE", n + 1, I, I, 5, 32)
    rng = np.random.default_rng(12)
    users = np.arange(1, n + 1)
    hu, hi = _random_history(rng, n, I, hist_max=20)
    _check(m, users, 300, hu, hi)


# ---- 5. link prediction ----------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,d,E", [("TransE", 64, 5000), ("DistMult", 32, 3000), ("RotatE", 32, 4500),
                                      ("ComplEx", 64, 4000), ("TorusE", 30, 2500)])
def test_link_prediction(name, d, E):
    U, I, R = 50, 40, 11
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(13)
    n = 200
    heads = rng.integers(1, E, n)
    rels = rng.integers(1, R - 1, n)
    hu, hi = _random_history(rng, n, E, hist_max=40)
    _check(m, heads, 300, hu, hi, rels=rels)


@pytest.mark.parametrize("name", ["TransH", "TransD"])
def test_link_prediction_stays_refused_for_projected_models(name):
    m = make_product_model(name, 50, 100, 300, 5, 16)
    with pytest.raises(NotImplementedError):
        m.full_sort_topk_kg(torch.arange(1, 4).cuda(), torch.ones(3, dtype=torch.long).cuda(), 200)


# ---- 6. cfg4 size ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["DistMult", "ComplEx"])
def test_cfg4_size(name):
    I, n, k = 200_001, 256, 1000
    m = make_product_model(name, 5000, I, I, 3, 64)
    rng = np.random.default_rng(14)
    users = rng.integers(1, 5000, n)
    hist = np.sort(rng.choice(np.arange(1, I), (n, 50)), axis=1)
    hu = np.repeat(np.arange(n), 50)
    hi = hist.reshape(-1)
    keep = np.concatenate([[True], (np.diff(hu) != 0) | (np.diff(hi) != 0)])   # (choice draws per row may repeat)
    _check(m, users, k, hu[keep], hi[keep], path="auto")


# ---- 7. chunking -------------------------------------------------------------------------------------------------------
def test_workspace_budget_chunks_rows():
    from hopwise_b200 import _abi

    I, n, k = 5000, 700, 400
    m = make_product_model("ComplEx", n + 1, I, I, 5, 24)
    rng = np.random.default_rng(15)
    users = torch.arange(1, n + 1).cuda()
    hu, hi = _random_history(rng, n, I)
    from hopwise_b200 import evaluator as ev

    ho, hv = ev.csr_from_pairs(hu, hi, n, "cuda")
    whole = m.full_sort_topk(users, k, ho, hv)
    st = m._model_struct(False)
    need = _abi.lib().kge_full_sort_topk_workspace_bytes(C.byref(st), n, I, k)
    assert need > 0
    budget = need // 5   # several chunks
    chunked = m.full_sort_topk(users, k, ho, hv, workspace_budget=budget)
    np.testing.assert_array_equal(chunked[0].cpu().numpy(), whole[0].cpu().numpy())
    np.testing.assert_array_equal(chunked[1].cpu().numpy(), whole[1].cpu().numpy())
    one_row = m.full_sort_topk(users[:40], k, ho[:41], hv, workspace_budget=1)   # one row per call
    np.testing.assert_array_equal(one_row[0].cpu().numpy(), whole[0][:40].cpu().numpy())


# ---- 8. metrics -------------------------------------------------------------------------------------------------------
def test_hits_and_metric_sums_at_k300():
    from hopwise_b200 import evaluator as ev

    rng = np.random.default_rng(16)
    n, I, k = 1500, 4000, 300
    ids = np.stack([rng.permutation(I)[:k] for _ in range(n)])
    pos = [np.sort(rng.choice(I, int(rng.integers(1, 400)), replace=False)) for _ in range(n)]
    pu = np.concatenate([[r] * len(p) for r, p in enumerate(pos)])
    pi = np.concatenate(pos)
    po, pv = ev.csr_from_pairs(pu, pi, n, "cuda")
    rec = ev.topk_hits(torch.from_numpy(ids).cuda(), po, pv)
    want_rec = ofs.hits(ids, pu, pi, I)
    np.testing.assert_array_equal(rec.cpu().numpy(), want_rec)
    sums = ev.topk_metric_sums(rec).cpu().numpy()
    mats = ofs.metric_matrices(want_rec[:, :k], want_rec[:, k])
    for row, name in enumerate(ev.METRIC_ORDER):
        np.testing.assert_allclose(sums[row], mats[name].sum(axis=0), rtol=1e-12, err_msg=name)


def test_evaluate_full_sort_and_collector_at_large_k():
    from hopwise_b200 import evaluator as ev

    name, U, I, d = "TransE", 400, 2500, 64
    m = make_product_model(name, U, I, I + 100, 9, d)
    rng = np.random.default_rng(17)
    users = np.arange(1, 301)
    n = len(users)
    hu, hi = _random_history(rng, n, I)
    pos = [rng.choice(np.arange(1, I), int(rng.integers(1, 6)), replace=False) for _ in range(n)]
    pu = np.concatenate([[r] * len(p) for r, p in enumerate(pos)])
    pi = np.concatenate(pos)
    ho, hv = ev.csr_from_pairs(hu, hi, n, "cuda")
    po, pv = ev.csr_from_pairs(pu, pi, n, "cuda")
    t = torch.from_numpy(users).cuda()
    got = ev.evaluate_full_sort(m, t, ho, hv, po, pv, topk=(10, 200, 500), decimals=None, user_block=128, gauc=True)
    dense = m.full_sort_predict({"user_id": t}).cpu().numpy()
    masked = ofs.mask_scores(dense, hu, hi)
    top, _ = ofs.topk_canonical(masked, 500)
    want = ofs.metric_values(ofs.hits(top, pu, pi, I), topk=(10, 200, 500))
    assert list(got)[:15] == list(want)
    for key, v in want.items():
        np.testing.assert_allclose(got[key], v, rtol=1e-12, atol=1e-15, err_msg=key)
    np.testing.assert_allclose(got["gauc"], go.gauc(go.meanrank(masked, pu, pi)), rtol=1e-9)
    coll = ev.FusedCollector({"topk": [10, 200], "metrics": ["Recall", "GAUC"]})
    coll.eval_batch_collect(m, t, (hu, hi), pu, pi)
    struct = coll.get_data_struct()
    np.testing.assert_array_equal(struct["rec.topk"].cpu().numpy(), ofs.hits(top[:, :200], pu, pi, I))
    assert struct["rec.meanrank"].shape == (n, 3)


# ---- 9. the trainer --------------------------------------------------------------------------------------------------
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref as oref  # noqa: E402


def _run(use_gpu):
    from hopwise.config import Config
    from hopwise.data import create_dataset, data_preparation
    from hopwise.utils import get_model, get_trainer, init_seed

    cfg = {"embedding_size": 64, "train_batch_size": 2048, "epochs": 1, "show_progress": False, "eval_step": 1,
           "seed": 2024, "reproducibility": True, "topk": [10, 200]}
    config = Config(model="TransE", dataset="ml-100k", config_dict=dict(cfg, use_gpu=use_gpu,
                                                                       gpu_id="0" if use_gpu else ""))
    init_seed(config["seed"], config["reproducibility"])
    dataset = create_dataset(config)
    train_data, valid_data, test_data = data_preparation(config, dataset)
    init_seed(config["seed"], config["reproducibility"])
    model = get_model(config["model"])(config, train_data.dataset).to(config["device"])
    trainer = get_trainer(config["MODEL_TYPE"], config["model"])(config, model)
    trainer.fit(train_data, valid_data, saved=False, show_progress=False)
    return trainer, test_data, trainer.evaluate(test_data, load_best_model=False)


@pytest.mark.skipif(not oref.ref_available(), reason="oracle/_ref is not built")
def test_trainer_takes_the_fused_path_at_k200(tmp_path):
    oref.import_ref()
    import hopwise_b200.trainer as fused
    from hopwise.utils import KnowledgeEvaluationType

    torch.zeros(1, device="cuda")
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        _, _, want = _run(False)
        fused.install()
        try:
            trainer, test_data, got = _run(True)
            assert isinstance(trainer, fused.FusedKGTrainer)
            assert trainer._fused_plan(test_data, KnowledgeEvaluationType.REC) is not None
        finally:
            fused.uninstall()
    finally:
        os.chdir(cwd)
        if visible is None:
            os.environ.pop("CUDA_VISIBLE_DEVICES", None)
        else:
            os.environ["CUDA_VISIBLE_DEVICES"] = visible

    def flat(result):
        if isinstance(result, dict) and KnowledgeEvaluationType.REC in result:
            result = result[KnowledgeEvaluationType.REC]
            if isinstance(result, (list, tuple)):
                result = result[1]
        return {k: float(v) for k, v in result.items()}

    want, got = flat(want), flat(got)
    assert list(got) == list(want) and "recall@200" in got
    for key in want:
        assert abs(got[key] - want[key]) <= 3e-4, (key, got[key], want[key])
