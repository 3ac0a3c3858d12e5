"""Exact full-catalogue ranks of listed targets (kge_full_sort_rank_counts) and GAUC on the fused path.

Counts are checked for equality against numpy counts on the product's own dense scores (the top-k tests establish
that the dense scores and the sweep share one fp32 chain), meanrank / GAUC against the oracle model's scores up to
fp32 near-ties, and the whole GAUC pipeline against hopwise's own trainer where the reference package is built."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

from kge_helpers import make_oracle_model, make_product_model
import gauc_oracle as go
from oracle import fullsort as ofs

pytestmark = pytest.mark.gpu


def _csr(rows, n):
    """offsets, values sorted per row (duplicates kept) from a list of per-row id lists."""
    off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    vals = np.concatenate([np.sort(np.asarray(r, dtype=np.int64)) for r in rows]) if n else np.zeros(0, np.int64)
    return off, vals


def _numpy_counts(masked, pos_off, pos_items):
    greater = np.zeros(len(pos_items), np.int64)
    equal = np.zeros(len(pos_items), np.int64)
    for r in range(masked.shape[0]):
        row = masked[r]
        for i in range(pos_off[r], pos_off[r + 1]):
            j = pos_items[i]
            s = row[j]
            greater[i] = (row > s).sum()
            equal[i] = (row == s).sum()
    return greater, equal, np.isfinite(masked).sum(axis=1)


def _rows_of(off):
    return np.repeat(np.arange(len(off) - 1), np.diff(off))


def _random_rows(rng, n, n_targets, hist_max=60, pos_lo=1, pos_hi=6):
    hist = [np.sort(rng.choice(np.arange(1, n_targets), int(rng.integers(0, min(hist_max, n_targets - 1))),
                               replace=False)) for _ in range(n)]
    pos = [rng.choice(np.arange(0, n_targets), int(rng.integers(pos_lo, pos_hi)), replace=False) for _ in range(n)]
    return hist, pos


def _check_counts(m, queries, hist, pos, dense, rels=None, mask_pad=True):
    """full_sort_rank == numpy counts on the masked dense rows, exactly; equal >= 1 for every unmasked positive;
    full_sort_meanrank == the oracle's meanrank of the same rows."""
    n = len(queries)
    ho, hi = _csr(hist, n)
    po, pi = _csr(pos, n)
    dev = "cuda"
    t = lambda x: torch.from_numpy(np.asarray(x)).to(dev)   # noqa: E731
    g, e, u = m.full_sort_rank(t(queries), t(po), t(pi), t(ho), t(hi), mask_pad=mask_pad,
                               relation_ids=None if rels is None else t(rels))
    masked = ofs.mask_scores(dense, _rows_of(ho), hi) if mask_pad else np.array(dense)
    if not mask_pad:
        masked[_rows_of(ho), hi] = -np.inf
    wg, we, wu = _numpy_counts(masked, po, pi)
    np.testing.assert_array_equal(g.cpu().numpy(), wg)
    np.testing.assert_array_equal(e.cpu().numpy(), we)
    np.testing.assert_array_equal(u.cpu().numpy(), wu)
    unmasked = np.isfinite(masked[_rows_of(po), pi])
    assert (e.cpu().numpy()[unmasked] >= 1).all()
    if mask_pad:
        mr = m.full_sort_meanrank(t(queries), t(po), t(pi), t(ho), t(hi), relation_ids=None if rels is None else t(rels))
        np.testing.assert_array_equal(mr.cpu().numpy(), go.meanrank(masked, _rows_of(po), pi))
    return masked, (ho, hi, po, pi)


def _transh_planes(m, R, d, rng):
    w = torch.from_numpy(rng.uniform(-0.3, 0.3, (R, d)).astype(np.float32))
    with torch.no_grad():
        m.norm_vec.weight.copy_(w.cuda())
    return w


@pytest.mark.parametrize("name,d,I", [("TransE", 30, 1500), ("DistMult", 64, 2000), ("DistMult", 40, 100),
                                      ("RotatE", 48, 777), ("ComplEx", 18, 1599), ("ComplEx", 64, 3001),
                                      ("TorusE", 30, 1300), ("TorusE", 64, 2500), ("TransH", 64, 2000),
                                      ("TransH", 50, 9000), ("TransD", 30, 100), ("TransD", 64, 9000)])
def test_rank_counts_equal_dense_counts(name, d, I):
    """Every model, d % 4 != 0, fewer items than one 128-row tile, and TransH / TransD also at >= 8,192 items."""
    U, E, R = 400, I + 300, 9
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(11)
    if name == "TransH":
        _transh_planes(m, R, d, rng)
    users = np.arange(1, 301)
    hist, pos = _random_rows(rng, len(users), I)
    dense = m.full_sort_predict({"user_id": torch.from_numpy(users).cuda()}).cpu().numpy()
    _check_counts(m, users, hist, pos, dense)


@pytest.mark.parametrize("name,d", [("TransE", 30), ("DistMult", 64), ("RotatE", 48), ("ComplEx", 18),
                                    ("TorusE", 64)])
def test_rank_counts_link_prediction(name, d):
    U, I, E, R = 100, 500, 1400, 9
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(12)
    heads = rng.integers(1, E, 150)
    rels = rng.integers(1, R - 1, 150)
    hist, pos = _random_rows(rng, len(heads), E, hist_max=30)
    dense = m.full_sort_predict_kg({"head_id": torch.from_numpy(heads).cuda(),
                                    "relation_id": torch.from_numpy(rels).cuda()}).cpu().numpy()
    _check_counts(m, heads, hist, pos, dense, rels=rels)


def _scores_as_distmult(scores):
    """A DistMult model whose full-sort scores are exactly `scores` (as in test_gpu_scoring.py)."""
    n, I = scores.shape
    m = make_product_model("DistMult", n, I, I, 3, I)
    with torch.no_grad():
        m.user_embedding.weight.copy_(torch.from_numpy(scores))
        m.relation_embedding.weight.fill_(1.0)
        m.entity_embedding.weight.copy_(torch.eye(I))
    return m


def test_rank_counts_edge_rows():
    I = 1500
    m = make_product_model("DistMult", 50, I, I + 10, 5, 32)
    rng = np.random.default_rng(13)
    users = np.arange(1, 9)
    h = lambda k: np.sort(rng.choice(np.arange(1, I), k, replace=False))   # noqa: E731
    hist = [h(20), h(20), h(20), h(40), h(10), h(5), [], h(30)]
    pos = [[],                                                    # no positives
           [hist[1][3], 17, 900],                                 # a positive that is also in the history
           [0, 5, 1400],                                          # id 0 with mask_pad
           np.setdiff1d(np.arange(1, I), hist[3]),                # every unmasked item
           rng.choice(np.arange(0, I), 1200, replace=False),      # > 1,000 positives (thresholds in global memory)
           [7, 7, 7, 300, 300, 1001],                             # duplicate ids
           [1, 2, 3],
           rng.choice(np.arange(0, I), 16, replace=False)]        # exactly the shared-memory capacity
    dense = m.full_sort_predict({"user_id": torch.from_numpy(users).cuda()}).cpu().numpy()
    _check_counts(m, users, hist, pos, dense)
    _check_counts(m, users, hist, pos, dense, mask_pad=False)
    # the target splits: a handful of rows spread over many blocks of targets
    for n in (1, 2, 31, 33):
        users = np.arange(1, n + 1)
        hist, pos = _random_rows(rng, n, I)
        dense = m.full_sort_predict({"user_id": torch.from_numpy(users).cuda()}).cpu().numpy()
        _check_counts(m, users, hist, pos, dense)


def test_rank_counts_all_equal_scores():
    scores = np.zeros((3, 300), dtype=np.float32)
    scores[1, 10:20] = 1.0
    m = _scores_as_distmult(scores)
    hist = [[3, 4], [], [12, 150]]
    pos = [[1, 3, 5, 299], [10, 11, 50], [0, 12, 13, 14]]
    _, (ho, hi, po, pi) = _check_counts(m, np.arange(3), hist, pos, scores)
    t = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    g, e, u = m.full_sort_rank(t(np.arange(3)), t(po), t(pi), t(ho), t(hi))
    assert u.tolist() == [297, 299, 297]
    assert (g[0].item(), e[0].item()) == (0, 297)    # row 0, item 1: tied with every unmasked item
    assert (g[1].item(), e[1].item()) == (297, 3)    # row 0, item 3 (history): above it every unmasked item, tied
                                                     # with the three masked ones


def test_meanrank_and_gauc_against_oracle_scores():
    """The oracle model's fp32 scores differ from the product's in the last bits (another summation order): ranks
    may move where two targets score within fp32 rounding of each other.  Such rows are counted and bounded."""
    from hopwise_b200 import evaluator as ev

    name, U, I, E, R, d = "TransE", 400, 2500, 2600, 9, 64
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(14)
    users = np.arange(1, 301)
    hist, pos = _random_rows(rng, len(users), I)
    ho, hi = _csr(hist, len(users))
    po, pi = _csr(pos, len(users))
    t = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    got = m.full_sort_meanrank(t(users), t(po), t(pi), t(ho), t(hi)).cpu().numpy()
    with torch.no_grad():
        o_dense = ora.full_sort_predict({"user_id": torch.from_numpy(users)}).numpy()
    o_masked = ofs.mask_scores(o_dense, _rows_of(ho), hi)
    want = go.meanrank(o_masked, _rows_of(po), pi)
    np.testing.assert_array_equal(got[:, 1:], want[:, 1:])
    diff = np.flatnonzero(got[:, 0] != want[:, 0])
    for r in diff:
        near = 0
        for j in set(pi[po[r]:po[r + 1]].tolist()):
            s = o_masked[r, j]
            if np.isfinite(s):
                near += int((np.abs(o_masked[r] - s) <= 4e-6 * abs(s) + 1e-9).sum()) - 1
        assert abs(got[r, 0] - want[r, 0]) <= near + 1e-3, r
    assert len(diff) <= 0.05 * len(users)   # (a row moves when any of its 1-5 positives has a near-tie among 2,500)
    assert abs(go.gauc(got) - go.gauc(want)) < 1e-5
    # the library evaluator, in user blocks, reports the same GAUC
    res = ev.evaluate_full_sort(m, t(users), t(ho), t(hi), t(po), t(pi), topk=(10,), user_block=128, gauc=True)
    assert res["gauc"] == round(go.gauc(got), 4)
    assert list(res)[:5] == ["recall@10", "mrr@10", "ndcg@10", "hit@10", "precision@10"]
    coll = ev.FusedCollector({"topk": [10], "metrics": ["Recall", "GAUC"]})
    coll.eval_batch_collect(m, t(users), (_rows_of(ho), hi), _rows_of(po), pi)
    np.testing.assert_array_equal(coll.get_data_struct()["rec.meanrank"].cpu().numpy(), got)


def test_cfg4_item_side():
    """BASELINE config 4 on the item side: 200,001 items, 512 users, 50 history items each, 1-5 positives."""
    name, U, I, E, R, d = "DistMult", 5000, 200001, 200001, 3, 64
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(15)
    n = 512
    users = rng.integers(1, U, n)
    hist = [np.sort(rng.choice(np.arange(1, I), 50, replace=False)) for _ in range(n)]
    pos = [rng.choice(np.arange(1, I), int(rng.integers(1, 6)), replace=False) for _ in range(n)]
    ho, hi = _csr(hist, n)
    po, pi = _csr(pos, n)
    t = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    mr = m.full_sort_meanrank(t(users), t(po), t(pi), t(ho), t(hi)).cpu().numpy()
    assert (mr[:, 1] == I - 51).all()
    dense = m.full_sort_predict({"user_id": t(users[:8])}).cpu().numpy()
    _check_counts(m, users[:8], hist[:8], pos[:8], dense)
    masked = ofs.mask_scores(dense, _rows_of(ho[:9]), hi[: ho[8]])
    want = go.meanrank(masked, _rows_of(po[:9]), pi[: po[8]])
    np.testing.assert_array_equal(mr[:8], want)
    assert abs(go.gauc(mr[:8]) - go.gauc(want)) <= 1e-7


# ---- two GPUs: sharded GAUC --------------------------------------------------------------------------------------
EVAL_SHAPE = dict(U=1501, I=9001, E=9101, R=4, d=32)


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _gauc_inputs():
    rng = np.random.default_rng(41)
    n = 1237
    users = rng.integers(1, EVAL_SHAPE["U"], n)
    hist, pos = _random_rows(rng, n, EVAL_SHAPE["I"], hist_max=40)
    return users, _csr(hist, n), _csr(pos, n)


def _gauc_worker(rank, world, port, out_dir):
    import torch.distributed as dist

    from hopwise_b200.distributed import reduce_gauc_sums, shard_bounds
    from hopwise_b200.evaluator import gauc_sums

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        dev = f"cuda:{rank}"
        m = make_product_model("DistMult", device=dev, **EVAL_SHAPE)
        users, (hoff, hist), (poff, pos) = _gauc_inputs()
        lo, hi = shard_bounds(len(users), rank, world)
        t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(dev)   # noqa: E731
        mr = m.full_sort_meanrank(t(users[lo:hi]), t(poff[lo:hi + 1] - poff[lo]), t(pos[poff[lo]:poff[hi]]),
                                  t(hoff[lo:hi + 1] - hoff[lo]), t(hist[hoff[lo]:hoff[hi]]))
        total = reduce_gauc_sums(gauc_sums(mr))
        np.savez(os.path.join(out_dir, f"gauc{rank}.npz"), sums=total.cpu().numpy())
    finally:
        dist.destroy_process_group()


def test_two_rank_sharded_gauc_matches_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    from hopwise_b200.evaluator import gauc_from_sums, gauc_sums

    mp.spawn(_gauc_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "gauc0.npz"), np.load(tmp_path / "gauc1.npz")
    np.testing.assert_array_equal(r0["sums"], r1["sums"])
    users, (hoff, hist), (poff, pos) = _gauc_inputs()
    m = make_product_model("DistMult", device="cuda:0", **EVAL_SHAPE)
    t = lambda x: torch.from_numpy(x).cuda()   # noqa: E731
    want = gauc_sums(m.full_sort_meanrank(t(users), t(poff), t(pos), t(hoff), t(hist)))
    assert abs(gauc_from_sums(torch.from_numpy(r0["sums"]), None) - gauc_from_sums(want, None)) <= 1e-12


# ---- hopwise's own pipeline ----------------------------------------------------------------------------------------
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref as oref  # noqa: E402


def _run_gauc(use_gpu):
    from hopwise.config import Config
    from hopwise.data import create_dataset, data_preparation
    from hopwise.utils import get_model, get_trainer, init_seed

    cfg = {"embedding_size": 64, "train_batch_size": 2048, "epochs": 1, "show_progress": False, "eval_step": 1,
           "seed": 2024, "reproducibility": True, "metrics": ["Recall", "NDCG", "GAUC"]}
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
def test_gauc_through_hopwise_pipeline(tmp_path):
    """Config 1 (TransE, d = 64, ml-100k) with metrics [Recall, NDCG, GAUC]: FusedKGTrainer evaluates on the fused
    path and its dictionary equals hopwise's own KGTrainer on the CPU."""
    oref.import_ref()
    import hopwise_b200.trainer as fused
    from hopwise.utils import KnowledgeEvaluationType

    torch.zeros(1, device="cuda")
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    cwd = os.getcwd()
    os.chdir(tmp_path)
    try:
        _, _, want = _run_gauc(False)
        fused.install()
        try:
            trainer, test_data, got = _run_gauc(True)
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
    assert list(got) == list(want) and "gauc" in got
    for key in want:
        assert abs(got[key] - want[key]) <= 3e-4, (key, got[key], want[key])
