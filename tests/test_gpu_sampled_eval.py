"""Sampled evaluation (uni-N / pop-N) over candidate lists: kge_candidate_select against the dense route.

The dense route is what hopwise's trainer and collector do per batch: predict on the candidate rows, torch.full(-inf)
over [users, n_items], a scatter of the scores, then torch.topk (rec.topk) or a sort and _average_rank
(rec.meanrank).  The fused route scores the same rows with the same kernel, so every comparison here is exact."""

import os
import socket
import sys

import numpy as np
import pytest
import torch

from kge_helpers import make_product_model
import gauc_oracle as go

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MODEL_DIMS = {"TransE": 30, "DistMult": 64, "RotatE": 24, "ComplEx": 18, "TorusE": 32, "TransH": 64, "TransD": 20}


def _rows(rng, n_items, lens, n_pos=None):
    """Candidate lists of the given lengths (ids drawn with replacement from [1, n_items), so lists repeat ids) and
    positives: 1-5 distinct ids of each list (none for an empty list)."""
    cands, pos = [], []
    for L in lens:
        c = rng.integers(1, n_items, L)
        cands.append(c)
        u = np.unique(c)
        p = rng.choice(u, min(len(u), int(rng.integers(1, 6)) if n_pos is None else n_pos), replace=False) if L else []
        pos.append(np.sort(np.asarray(p, dtype=np.int64)))
    return cands, pos


EDGE_LENS = [1, 5, 101, 0, 505, 512, 513, 3000, 8192, 8193, 9000, 60000] + [101 * q for q in (1, 2, 3, 4, 5)] * 6


def _flat(users, cands, pos):
    n = len(cands)
    off = np.concatenate([[0], np.cumsum([len(c) for c in cands])]).astype(np.int64)
    user_col = np.repeat(np.asarray(users, dtype=np.int64), np.diff(off))
    item_col = np.concatenate(cands).astype(np.int64) if n else np.zeros(0, np.int64)
    poff = np.concatenate([[0], np.cumsum([len(p) for p in pos])]).astype(np.int64)
    pitems = np.concatenate(pos).astype(np.int64) if n else np.zeros(0, np.int64)
    return off, user_col, item_col, poff, pitems


def _dense(m, user_col, item_col, off, n_items):
    """predict -> full(-inf) -> scatter: the rows _neg_sample_batch_eval hands to the collector."""
    dev = "cuda"
    u, i = torch.from_numpy(user_col).to(dev), torch.from_numpy(item_col).to(dev)
    scores = m.predict({"user_id": u, "item_id": i})
    n = len(off) - 1
    row = torch.from_numpy(np.repeat(np.arange(n), np.diff(off))).to(dev)
    dense = torch.full((n, n_items), -np.inf, device=dev)
    dense[row, i] = scores
    return dense


def _pos_matrix(dense, poff, pitems):
    pm = torch.zeros_like(dense, dtype=torch.int)
    prow = torch.from_numpy(np.repeat(np.arange(len(poff) - 1), np.diff(poff))).cuda()
    pm[prow, torch.from_numpy(pitems).cuda()] = 1
    return pm


def _numpy_counts(row, items):
    return np.array([(row > row[j]).sum() for j in items]), np.array([(row == row[j]).sum() for j in items])


def _transh_planes(m, d, seed=3):
    if hasattr(m, "norm_vec"):
        w = np.random.default_rng(seed).uniform(-0.3, 0.3, tuple(m.norm_vec.weight.shape)).astype(np.float32)
        with torch.no_grad():
            m.norm_vec.weight.copy_(torch.from_numpy(w).cuda())


@pytest.mark.parametrize("k", [1, 10, 128, 200, 1000])
@pytest.mark.parametrize("name", list(MODEL_DIMS))
def test_candidate_topk_equals_dense_route(name, k):
    """ids and scores = a stable (score desc, id asc) sort of the dense rows; rec.topk = pos_matrix gathered at the
    dense route's own torch.topk ids.  Rows: single candidates, shorter than k, empty, both sides of every regime
    boundary (512 / 8,192 keys), above 50,000, and the 101..505 of uni100 with 1-5 positives."""
    from hopwise_b200.evaluator import topk_hits

    U, I, E, R = 300, 70001, 70101, 5
    m = make_product_model(name, U, I, E, R, MODEL_DIMS[name])
    _transh_planes(m, MODEL_DIMS[name])
    rng = np.random.default_rng(7)
    cands, pos = _rows(rng, I, EDGE_LENS)
    users = rng.integers(1, U, len(cands))
    off, uc, ic, poff, pitems = _flat(users, cands, pos)
    t = lambda x: torch.from_numpy(x).cuda()   # noqa: E731
    ids, scores = m.candidate_topk(t(uc), t(ic), t(off), k)
    dense = _dense(m, uc, ic, off, I)
    want_s, want_i = torch.sort(dense, dim=1, descending=True, stable=True)
    assert torch.equal(ids, want_i[:, :k])
    assert torch.equal(scores, want_s[:, :k])
    _, topk_idx = torch.topk(dense, k, dim=-1)
    pm = _pos_matrix(dense, poff, pitems)
    want_rec = torch.cat([torch.gather(pm, 1, topk_idx), pm.sum(dim=1, keepdim=True)], dim=1)
    assert torch.equal(topk_hits(ids, t(poff), t(pitems)), want_rec)
    # host offsets give the same result
    ids2, none = m.candidate_topk(t(uc), t(ic), torch.from_numpy(off), k, return_scores=False)
    assert none is None and torch.equal(ids2, ids)


@pytest.mark.parametrize("name", list(MODEL_DIMS))
def test_candidate_meanrank_equals_dense_sort(name):
    """rank counts = numpy counts on the dense rows; meanrank rows = average_rank on the sorted dense rows."""
    U, I, E, R = 300, 70001, 70101, 5
    m = make_product_model(name, U, I, E, R, MODEL_DIMS[name])
    _transh_planes(m, MODEL_DIMS[name])
    rng = np.random.default_rng(8)
    cands, pos = _rows(rng, I, EDGE_LENS)
    pos[11] = np.sort(rng.choice(np.unique(cands[11]), 1500, replace=False))   # many positives in a long row
    pos[5] = np.sort(np.concatenate([pos[5], [pos[5][0]], [I - 1]]))           # a duplicate and a non-candidate
    users = rng.integers(1, U, len(cands))
    off, uc, ic, poff, pitems = _flat(users, cands, pos)
    t = lambda x: torch.from_numpy(x).cuda()   # noqa: E731
    _, _, g, e, nu = m._candidate_select(t(uc), t(ic), t(off), 1, False, False, t(poff), t(pitems))
    dense = _dense(m, uc, ic, off, I).cpu().numpy()
    for r in range(len(cands)):
        wg, we = _numpy_counts(dense[r], pitems[poff[r]:poff[r + 1]])
        np.testing.assert_array_equal(g[poff[r]:poff[r + 1]].cpu().numpy(), wg)
        np.testing.assert_array_equal(e[poff[r]:poff[r + 1]].cpu().numpy(), we)
    np.testing.assert_array_equal(nu.cpu().numpy(), [len(np.unique(c)) for c in cands])
    mr = m.candidate_meanrank(t(uc), t(ic), t(off), t(poff), t(pitems)).cpu().numpy()
    prow = np.repeat(np.arange(len(cands)), np.diff(poff))
    np.testing.assert_array_equal(mr, go.meanrank(dense, prow, pitems))


@pytest.mark.parametrize("name", ["DistMult", "TransE"])
def test_all_equal_scores(name):
    """Zeroed tables: every candidate ties, so ids come in ascending order, then the padding; equal counts are the
    distinct candidates."""
    I = 600
    m = make_product_model(name, 20, I, I + 5, 4, 16)
    with torch.no_grad():
        for p in m.parameters():
            p.zero_()
    m.invalidate_target_image()
    cands = [np.array([9, 3, 3, 7, 500, 9]), np.array([4]), np.arange(599, 0, -1), np.array([], np.int64)]
    pos = [np.array([3, 500]), np.array([4]), np.array([1, 2, 599]), np.array([], np.int64)]
    off, uc, ic, poff, pitems = _flat([1, 2, 3, 4], cands, pos)
    t = lambda x: torch.from_numpy(x).cuda()   # noqa: E731
    ids, scores = m.candidate_topk(t(uc), t(ic), t(off), 8)
    assert ids.tolist() == [[3, 7, 9, 500, 0, 1, 2, 4], [4, 0, 1, 2, 3, 5, 6, 7], list(range(1, 9)),
                            list(range(8))]
    assert torch.isinf(scores[0, 4:]).all() and (scores[0, :4] == 0).all()
    _, _, g, e, nu = m._candidate_select(t(uc), t(ic), t(off), 8, False, False, t(poff), t(pitems))
    assert nu.tolist() == [4, 1, 599, 0]
    assert g.tolist() == [0, 0, 0, 0, 0, 0] and e.tolist() == [4, 4, 1, 599, 599, 599]
    dense = _dense(m, uc, ic, off, I)
    want_s, want_i = torch.sort(dense, dim=1, descending=True, stable=True)
    assert torch.equal(ids, want_i[:, :8])


def _loader_batches(rng, n_items, sizes, neg=100):
    """Batches shaped like NegSampleEvalDataLoader's: per user its positives then `neg` negatives per positive,
    (interaction, row_idx, positive_u, positive_i); `sizes` users per batch."""
    batches, uid = [], 1
    for b in sizes:
        users, items, row_idx, pu, pi = [], [], [], [], []
        for j in range(b):
            p = rng.choice(np.arange(1, n_items), int(rng.integers(1, 6)), replace=False)
            if j % 7 == 3:
                p = np.concatenate([p, p[:1]])           # a repeated test interaction
            c = np.concatenate([p, rng.integers(1, n_items, len(p) * neg)])
            users.append(np.full(len(c), uid))
            items.append(c)
            row_idx += [j] * len(c)
            pu += [j] * len(p)
            pi.append(p)
            uid += 1
        inter = {"user_id": torch.from_numpy(np.concatenate(users)), "item_id": torch.from_numpy(np.concatenate(items))}
        batches.append((inter, row_idx, torch.tensor(pu, dtype=torch.int64), torch.from_numpy(np.concatenate(pi))))
    return batches


def _dense_collect(m, batches, k, n_items):
    """trainer.py _neg_sample_batch_eval + collector.py rec.topk / rec.meanrank, batch by batch."""
    recs, mrs = [], []
    for inter, row_idx, pu, pi in batches:
        scores = m.predict({"user_id": inter["user_id"].cuda(), "item_id": inter["item_id"].cuda()})
        n = int(pu[-1]) + 1
        dense = torch.full((n, n_items), -np.inf, device="cuda")
        dense[torch.tensor(row_idx).cuda(), inter["item_id"].cuda()] = scores
        _, topk_idx = torch.topk(dense, k, dim=-1)
        pm = torch.zeros_like(dense, dtype=torch.int)
        pm[pu.cuda(), pi.cuda()] = 1
        # (int32 hits next to int64 sums promote to int64; kge_topk_metric_sums reads the int32 rows rec.topk holds)
        recs.append(torch.cat([torch.gather(pm, 1, topk_idx), pm.sum(dim=1, keepdim=True)], dim=1).to(torch.int32))
        mrs.append(go.meanrank(dense.cpu().numpy(), pu.numpy(), pi.numpy()))
    return torch.cat(recs), np.concatenate(mrs)


@pytest.mark.parametrize("name,block", [("DistMult", None), ("ComplEx", 37), ("TransD", 1000)])
def test_metric_dictionary_equals_dense_route(name, block):
    from hopwise_b200 import evaluator as ev

    I = 20001
    m = make_product_model(name, 400, I, I + 50, 4, 32)
    rng = np.random.default_rng(21)
    batches = _loader_batches(rng, I, [41, 3, 40, 1, 57, 12])
    want_rec, want_mr = _dense_collect(m, batches, 20, I)
    it = iter(batches)
    struct, nb = ev.collect_sampled(m, it, 20, meanrank=True, user_block=block)
    assert nb == len(batches) and next(it, None) is None
    assert torch.equal(struct["rec.topk"], want_rec)
    np.testing.assert_array_equal(struct["rec.meanrank"].cpu().numpy(), want_mr)
    assert torch.equal(struct["rec.users"].cpu(), torch.cat([b[0]["user_id"] for b in batches]))
    n = want_rec.shape[0]
    got = ev.metrics_from_sums(ev.topk_metric_sums(struct["rec.topk"]), n, [10, 20],
                               metrics=("recall", "mrr", "ndcg", "hit", "precision"))
    want = ev.metrics_from_sums(ev.topk_metric_sums(want_rec), n, [10, 20],
                                metrics=("recall", "mrr", "ndcg", "hit", "precision"))
    assert got == want
    assert ev.gauc_from_sums(ev.gauc_sums(struct["rec.meanrank"])) == round(go.gauc(want_mr), 4)


# ---- two GPUs ------------------------------------------------------------------------------------------------------
def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist

    from hopwise_b200 import evaluator as ev

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        dev = f"cuda:{rank}"
        m = make_product_model("DistMult", 400, 20001, 20051, 4, 32, device=dev)
        batches = _loader_batches(np.random.default_rng(31), 20001, [41, 40, 12, 33, 9, 40])
        struct, _ = ev.collect_sampled(m, batches[rank::world], 20, meanrank=True)
        sums = ev.topk_metric_sums(struct["rec.topk"])
        g = ev.gauc_sums(struct["rec.meanrank"])
        n = torch.tensor([struct["rec.topk"].shape[0]], dtype=torch.float64, device=dev)
        for x in (sums, g, n):
            dist.all_reduce(x)
        np.savez(os.path.join(out_dir, f"s{rank}.npz"), sums=sums.cpu().numpy(), g=g.cpu().numpy(), n=n.cpu().numpy())
    finally:
        dist.destroy_process_group()


def test_two_rank_sharded_sampled_eval_matches_single_gpu(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    from hopwise_b200 import evaluator as ev

    mp.spawn(_sharded_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    r0 = np.load(tmp_path / "s0.npz")
    m = make_product_model("DistMult", 400, 20001, 20051, 4, 32, device="cuda:0")
    struct, _ = ev.collect_sampled(m, _loader_batches(np.random.default_rng(31), 20001, [41, 40, 12, 33, 9, 40]), 20,
                                   meanrank=True)
    n = struct["rec.topk"].shape[0]
    assert int(r0["n"][0]) == n
    # (float64 sums over the users in another order: equal up to the last bits)
    want = ev.metrics_from_sums(ev.topk_metric_sums(struct["rec.topk"]), n, [10, 20], decimals=None)
    got = ev.metrics_from_sums(torch.from_numpy(r0["sums"]), n, [10, 20], decimals=None)
    assert list(got) == list(want) and all(abs(got[key] - want[key]) <= 1e-12 for key in want)
    want_g = ev.gauc_from_sums(ev.gauc_sums(struct["rec.meanrank"]), None)
    assert abs(ev.gauc_from_sums(torch.from_numpy(r0["g"]), None) - want_g) <= 1e-12


# ---- hopwise's own pipeline ----------------------------------------------------------------------------------------
sys.path.insert(0, ROOT)
from oracle import ref as oref  # noqa: E402


def _run_uni100(fused_eval):
    from hopwise.config import Config
    from hopwise.data import create_dataset, data_preparation
    from hopwise.utils import get_model, get_trainer, init_seed

    cfg = {"embedding_size": 64, "train_batch_size": 2048, "epochs": 1, "show_progress": False, "eval_step": 1,
           "seed": 2024, "reproducibility": True, "metrics": ["Recall", "MRR", "NDCG", "Hit", "Precision", "GAUC"],
           "topk": [10, 20], "eval_args": {"mode": "uni100"}, "kge_fused_eval": fused_eval, "use_gpu": True,
           "gpu_id": "0"}
    config = Config(model="TransE", dataset="ml-100k", config_dict=cfg)
    init_seed(config["seed"], config["reproducibility"])
    dataset = create_dataset(config)
    train_data, valid_data, test_data = data_preparation(config, dataset)
    init_seed(config["seed"], config["reproducibility"])
    model = get_model(config["model"])(config, train_data.dataset).to(config["device"])
    trainer = get_trainer(config["MODEL_TYPE"], config["model"])(config, model)
    trainer.fit(train_data, valid_data, saved=False, show_progress=False)
    valid = trainer.evaluate(valid_data, load_best_model=False)
    test = trainer.evaluate(test_data, load_best_model=False)
    state = np.random.get_state()
    # the epoch after the evaluations: its step losses depend on the negatives drawn from the same stream
    losses = []
    orig = model.train_step

    def record(interaction):
        loss = orig(interaction)
        losses.append(float(loss))
        return loss

    model.train_step = record
    trainer._train_epoch(train_data, 1)
    return trainer, valid_data, valid, test, state, losses


@pytest.mark.skipif(not oref.ref_available(), reason="oracle/_ref is not built")
def test_uni100_through_hopwise_pipeline(tmp_path):
    """TransE on ml-100k with eval_args.mode uni100: FusedKGTrainer with kge_fused_eval on and off gives the same
    validation and test dictionaries, leaves the same MT19937 state behind and trains the next epoch identically."""
    oref.import_ref()
    import hopwise_b200.trainer as fused
    from hopwise.utils import KnowledgeEvaluationType

    torch.zeros(1, device="cuda")
    visible = os.environ.get("CUDA_VISIBLE_DEVICES")
    cwd = os.getcwd()
    os.chdir(tmp_path)
    fused.install()
    try:
        off = _run_uni100(False)
        on = _run_uni100(True)
        assert on[0]._fused_sampled(on[1], KnowledgeEvaluationType.REC)
        assert not off[0]._fused_sampled(off[1], KnowledgeEvaluationType.REC)
    finally:
        fused.uninstall()
        os.chdir(cwd)
        if visible is None:
            os.environ.pop("CUDA_VISIBLE_DEVICES", None)
        else:
            os.environ["CUDA_VISIBLE_DEVICES"] = visible
    assert on[2] == off[2] and on[3] == off[3]
    assert "gauc" in str(on[3])
    s_on, s_off = on[4], off[4]
    assert s_on[0] == s_off[0] and np.array_equal(s_on[1], s_off[1]) and s_on[2:] == s_off[2:]
    assert on[5] == off[5] and len(on[5]) > 0
