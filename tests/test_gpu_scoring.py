"""Parity of predict / dense full-sort / fused full-sort top-k (through the C ABI) against the
oracle and the reference's golden Collector/Evaluator outputs.  Scores: 1e-5 relative (fp32);
top-k ids: exact under (score desc, id asc)."""

import numpy as np
import pytest
import torch

from conftest import load_golden
from kge_helpers import make_oracle_model, make_product_model
from oracle import fullsort as ofs

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _score_atol(x):
    return 1e-6 * float(np.abs(x).max())


@pytest.mark.parametrize(
    "name,d", [("TransE", 100), ("TransE", 30), ("DistMult", 64), ("RotatE", 48), ("ComplEx", 64), ("ComplEx", 18),
               ("RotatE", 256), ("TorusE", 100), ("TorusE", 30), ("TransH", 100), ("TransH", 30), ("TransH", 50),
               ("TransD", 100), ("TransD", 30)]
)
def test_scores_against_oracle(name, d):
    U, I, E, R = 150, 333, 700, 9
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(1)
    users = torch.from_numpy(rng.integers(1, U, 77))
    items = torch.from_numpy(rng.integers(0, I, 77))
    heads = torch.from_numpy(rng.integers(1, E, 41))
    rels = torch.from_numpy(rng.integers(1, R - 1, 41))
    tails = torch.from_numpy(rng.integers(1, E, 41))
    if name == "TransH":   # a hyperplane vector of ordinary size (xavier rows sum to ~0: the projection would be ~identity)
        w = torch.from_numpy(rng.uniform(-0.3, 0.3, (R, d)).astype(np.float32))
        with torch.no_grad():
            ora.norm_vec.weight.copy_(w)
            m.norm_vec.weight.copy_(w.cuda())
    with torch.no_grad():
        want_p = ora.predict({"user_id": users, "item_id": items}).numpy()
        want_fs = ora.full_sort_predict({"user_id": users}).numpy()
    got_p = m.predict({"user_id": users.cuda(), "item_id": items.cuda()}).cpu().numpy()
    got_fs = m.full_sort_predict({"user_id": users.cuda()}).cpu().numpy()
    np.testing.assert_allclose(got_p, want_p, rtol=RTOL, atol=_score_atol(want_p))
    np.testing.assert_allclose(got_fs, want_fs, rtol=RTOL, atol=_score_atol(want_fs))
    if name != "TransH":   # (transh.py scores users against items only)
        with torch.no_grad():
            want_pk = ora.predict_kg({"head_id": heads, "relation_id": rels, "tail_id": tails}).numpy()
        got_pk = m.predict_kg({"head_id": heads.cuda(), "relation_id": rels.cuda(), "tail_id": tails.cuda()}).cpu().numpy()
        np.testing.assert_allclose(got_pk, want_pk, rtol=RTOL, atol=_score_atol(want_pk))
    if name not in ("TransH", "TransD"):   # (TransD's dense KG full-sort is not mirrored, transd.py:192-217)
        with torch.no_grad():
            want_fk = ora.full_sort_predict_kg({"head_id": heads, "relation_id": rels}).numpy()
        got_fk = m.full_sort_predict_kg({"head_id": heads.cuda(), "relation_id": rels.cuda()}).cpu().numpy()
        np.testing.assert_allclose(got_fk, want_fk, rtol=RTOL, atol=_score_atol(want_fk))
    # the dense tensor is the caller's to mutate (trainer.py:731-734)
    t = m.full_sort_predict({"user_id": users.cuda()})
    t[:, 0] = -np.inf
    assert torch.isinf(t[:, 0]).all()


def _scores_as_distmult(scores):
    """A DistMult model whose full-sort scores are exactly `scores`: user rows = score rows,
    relation row = ones, entity table = identity (products by 1 and sums with 0 are exact)."""
    n, I = scores.shape
    m = make_product_model("DistMult", n, I, I, 3, I)
    with torch.no_grad():
        m.user_embedding.weight.copy_(torch.from_numpy(scores))
        m.relation_embedding.weight.fill_(1.0)
        m.entity_embedding.weight.copy_(torch.eye(I))
    return m


def test_golden_collector_and_metrics():
    """Reference Collector.eval_batch_collect + Evaluator.evaluate on masked random scores."""
    from hopwise_b200 import evaluator as ev

    g = load_golden("eval.npz")
    scores = g["scores"]
    n, I = scores.shape
    k = int(g["k"])
    m = _scores_as_distmult(scores)
    users = torch.arange(n).cuda()
    dense = m.full_sort_predict({"user_id": users}).cpu().numpy()
    np.testing.assert_array_equal(dense, scores)
    hist_off, hist_items = ev.csr_from_pairs(g["hist_u"], g["hist_i"], n, "cuda")
    ids, sc = m.full_sort_topk(users, k, hist_off, hist_items)
    masked = ofs.mask_scores(scores, g["hist_u"], g["hist_i"])
    ref_sc = np.take_along_axis(masked, g["topk_ids"], axis=1)
    # user 3 has fewer than k unmasked items: the tail of its reference list is -inf ties whose
    # order torch leaves unspecified; ids are compared on the finite prefix, scores everywhere
    finite = np.isfinite(ref_sc)
    assert not finite[3].all() and finite[np.arange(n) != 3].all()
    np.testing.assert_array_equal(ids.cpu().numpy()[finite], g["topk_ids"][finite])
    np.testing.assert_array_equal(sc.cpu().numpy(), ref_sc)
    want_ids, _ = ofs.topk_canonical(masked, k)
    np.testing.assert_array_equal(ids.cpu().numpy(), want_ids)            # canonical order incl. the -inf tail
    pos_off, pos_items = ev.csr_from_pairs(g["pos_u"], g["pos_i"], n, "cuda")
    rec = ev.topk_hits(ids, pos_off, pos_items)
    np.testing.assert_array_equal(rec.cpu().numpy(), g["rec_topk"])
    sums = ev.topk_metric_sums(rec).cpu().numpy()
    for row, name in enumerate(ev.METRIC_ORDER):
        np.testing.assert_allclose(sums[row] / n, g["matrix/" + name].mean(axis=0), rtol=1e-12, atol=1e-15)
    got = ev.metrics_from_sums(torch.from_numpy(sums), n, [5, k], decimals=4)
    want = dict(zip([str(x) for x in g["metric_names"]], g["metric_values"]))
    assert set(got) == set(want)
    for key, v in want.items():
        assert got[key] == pytest.approx(v, abs=1e-12), key
    # the collector twin, fed with the loader's COO tuples in two batches
    coll = ev.FusedCollector({"topk": [5, k]})
    for lo, hi in ((0, 17), (17, n)):
        hsel = (g["hist_u"] >= lo) & (g["hist_u"] < hi)
        psel = (g["pos_u"] >= lo) & (g["pos_u"] < hi)
        coll.eval_batch_collect(m, users[lo:hi], (g["hist_u"][hsel] - lo, g["hist_i"][hsel]),
                                g["pos_u"][psel] - lo, g["pos_i"][psel])
    struct = coll.get_data_struct()
    np.testing.assert_array_equal(struct["rec.topk"].cpu().numpy(), g["rec_topk"])


def test_reference_metric_known_answers():
    """/root/reference/tests/metrics/test_topk_metrics.py:26-108 through the metric kernel."""
    from hopwise_b200 import evaluator as ev

    pos_idx = np.array([[0, 0, 0], [1, 1, 1], [1, 0, 1], [0, 0, 1]], dtype=np.int32)
    pos_len = np.array([1, 3, 4, 2], dtype=np.int32)
    rec = torch.from_numpy(np.concatenate([pos_idx, pos_len[:, None]], axis=1)).cuda()
    sums = ev.topk_metric_sums(rec).cpu().numpy()
    want = {
        "hit": np.array([[0, 0, 0], [1, 1, 1], [1, 1, 1], [0, 0, 1]]),
        "mrr": np.array([[0, 0, 0], [1, 1, 1], [1, 1, 1], [0, 0, 1 / 3]]),
        "recall": np.array([[0, 0, 0], [1 / 3, 2 / 3, 3 / 3], [1 / 4, 1 / 4, 2 / 4], [0, 0, 1 / 2]]),
        "precision": np.array([[0, 0, 0], [1 / 1, 2 / 2, 3 / 3], [1 / 1, 1 / 2, 2 / 3], [0, 0, 1 / 3]]),
        "ndcg": np.array(
            [
                [0, 0, 0],
                [1, 1, 1],
                [1, (1 / np.log2(2) / (1 / np.log2(2) + 1 / np.log2(3))),
                 ((1 / np.log2(2) + 1 / np.log2(4)) / (1 / np.log2(2) + 1 / np.log2(3) + 1 / np.log2(4)))],
                [0, 0, (1 / np.log2(4) / (1 / np.log2(2) + 1 / np.log2(3)))],
            ]
        ),
    }
    for row, name in enumerate(ev.METRIC_ORDER):
        np.testing.assert_allclose(sums[row], want[name].sum(axis=0), rtol=1e-12, err_msg=name)


@pytest.mark.parametrize("name,d,I,k", [("TransE", 100, 3001, 10), ("DistMult", 64, 5000, 20), ("ComplEx", 32, 1599, 10),
                                        ("RotatE", 64, 777, 50), ("TransE", 22, 130, 128), ("TorusE", 64, 2500, 20),
                                        ("TransH", 64, 2000, 20), ("TransD", 64, 2500, 20), ("TransD", 64, 9000, 20),
                                        ("TransH", 64, 9000, 20)])   # (>= 8192 items: "auto" takes the tensor cores)
def test_topk_against_oracle(name, d, I, k):
    U, E, R = 400, I + 500, 9
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(4)
    users = np.arange(1, 301)
    hist_u, hist_i = [], []
    for row in range(len(users)):
        nh = int(rng.integers(0, 60)) if row != 5 else I - 1 - 3   # row 5: fewer than k unmasked items
        items = rng.choice(np.arange(1, I), size=min(nh, I - 1), replace=False)
        hist_u += [row] * len(items)
        hist_i += list(items)
    from hopwise_b200 import evaluator as ev

    hist_off, hist_items = ev.csr_from_pairs(np.array(hist_u), np.array(hist_i), len(users), "cuda")
    ids, sc = m.full_sort_topk(torch.from_numpy(users).cuda(), k, hist_off, hist_items)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    # (1) self-consistency: canonical top-k of the product's own dense scores, exactly
    dense = m.full_sort_predict({"user_id": torch.from_numpy(users).cuda()}).cpu().numpy()
    masked = ofs.mask_scores(dense, np.array(hist_u), np.array(hist_i))
    want_ids, want_sc = ofs.topk_canonical(masked, k)
    np.testing.assert_array_equal(ids, want_ids)
    np.testing.assert_array_equal(sc, want_sc)
    # (2) against the oracle's scores: ids equal except where the oracle's own gap is within
    # fp32 rounding of the two summation orders (SURVEY.md H6); count and bound those
    with torch.no_grad():
        o_dense = ora.full_sort_predict({"user_id": torch.from_numpy(users)}).numpy()
    o_masked = ofs.mask_scores(o_dense, np.array(hist_u), np.array(hist_i))
    o_ids, o_sc = ofs.topk_canonical(o_masked, k)
    diff = ids != o_ids
    if diff.any():
        rows, cols = np.nonzero(diff)
        a = np.take_along_axis(o_masked, ids, axis=1)[rows, cols]
        b = o_sc[rows, cols]
        finite = np.isfinite(a) & np.isfinite(b)
        assert np.all(np.abs(a[finite] - b[finite]) <= 4e-6 * np.abs(b[finite]) + 1e-9), "top-k differs beyond fp32 ties"
        assert diff.mean() < 0.01
    fin = np.isfinite(o_sc)
    np.testing.assert_allclose(sc[fin & ~diff], o_sc[fin & ~diff], rtol=RTOL, atol=_score_atol(o_sc[fin]))


def test_topk_without_history_and_small_batches():
    name, U, I, E, R, d, k = "DistMult", 50, 999, 1200, 5, 40, 10
    m = make_product_model(name, U, I, E, R, d)
    for n in (1, 2, 31, 33):   # the reference evaluates max(eval_batch_size // I, 1) users per batch
        users = torch.arange(1, n + 1).cuda()
        ids, sc = m.full_sort_topk(users, k)
        dense = m.full_sort_predict({"user_id": users}).cpu().numpy()
        want_ids, want_sc = ofs.topk_canonical(ofs.mask_scores(dense), k)
        np.testing.assert_array_equal(ids.cpu().numpy(), want_ids)
        np.testing.assert_array_equal(sc.cpu().numpy(), want_sc)
    ids, _ = m.full_sort_topk(torch.arange(1, 4).cuda(), k, mask_pad=False)
    dense = m.full_sort_predict({"user_id": torch.arange(1, 4).cuda()}).cpu().numpy()
    np.testing.assert_array_equal(ids.cpu().numpy(), ofs.topk_canonical(dense, k)[0])


def test_topk_ties_break_by_id():
    """All-equal scores: the canonical order is ascending item id (after the masked pad item)."""
    scores = np.zeros((3, 64), dtype=np.float32)
    scores[1, 10:20] = 1.0
    m = _scores_as_distmult(scores)
    ids, _ = m.full_sort_topk(torch.arange(3).cuda(), 12)
    ids = ids.cpu().numpy()
    np.testing.assert_array_equal(ids[0], np.arange(1, 13))
    np.testing.assert_array_equal(ids[1], np.concatenate([np.arange(10, 20), [1, 2]]))


def test_full_size_topk_properties():
    """BASELINE config 4 shape on the item side (200k items, k=20), a block of users: sortedness,
    uniqueness, no masked id, score consistency with predict(), and threshold property."""
    name, U, I, E, R, d, k = "DistMult", 5000, 200001, 200001, 3, 64, 20
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(6)
    n = 512
    users = torch.from_numpy(rng.integers(1, U, n)).cuda()
    hist = np.sort(rng.integers(1, I, (n, 50)), axis=1)
    hist_off = torch.arange(0, 50 * n + 1, 50, dtype=torch.long).cuda()
    hist_items = torch.from_numpy(hist.reshape(-1)).cuda()
    ids, sc = m.full_sort_topk(users, k, hist_off, hist_items)
    ids_c, sc_c = ids.cpu().numpy(), sc.cpu().numpy()
    assert np.all(np.diff(sc_c, axis=1) <= 0)
    assert all(len(set(r)) == k for r in ids_c)
    assert np.all(ids_c != 0)
    assert not any(set(r) & set(h) for r, h in zip(ids_c, hist))
    p = m.predict({"user_id": users.repeat_interleave(k), "item_id": ids.reshape(-1)}).reshape(n, k)
    np.testing.assert_allclose(p.cpu().numpy(), sc_c, rtol=1e-5, atol=1e-9)
    # nothing unmasked beats the k-th score: check 8 users against their dense rows
    dense = m.full_sort_predict({"user_id": users[:8]}).cpu().numpy()
    masked = np.array(dense)
    masked[:, 0] = -np.inf
    for r in range(8):
        masked[r, hist[r]] = -np.inf
        assert (masked[r] > sc_c[r, -1]).sum() == k - 1
        np.testing.assert_array_equal(ids_c[r], ofs.topk_canonical(masked[r : r + 1], k)[0][0])


# ---- tensor-core (tcgen05) path: identical results to the fp32 CUDA-core path -----------------------
def _f16_round(x):
    """fp16 rounding after the power-of-two scaling of csrc/mma_topk.cu (largest element into [2^7, 2^8))."""
    x = np.ascontiguousarray(x, dtype=np.float32)
    e = 7 - int(np.floor(np.log2(np.abs(x).max())))
    return np.ldexp(np.ldexp(x, e).astype(np.float16).astype(np.float32), -e)


@pytest.mark.parametrize("name,d", [("DistMult", 64), ("ComplEx", 32), ("TransE", 100), ("RotatE", 24)])
def test_mma_raw_scores_match_fp16_emulation(name, d):
    """The raw tensor-core scores (unscaled by the kernel's debug dump) equal q^ . t^ (scaled fp16 operands, fp32
    accumulation): checks the operand layouts, descriptors, scaling and the TMEM read-back independently of the
    top-k logic."""
    U, I, E, R, k = 400, 1000, 1300, 7, 10
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    users = torch.arange(1, 301)
    ids, sc, raw = m.full_sort_topk(users.cuda(), k, path="mma", _debug_scores=True)
    raw = raw.cpu().numpy()[:, :I]
    sd = {k_: v.numpy().astype(np.float64) for k_, v in ora.state_dict().items()}
    un, en, rn = [[sd[t + ".weight"] for t in names] for names in
                  (type(m).USER_TABLES, type(m).ENTITY_TABLES, type(m).RELATION_TABLES)]
    u = [t[users.numpy()].astype(np.float32) for t in un]
    r = [t[m._ui_row(True)].astype(np.float32) for t in rn]
    if name == "TransE":
        q = [u[0] + r[0]]
    elif name == "DistMult":
        q = [u[0] * r[0]]
    elif name == "RotatE":
        c, s = np.cos(r[0]), np.sin(r[0])
        q = [c * u[0] - s * u[1], c * u[1] + s * u[0]]
    else:
        q = [u[0] * r[0], u[1] * r[0] + u[0] * r[1] - u[1] * r[1]]
    qc = np.concatenate(q, axis=1)
    tc = np.concatenate([t[:I].astype(np.float32) for t in en], axis=1)
    want = np.stack([_f16_round(row) for row in qc]).astype(np.float64) @ _f16_round(tc).astype(np.float64).T
    if name in ("TransE", "RotatE"):
        want = want - 0.5 * (tc.astype(np.float64) ** 2).sum(1)[None, :]
    scale = np.abs(want).max()
    np.testing.assert_allclose(raw, want, rtol=0, atol=3e-4 * scale)   # q of RotatE differs by sincos ulps
    assert np.abs(raw - want).mean() < 3e-5 * scale


@pytest.mark.parametrize("name,d,I,k", [("DistMult", 64, 20000, 20), ("ComplEx", 64, 9000, 20), ("TransE", 100, 12000, 10),
                                        ("RotatE", 32, 8200, 32), ("DistMult", 50, 4099, 5)])
def test_mma_topk_equals_cuda_core_topk(name, d, I, k):
    U, E, R = 900, I + 100, 6
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(8)
    n = 700
    users = torch.from_numpy(rng.integers(1, U, n)).cuda()
    lens = rng.integers(0, 80, n)
    lens[7] = I - 1 - 3              # fewer than k unmasked items -> must be recomputed exactly
    hist = [np.sort(rng.choice(np.arange(1, I), size=int(l), replace=False)) for l in lens]
    off = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).cuda()
    items = torch.from_numpy(np.concatenate(hist)).cuda()
    ids_c, sc_c = m.full_sort_topk(users, k, off, items, path="cuda")
    ids_m, sc_m = m.full_sort_topk(users, k, off, items, path="mma")
    assert m._mma_last_fallback_rows >= 1
    assert m._mma_last_fallback_rows < 0.1 * n   # flagged rows are rare (k = 32 is the tightest case)
    np.testing.assert_array_equal(ids_m.cpu().numpy(), ids_c.cpu().numpy())
    np.testing.assert_array_equal(sc_m.cpu().numpy(), sc_c.cpu().numpy())
    # no history, no pad masking, a user count that is not a multiple of the CTA tile
    ids_c, sc_c = m.full_sort_topk(users[:300], k, mask_pad=False, path="cuda")
    ids_m, sc_m = m.full_sort_topk(users[:300], k, mask_pad=False, path="mma")
    np.testing.assert_array_equal(ids_m.cpu().numpy(), ids_c.cpu().numpy())
    np.testing.assert_array_equal(sc_m.cpu().numpy(), sc_c.cpu().numpy())


@pytest.mark.parametrize("cfg,name,d,I,k", [("a", "DistMult", 64, 20000, 20), ("f", "DistMult", 64, 20000, 20),
                                            ("c", "DistMult", 64, 20000, 20), ("f", "RotatE", 20, 9000, 10),
                                            ("", "RotatE", 120, 8300, 10), ("", "ComplEx", 128, 8300, 20),
                                            ("k", "DistMult", 64, 20000, 20), ("", "RotatE", 128, 8300, 10),
                                            ("", "RotatE", 256, 8300, 20), ("", "TransE", 500, 8300, 20),
                                            ("", "ComplEx", 300, 8300, 5)])
def test_mma_tile_shapes(monkeypatch, cfg, name, d, I, k):
    """Every sweep shape (csrc/mma_topk.cu plan_mma: a = two CTAs per SM, f = column-sliced single CTA, c = 64-wide
    tiles for K > 195, k = 128-row CTAs with K-chunked tiles for K > 256: RotatE d = 128 / 256 are K = 272 / 528) gives
    the CUDA-core kernel's ids and scores bit for bit; "" = the shape the plan picks (K = 256 lands on c)."""
    if cfg:
        monkeypatch.setenv("KGE_MMA_CFG", cfg)
    else:
        monkeypatch.delenv("KGE_MMA_CFG", raising=False)
    U, E, R = 700, I + 50, 5
    m = make_product_model(name, U, I, E, R, d)   # fresh model: the cached target image depends on the tile width
    rng = np.random.default_rng(11)
    n = 600
    users = torch.from_numpy(rng.integers(1, U, n)).cuda()
    lens = rng.integers(0, 60, n)
    hist = [np.sort(rng.choice(np.arange(1, I), size=int(l), replace=False)) for l in lens]
    off = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).cuda()
    items = torch.from_numpy(np.concatenate(hist)).cuda()
    ids_c, sc_c = m.full_sort_topk(users, k, off, items, path="cuda")
    ids_m, sc_m = m.full_sort_topk(users, k, off, items, path="mma")
    assert m._mma_last_fallback_rows < 0.1 * n
    np.testing.assert_array_equal(ids_m.cpu().numpy(), ids_c.cpu().numpy())
    np.testing.assert_array_equal(sc_m.cpu().numpy(), sc_c.cpu().numpy())


def test_mma_topk_trained_like_weights_and_cache_invalidation():
    """Heavy-tailed item norms (a few items dominate) and a weight update between calls."""
    name, U, I, E, R, d, k = "DistMult", 600, 30000, 30000, 4, 64, 20
    m = make_product_model(name, U, I, E, R, d)
    with torch.no_grad():
        m.entity_embedding.weight[100:130] *= 25.0
        m.entity_embedding.weight[5000:5010] *= -40.0
    users = torch.arange(1, 513).cuda()
    for _ in range(2):
        ids_c, sc_c = m.full_sort_topk(users, k, path="cuda")
        ids_m, sc_m = m.full_sort_topk(users, k, path="mma")
        np.testing.assert_array_equal(ids_m.cpu().numpy(), ids_c.cpu().numpy())
        np.testing.assert_array_equal(sc_m.cpu().numpy(), sc_c.cpu().numpy())
        with torch.no_grad():
            m.entity_embedding.weight.mul_(-1.0)   # the cached operand image must be rebuilt


# ---- link-prediction twin: (head entity, relation) rows against every entity -------------------------------
@pytest.mark.parametrize("name,d,E,k,path", [("TransE", 64, 9000, 10, "mma"), ("DistMult", 32, 2000, 10, "cuda"),
                                             ("RotatE", 32, 8500, 20, "mma"), ("ComplEx", 64, 8300, 5, "mma"),
                                             ("ComplEx", 16, 700, 10, "auto")])
def test_topk_kg_against_dense_and_oracle(name, d, E, k, path):
    """full_sort_topk_kg = canonical top-k of the product's own full_sort_predict_kg after the trainer's
    masking (trainer.py:731-734), and of the oracle's up to fp32 ties; CUDA-core and tensor-core paths."""
    U, I, R = 50, 40, 11
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    rng = np.random.default_rng(11)
    n = 260
    heads = rng.integers(1, E, n)
    rels = rng.integers(1, R - 1, n)
    hist_u, hist_i = [], []
    for row in range(n):
        tails = rng.choice(np.arange(1, E), size=int(rng.integers(0, 40)), replace=False)
        hist_u += [row] * len(tails)
        hist_i += list(tails)
    from hopwise_b200 import evaluator as ev

    hist_off, hist_items = ev.csr_from_pairs(np.array(hist_u), np.array(hist_i), n, "cuda")
    ids, sc = m.full_sort_topk_kg(torch.from_numpy(heads).cuda(), torch.from_numpy(rels).cuda(), k, hist_off, hist_items,
                                  path=path)
    ids, sc = ids.cpu().numpy(), sc.cpu().numpy()
    batch = {"head_id": torch.from_numpy(heads).cuda(), "relation_id": torch.from_numpy(rels).cuda()}
    dense = m.full_sort_predict_kg(batch).cpu().numpy().reshape(n, E)
    masked = ofs.mask_scores(dense, np.array(hist_u), np.array(hist_i))
    want_ids, want_sc = ofs.topk_canonical(masked, k)
    np.testing.assert_array_equal(ids, want_ids)
    np.testing.assert_array_equal(sc, want_sc)
    with torch.no_grad():
        o_dense = ora.full_sort_predict_kg({"head_id": torch.from_numpy(heads), "relation_id": torch.from_numpy(rels)}).numpy()
    np.testing.assert_allclose(dense, o_dense, rtol=RTOL, atol=_score_atol(o_dense))
    o_ids, o_sc = ofs.topk_canonical(ofs.mask_scores(o_dense, np.array(hist_u), np.array(hist_i)), k)
    assert (ids != o_ids).mean() < 0.01


def test_toruse_scores_with_weights_beyond_the_unit_interval():
    """TorusE scores take frac() of every embedding (toruse.py:66-76; torch.frac keeps the sign): weights of magnitude
    up to 3 exercise the truncation on both signs, on all four scoring entry points and the CUDA-core top-k; the
    tensor-core path refuses the model (its scorer is not a contraction)."""
    U, I, E, R, d = 90, 9000, 9100, 7, 40
    ora = make_oracle_model("TorusE", U, I, E, R, d)
    m = make_product_model("TorusE", U, I, E, R, d)
    rng = np.random.default_rng(8)
    with torch.no_grad():
        for (_, po), (_, pp) in zip(ora.named_parameters(), m.named_parameters()):
            w = torch.from_numpy(rng.uniform(-3, 3, tuple(po.shape)).astype(np.float32))
            po.copy_(w)
            pp.copy_(w.cuda())
    m.invalidate_target_image()
    users = torch.from_numpy(rng.integers(1, U, 64))
    items = torch.from_numpy(rng.integers(0, I, 64))
    with torch.no_grad():
        want_p = ora.predict({"user_id": users, "item_id": items}).numpy()
        want_fs = ora.full_sort_predict({"user_id": users}).numpy()
    got_p = m.predict({"user_id": users.cuda(), "item_id": items.cuda()}).cpu().numpy()
    got_fs = m.full_sort_predict({"user_id": users.cuda()}).cpu().numpy()
    # sums of d terms of magnitude <= 1 with both signs: the absolute floor is that of the terms, not of the sum
    np.testing.assert_allclose(got_p, want_p, rtol=RTOL, atol=4 * d * 1e-6)
    np.testing.assert_allclose(got_fs, want_fs, rtol=RTOL, atol=4 * d * 1e-6)
    ids, sc = m.full_sort_topk(users.cuda(), 20)           # "auto": 9,000 targets would take tcgen05 for a contraction
    want_ids, want_sc = ofs.topk_canonical(ofs.mask_scores(got_fs), 20)
    np.testing.assert_array_equal(ids.cpu().numpy(), want_ids)
    np.testing.assert_array_equal(sc.cpu().numpy(), want_sc)
    with pytest.raises(Exception):
        m.full_sort_topk(users.cuda(), 20, path="mma")
