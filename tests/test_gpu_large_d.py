"""Embedding sizes past the 512 / 256 layouts on the B200: the three row layouts (4, 32, 8), (1, 32, 16) and
(1, 32, 32) and the 16-row query block of the full-sort tile kernel, against float64 closed forms.

The ladder (tests/test_large_d_cpu.py) reaches every new layout at its first and last chunk count, with partial and
empty last chunks.  The checks are test_gpu_row_layouts.py's: the gradient bound is per element, from the sum of
each contributing pair's largest term; the optimiser kernels are fed the kernel's own gradient.  Scoring results of
the fused paths must equal the canonical top-k / rank counts of the model's own dense rows exactly."""

import os
import socket

import numpy as np
import pytest
import torch

from kge_helpers import assert_weights_close, make_product_model, random_batch, to_device_batch
from oracle import fullsort as ofs
from test_gpu_row_layouts import (FAMILIES, HINGE, N_ISO, RMSPROP_ALPHA, E, I, R, U, _batch,
                                  _check_adam_first_step, _check_against_dense, _check_forward, _check_scores,
                                  _dense_adam_step, _f64, _forward_state, _init_tables, _run_three_steps,
                                  _set_margin_and_resample, _tables)
from test_large_d_cpu import LARGE_D_LADDER, pick_rowcfg

pytestmark = pytest.mark.gpu

MODELS = ("TransE", "RotatE", "DistMult", "ComplEx", "TorusE", "TransH", "TransD")
TRAIN_KINDS = ("TransE", "DistMult", "RotatE", "ComplEx", "TransH", "TransD")   # (TorusE trains as TransE)
# ladder points that run K negatives (k_rec = 2, k_kg = 3): at least one per layout
K_NEG_D = (301, 600, 1021)


def _sizes(d, n_sm, idx):
    """(n_rec, n_kg): one half runs two passes of the grid-stride loop (the grid is capped at 8 CTAs of 8 groups per
    SM), the other one pass; which half alternates along the ladder."""
    per_pass = n_sm * 8 * (256 // pick_rowcfg(d)[1])
    two, one = per_pass + 37 + idx, 613 + 7 * idx
    return (two, one) if idx % 2 == 0 else (one, two)


# ---- the forward pass and the first Adam step -------------------------------------------------------------------
@pytest.mark.parametrize("name,d", [(n, d) for n in TRAIN_KINDS for d in LARGE_D_LADDER],
                         ids=[f"{n}-d{d}" for n in TRAIN_KINDS for d in LARGE_D_LADDER])
def test_forward_and_adam_large_d(name, d):
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    idx = LARGE_D_LADDER.index(d) + TRAIN_KINDS.index(name)
    n_rec, n_kg = _sizes(d, n_sm, idx)
    k = (2, 3) if d in K_NEG_D else (1, 1)
    rng = np.random.default_rng(7000 + d + 13 * TRAIN_KINDS.index(name))
    m = make_product_model(name, U, I, E, R, d)
    _init_tables(m, name, d, rng)
    tabs = _tables(m)
    b, pr, pk = _batch(rng, n_rec, n_kg, *k, U, I, E, R)
    margin = _set_margin_and_resample(m, name, _f64(tabs), b, pr, pk, *k, rng, I, E - N_ISO)
    iso = np.arange(E - N_ISO, E) if (name in HINGE and k[1] == 1) else None
    loss = m._launch_forward(to_device_batch(b), with_grad=True)
    g, marked = _check_forward(m, name, tabs, b, k, margin, loss, f"{name} d={d}", iso)
    _check_adam_first_step(m, tabs, g, marked, f"{name} d={d}")


# ---- the optimisers over several steps ------------------------------------------------------------------------------
@pytest.mark.parametrize("name,d", [("ComplEx", 600), ("TransD", 301), ("RotatE", 767), ("TransH", 1000)],
                         ids=lambda x: str(x))
def test_lazy_adam_replay_and_flush_large_d(name, d):
    """Rows idle in some steps are replayed by the next forward / Adam step and the flush; against float64 dense Adam
    on whole tables with zero gradients on idle rows."""
    rng = np.random.default_rng(500 + d)
    m = make_product_model(name, U, I, E, R, d)
    _init_tables(m, name, d, rng)
    ref = _f64(_tables(m))
    mo = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    vo = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    move = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    m_abs = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    for step, g in enumerate(_run_three_steps(m, rng), start=1):
        _dense_adam_step(ref, mo, vo, move, m_abs, g, step)
    _check_against_dense(m, ref, vo, move, f"{name} d={d}", want_m=mo, m_scale=m_abs)


@pytest.mark.parametrize("learner,lr", [("sgd", 0.5), ("adagrad", 0.05), ("rmsprop", 1e-3)])
@pytest.mark.parametrize("name,d", [("DistMult", 600), ("ComplEx", 301), ("TransE", 767)], ids=lambda x: str(x))
def test_other_learners_large_d(name, d, learner, lr):
    """SGD, Adagrad and RMSprop against torch.optim in float64 fed the kernel's gradients."""
    rng = np.random.default_rng(600 + d)
    m = make_product_model(name, U, I, E, R, d, learner=learner, lr=lr)
    _init_tables(m, name, d, rng)
    init = _f64(_tables(m))
    params = {f: [torch.tensor(t, requires_grad=True) for t in ts] for f, ts in init.items()}
    flat = [t for f in FAMILIES for t in params[f]]
    lr32 = float(np.float32(lr))
    opt = {"sgd": lambda: torch.optim.SGD(flat, lr=lr32), "adagrad": lambda: torch.optim.Adagrad(flat, lr=lr32),
           "rmsprop": lambda: torch.optim.RMSprop(flat, lr=lr32, alpha=RMSPROP_ALPHA)}[learner]()
    move = {f: [np.zeros_like(t) for t in ts] for f, ts in init.items()}
    for g in _run_three_steps(m, rng):
        old = {f: [t.detach().numpy().copy() for t in params[f]] for f in FAMILIES}
        for f in FAMILIES:
            for p, t in enumerate(params[f]):
                t.grad = torch.from_numpy(g[f][p])
        opt.step()
        for f in FAMILIES:
            for p, t in enumerate(params[f]):
                move[f][p] += np.abs(t.detach().numpy() - old[f][p])
    want_w = {f: [t.detach().numpy() for t in params[f]] for f in FAMILIES}
    key = {"adagrad": "sum", "rmsprop": "square_avg"}.get(learner)
    want_v = None if key is None else {f: [opt.state[t][key].numpy() for t in params[f]] for f in FAMILIES}
    _check_against_dense(m, want_w, want_v, move, f"{learner} {name} d={d}")


# ---- the row-sparse exchange ------------------------------------------------------------------------------------
@pytest.mark.parametrize("name,d", [("TransD", 600), ("RotatE", 301), ("ComplEx", 767)], ids=lambda x: str(x))
def test_row_sparse_exchange_large_d(name, d):
    """kge_grad_pack hands out exactly the marked rows' accumulators and clears them; kge_grad_add into a twin with
    the same weights restores them bit for bit, and the next Adam step of both is identical."""
    from hopwise_b200.distributed import FlatLayout, _cuda_add, _cuda_pack

    models = []
    for _ in range(2):
        m = make_product_model(name, U, I, E, R, d)
        _init_tables(m, name, d, np.random.default_rng(900 + d))
        models.append(m)
    m1, m2 = models
    b, _, _ = _batch(np.random.default_rng(901 + d), 2000, 3000, 1, 2, U, I, E, R)
    m1._launch_forward(to_device_batch(b), with_grad=True)
    g, marked = _forward_state(m1)
    rows_of = {"user": U, "entity": E, "relation": R}
    parts = [len(g[f]) for f in FAMILIES]
    lay = FlatLayout([rows_of[f] for f in FAMILIES], parts, d)
    buf = torch.zeros(lay.nbytes, dtype=torch.uint8, device="cuda")
    for which, f in enumerate(FAMILIES):
        count, ids, rows = lay.views(buf, which)
        _cuda_pack(m1, which, 1, count, ids, rows)
        n = int(count.item())
        got_ids = ids[:n].cpu().numpy()
        np.testing.assert_array_equal(np.sort(got_ids), np.flatnonzero(marked[f]), err_msg=f"{f} packed ids")
        packed = rows[:n].view(n, parts[which], d).cpu().numpy()
        for p in range(parts[which]):
            assert np.array_equal(packed[:, p], g[f][p][got_ids]), f"{f}[{p}] packed rows"
            assert not m1._state[f]["g"][p].any(), f"{f}[{p}] accumulator not zeroed by the pack"
        assert bool((m1._state[f]["row_state"][:, 1] == -1).all()), f"{f} marks not cleared"
    m2._ensure_state(torch.device("cuda"))
    for which, f in enumerate(FAMILIES):
        count, ids, rows = lay.views(buf, which)
        for m in (m1, m2):
            _cuda_add(m, which, 1, count, ids, rows)
        got, mk = _forward_state(m2)
        for p in range(parts[which]):
            assert np.array_equal(got[f][p], g[f][p]), f"{f}[{p}] accumulator after the add"
        np.testing.assert_array_equal(mk[f], marked[f], err_msg=f"{f} marks after the add")
    m2._pending = True
    for m in (m1, m2):
        m._launch_apply(None)
    for f, names in zip(FAMILIES, (m1.USER_TABLES, m1.ENTITY_TABLES, m1.RELATION_TABLES)):
        for p, n in enumerate(names):
            assert torch.equal(getattr(m1, n).weight, getattr(m2, n).weight), f"{n} after the step"


# ---- two GPUs: row-sparse route and owner-sharded Adam at d = 1,000 ------------------------------------------------
SHAPE_2GPU = dict(U=3000, I=2500, E=9000, R=9, d=1000)
N_REC, N_KG, STEPS = 192, 160, 3


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _batches_2gpu(k):
    rng = np.random.default_rng(5)
    S = SHAPE_2GPU
    return [random_batch(rng, S["U"], S["I"], S["E"], S["R"], 2 * N_REC, 2 * N_KG, k, k) for _ in range(STEPS)]


def _shard(b, rank, k):
    out = {}
    for key, v in b.items():
        if key.startswith("neg_"):
            n = v.shape[0] // k
            out[key] = v.reshape(k, n)[:, rank * (n // 2):(rank + 1) * (n // 2)].reshape(-1)
        else:
            out[key] = v[rank * (len(v) // 2):(rank + 1) * (len(v) // 2)]
    return out


def _worker(rank, world, port, name, owner, k, out_dir):
    import torch.distributed as dist

    from hopwise_b200.distributed import broadcast_weights, enable_row_sparse_data_parallel

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        dev = f"cuda:{rank}"
        m = make_product_model(name, device=dev, seed=2024 + rank, **SHAPE_2GPU)
        broadcast_weights(m)
        ex = enable_row_sparse_data_parallel(m, owner_adam=owner)
        assert ex.dense == ([True, True, True] if owner else [False, False, True])
        losses = []
        for b in _batches_2gpu(k):
            loss = m.calculate_loss(to_device_batch(_shard(b, rank, k), dev))
            loss.backward()
            losses.append(float(loss.item()))
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), losses=np.array(losses),
                 **{key: v.cpu().numpy() for key, v in m.state_dict().items()})
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("name,owner", [("TransE", False), ("ComplEx", False), ("RotatE", True)])
def test_two_gpu_step_at_d1000(name, owner, tmp_path):
    """The row-sparse route (owner=False) and owner-sharded Adam over the switch at d = 1,000: replicas bit-identical
    and equal to the single-GPU step on the whole batch."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    k = 3 if name in ("RotatE", "ComplEx") else 1
    mp.spawn(_worker, args=(2, _free_port(), name, owner, k, str(tmp_path)), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    for key in r0.files:
        if key != "losses":
            np.testing.assert_array_equal(r0[key], r1[key], err_msg=key)
    m = make_product_model(name, device="cuda:0", seed=2024, **SHAPE_2GPU)
    losses = []
    for b in _batches_2gpu(k):
        loss = m.calculate_loss(to_device_batch(b, "cuda:0"))
        loss.backward()
        losses.append(float(loss.item()))
    np.testing.assert_allclose(0.5 * (r0["losses"] + r1["losses"]), losses, rtol=1e-5)
    for key, v in m.state_dict().items():
        assert_weights_close(r0[key], v.cpu().numpy(), rtol=1e-5, atol=5e-7, err_msg=f"{name} {key}")


# ---- scoring --------------------------------------------------------------------------------------------------------
def _csr(rng, n, lo, hi, max_len):
    from hopwise_b200 import evaluator as ev

    rows = np.repeat(np.arange(n), rng.integers(0, max_len, n))
    items = rng.integers(lo, hi, len(rows))
    off, its = ev.csr_from_pairs(rows, items, n, "cuda")
    return rows, items, off, its


def _rank_counts(dense, pos_rows, pos_items, pos_off):
    """greater / equal of every listed target over its row of masked dense scores (itself included in equal)."""
    items = pos_items.cpu().numpy()
    off = pos_off.cpu().numpy()
    g, e = np.empty(len(items), np.int64), np.empty(len(items), np.int64)
    for r in range(len(off) - 1):
        for i in range(off[r], off[r + 1]):
            s = dense[r, items[i]]
            g[i], e[i] = (dense[r] > s).sum(), (dense[r] == s).sum()
    return g, e


def _check_fused(m, name, queries, dense, rng, err, rels=None):
    """full_sort_topk at k = 20, 128 and 300 and full_sort_rank against the masked dense rows, exactly."""
    cuda = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    n, n_t = dense.shape
    hist_u, hist_i, hist_off, hist_items = _csr(rng, n, 1, n_t, 40)
    masked = ofs.mask_scores(dense, hist_u, hist_i)
    for k in (20, 128, 300):
        if rels is None:
            ids, sc = m.full_sort_topk(cuda(queries), k, hist_off, hist_items, path="cuda")
        else:
            ids, sc = m.full_sort_topk_kg(cuda(queries), cuda(rels), k, hist_off, hist_items, path="cuda")
        want_ids, want_sc = ofs.topk_canonical(masked, k)
        np.testing.assert_array_equal(ids.cpu().numpy(), want_ids, err_msg=f"{err} top-{k} ids")
        np.testing.assert_array_equal(sc.cpu().numpy(), want_sc, err_msg=f"{err} top-{k} scores")
    _, _, pos_off, pos_items = _csr(rng, n, 0, n_t, 6)
    greater, equal, n_unm = m.full_sort_rank(cuda(queries), pos_off, pos_items, hist_off, hist_items,
                                             relation_ids=None if rels is None else cuda(rels))
    want_g, want_e = _rank_counts(masked, None, pos_items, pos_off)
    np.testing.assert_array_equal(greater.cpu().numpy(), want_g, err_msg=f"{err} rank greater")
    np.testing.assert_array_equal(equal.cpu().numpy(), want_e, err_msg=f"{err} rank equal")
    np.testing.assert_array_equal(n_unm.cpu().numpy(), np.isfinite(masked).sum(1), err_msg=f"{err} unmasked")


@pytest.mark.parametrize("name,d", [(n, d) for n in MODELS for d in LARGE_D_LADDER],
                         ids=[f"{n}-d{d}" for n in MODELS for d in LARGE_D_LADDER])
def test_scores_large_d(name, d):
    """predict / predict_kg / the dense full-sort scorers against the float64 scores, and the fused top-k (k = 20,
    128, 300) and rank counts against the model's own dense rows, users -> items and link prediction."""
    U_, I_, E_, R_ = 60, 700, 900, 9
    rng = np.random.default_rng(3000 + d + 11 * MODELS.index(name))
    m = make_product_model(name, U_, I_, E_, R_, d)
    _init_tables(m, name, d, rng)
    tabs = _f64(_tables(m))
    margin = float(np.float32(m.margin))
    ui = m._ui_row(False)
    err = f"{name} d={d}"
    cuda = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    rel = lambda ids: [t[ids] for t in tabs["relation"]]   # noqa: E731
    users, items = rng.integers(0, U_, 97), rng.integers(0, I_, 97)
    got = m.predict({"user_id": cuda(users), "item_id": cuda(items)}).cpu().numpy()
    _check_scores(got, name, [t[users] for t in tabs["user"]], rel(np.full(97, ui)),
                  [t[items] for t in tabs["entity"]], margin, f"{err} predict")
    if name != "TransH":
        heads, rels, tails = rng.integers(0, E_, 53), rng.integers(0, R_ - 1, 53), rng.integers(0, E_, 53)
        got = m.predict_kg({"head_id": cuda(heads), "relation_id": cuda(rels), "tail_id": cuda(tails)}).cpu().numpy()
        _check_scores(got, name, [t[heads] for t in tabs["entity"]], rel(rels), [t[tails] for t in tabs["entity"]],
                      margin, f"{err} predict_kg")
    qu = rng.integers(1, U_, 37)   # (more than one query block of 32 and of 16 rows)
    dense = m.full_sort_predict({"user_id": cuda(qu)}).cpu().numpy()
    _check_scores(dense, name, [t[qu] for t in tabs["user"]], rel(np.full(37, m._ui_row(True))),
                  [t[:I_] for t in tabs["entity"]], margin, f"{err} full_sort_predict")
    _check_fused(m, name, qu, dense, rng, f"{err} users")
    if name not in ("TransH", "TransD"):
        qh, qr = rng.integers(1, E_, 19), rng.integers(0, R_ - 1, 19)
        dense_kg = m.full_sort_predict_kg({"head_id": cuda(qh), "relation_id": cuda(qr)}).cpu().numpy()
        _check_scores(dense_kg, name, [t[qh] for t in tabs["entity"]], rel(qr), tabs["entity"], margin,
                      f"{err} full_sort_predict_kg")
        _check_fused(m, name, qh, dense_kg, rng, f"{err} link prediction", rels=qr)


@pytest.mark.parametrize("name", MODELS)
def test_candidate_topk_d1000(name):
    """Sampled evaluation at d = 1,000: the top-k of each row's candidates by the model's own predict scores."""
    U_, I_, E_, R_, d = 40, 600, 800, 9, 1000
    rng = np.random.default_rng(41 + MODELS.index(name))
    m = make_product_model(name, U_, I_, E_, R_, d)
    _init_tables(m, name, d, rng)
    n, k = 24, 20
    lens = rng.integers(5, 130, n)
    off = np.concatenate([[0], np.cumsum(lens)])
    users = np.repeat(rng.integers(1, U_, n), lens)
    items = rng.integers(0, I_, off[-1])
    cuda = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    ids, sc = m.candidate_topk(cuda(users), cuda(items), torch.from_numpy(off), k)
    pred = m.predict({"user_id": cuda(users), "item_id": cuda(items)}).cpu().numpy()
    dense = np.full((n, I_), -np.inf, dtype=np.float32)
    for r in range(n):
        dense[r, items[off[r]:off[r + 1]]] = pred[off[r]:off[r + 1]]
    want_ids, want_sc = ofs.topk_canonical(dense, k)
    np.testing.assert_array_equal(ids.cpu().numpy(), want_ids, err_msg=name)
    np.testing.assert_array_equal(sc.cpu().numpy(), want_sc, err_msg=name)


@pytest.mark.parametrize("name", ("DistMult", "TransE"))
def test_tensor_core_path_at_d600(name):
    """K = 600 (DistMult) / 603 (TransE) reaches the tensor-core path under "auto"; its ids and scores equal the
    CUDA-core path's bit for bit, the rows of its exact fallback (the tile kernel) included."""
    U_, I_, E_, R_, d = 300, 9000, 9500, 9, 600
    rng = np.random.default_rng(60 + len(name))
    m = make_product_model(name, U_, I_, E_, R_, d)
    _init_tables(m, name, d, rng)
    assert m._mma_supported(32, I_)
    n = 300
    qu = torch.from_numpy(rng.integers(1, U_, n)).cuda()
    lens = rng.integers(0, 80, n)
    lens[7] = I_ - 1 - 3   # fewer than k unmasked items (k > 3): recomputed by the exact fallback
    lens[9] = I_ - 1       # no unmasked item: the same for every k
    hist = [np.sort(rng.choice(np.arange(1, I_), size=int(x), replace=False)) for x in lens]
    off = torch.from_numpy(np.concatenate([[0], np.cumsum(lens)])).cuda()
    items = torch.from_numpy(np.concatenate(hist)).cuda()
    for k in (1, 20, 32):
        want = m.full_sort_topk(qu, k, off, items, path="cuda")
        for path in ("mma", "auto"):
            calls = len(m._mma_counters)
            got = m.full_sort_topk(qu, k, off, items, path=path)
            assert len(m._mma_counters) == calls + 1, (name, k, path)   # the tensor-core path ran
            assert m._mma_last_fallback_rows >= 1, (name, k, path)
            assert torch.equal(got[0], want[0]) and torch.equal(got[1], want[1]), (name, k, path)
