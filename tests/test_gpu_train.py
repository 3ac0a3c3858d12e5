"""Parity of the fused CUDA train step (gather -> score -> loss -> scatter -> lazy Adam), called
through the C ABI, against (1) the golden vectors produced by the unmodified reference and
(2) the torch-CPU oracle on seeded random inputs.  Tolerance: 1e-5 relative (fp32), as
BASELINE.json's north_star states; atol covers values whose magnitude is near zero."""

import numpy as np
import pytest
import torch

from conftest import MODELS, load_golden
from kge_helpers import (
    BATCH_KEYS,
    assert_weights_close,
    make_oracle_model,
    make_product_model,
    random_batch,
    tile_batch,
    to_cpu_batch,
    to_device_batch,
)
from oracle.kge_torch import make_optimizer, train_step

pytestmark = pytest.mark.gpu

RTOL = 1e-5


def _golden_model(name, g):
    U, I, E, R, d = (int(x) for x in g["shape"])
    m = make_product_model(name, U, I, E, R, d, margin=float(g["margin"]))
    sd = {k[5:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("init/")}
    m.load_state_dict(sd, strict=True)
    return m


def _gbatch(g, i):
    return {k: torch.from_numpy(g[f"batch{i}/{k}"]).cuda() for k in BATCH_KEYS}


def _trainer_step(model, opt, batch):
    """The reference's loop body (trainer/trainer.py:243-265)."""
    opt.zero_grad()
    loss = model.calculate_loss(batch)
    value = loss.item()
    assert not torch.isnan(loss)
    loss.backward()
    opt.step()
    return value


@pytest.mark.parametrize("tag", ["d20", "d10"])
@pytest.mark.parametrize("name", MODELS)
def test_golden_trajectory(name, tag):
    g = load_golden(f"model_{name}_{tag}.npz")
    m = _golden_model(name, g)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)  # what KGTrainer builds; must stay a no-op
    for step, bi in enumerate(g["schedule"], start=1):
        loss = _trainer_step(m, opt, _gbatch(g, int(bi)))
        np.testing.assert_allclose(loss, g["losses"][step - 1], rtol=RTOL, err_msg=f"{name} loss step {step}")
        if step in (1, 4, 12):
            sd = m.state_dict()
            for k, v in sd.items():
                np.testing.assert_allclose(
                    v.cpu().numpy(), g[f"step{step}/{k}"], rtol=RTOL, atol=2e-7, err_msg=f"{name} {k} step {step}"
                )
    # no parameter ever received a dense gradient
    assert all(p.grad is None for p in m.parameters())


@pytest.mark.parametrize("name", MODELS)
def test_golden_gradients(name):
    g = load_golden(f"model_{name}_d20.npz")
    m = _golden_model(name, g)
    m._launch_forward(_gbatch(g, 1), with_grad=True)  # schedule[0] == 1
    torch.cuda.synchronize()
    fams = (("user", m.USER_TABLES), ("entity", m.ENTITY_TABLES), ("relation", m.RELATION_TABLES))
    for fam, names in fams:
        for p, tname in enumerate(names):
            got = m._state[fam]["g"][p].cpu().numpy()
            want = g[f"grad1/{tname}.weight"]
            np.testing.assert_allclose(got, want, rtol=1e-4, atol=1e-8, err_msg=f"{name} {tname}")
        # every row with a non-zero gradient is marked as touched in step 1, and nothing untouched is
        touched = np.flatnonzero(m._state[fam]["row_state"][:, 1].cpu().numpy() == 1)
        nz = np.flatnonzero(np.any(np.stack([g[f"grad1/{t}.weight"] for t in names]) != 0, axis=(0, 2)))
        assert set(nz) <= set(touched)
        got_all = np.stack([m._state[fam]["g"][p].cpu().numpy() for p in range(len(names))])
        assert not np.any(got_all[:, np.setdiff1d(np.arange(got_all.shape[1]), touched)])
    m.flush()


@pytest.mark.parametrize("name", MODELS)
def test_golden_scores(name):
    for tag in ("d20", "d10"):
        g = load_golden(f"model_{name}_{tag}.npz")
        m = _golden_model(name, g)
        m.load_state_dict({k[7:]: torch.from_numpy(g[k]) for k in g.files if k.startswith("step12/")})
        m.eval()
        b = _gbatch(g, 0)
        np.testing.assert_allclose(m.predict(b).cpu().numpy(), g["predict"], rtol=RTOL, atol=1e-6)
        users = torch.from_numpy(g["fullsort_users"]).cuda()
        fs = m.full_sort_predict({"user_id": users})
        assert fs.shape == g["fullsort"].shape
        np.testing.assert_allclose(fs.cpu().numpy(), g["fullsort"], rtol=RTOL, atol=1e-6)
        kb = {"head_id": b["head_id"][:5], "relation_id": b["relation_id"][:5]}
        if "predict_kg" in g.files:
            np.testing.assert_allclose(m.predict_kg(b).cpu().numpy(), g["predict_kg"], rtol=RTOL, atol=1e-6)
        else:   # transh.py scores users against items only: the KG entry points refuse
            with pytest.raises(NotImplementedError):
                m.predict_kg(b)
        if "fullsort_kg" in g.files:
            np.testing.assert_allclose(m.full_sort_predict_kg(kb).cpu().numpy(), g["fullsort_kg"], rtol=RTOL, atol=1e-6)
        else:   # (and TransD's dense KG full-sort, whose reference version is not mirrored)
            with pytest.raises(NotImplementedError):
                m.full_sort_predict_kg(kb)


CASES = [
    # name, U, I, E, R, d, n_rec, n_kg, k_rec, k_kg, steps
    ("TransE", 300, 200, 900, 12, 100, 512, 512, 1, 1, 25),
    ("TransE", 300, 200, 900, 12, 64, 300, 200, 1, 1, 10),
    ("DistMult", 300, 200, 900, 12, 64, 512, 512, 1, 1, 25),
    ("RotatE", 200, 150, 700, 9, 256, 128, 128, 1, 1, 12),
    ("ComplEx", 300, 200, 900, 12, 64, 512, 512, 1, 1, 25),
    ("TransE", 300, 200, 900, 12, 128, 0, 400, 1, 1, 6),     # KG half only
    ("DistMult", 300, 200, 900, 12, 32, 400, 0, 1, 1, 6),    # rec half only (BCE models give NaN there, as the reference does)
    ("DistMult", 120, 80, 300, 7, 50, 128, 96, 1, 1, 8),     # d % 4 != 0: scalar row path
    ("RotatE", 120, 80, 300, 7, 24, 64, 64, 4, 3, 8),        # K negatives, compact layout
    ("TransE", 120, 80, 300, 7, 36, 64, 64, 5, 2, 8),
    ("ComplEx", 120, 80, 300, 7, 16, 64, 64, 2, 6, 8),
    ("DistMult", 120, 80, 300, 7, 512, 32, 32, 1, 1, 4),     # largest supported d
    ("TransH", 300, 200, 900, 12, 100, 512, 512, 1, 1, 25),  # projection + hyperplane-vector gradient
    ("TransH", 120, 80, 300, 7, 36, 64, 64, 3, 2, 8),
    ("TransH", 120, 80, 300, 7, 50, 96, 0, 1, 1, 6),         # d % 4 != 0, rec half only
    ("TorusE", 300, 200, 900, 12, 64, 300, 200, 1, 1, 10),   # TransE's step under another name
    ("TransD", 300, 200, 900, 12, 100, 512, 512, 1, 1, 25),  # transfer vectors: six tables, three dot products per row
    ("TransD", 120, 80, 300, 7, 36, 64, 64, 3, 2, 8),
    ("TransD", 120, 80, 300, 7, 50, 0, 96, 1, 1, 6),         # d % 4 != 0, KG half only
]


@pytest.mark.parametrize("case", CASES, ids=lambda c: f"{c[0]}-d{c[5]}-k{c[8]}x{c[9]}")
def test_oracle_trajectory(case):
    name, U, I, E, R, d, n_rec, n_kg, k_rec, k_kg, steps = case
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    for (ka, va), (kb, vb) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert ka == kb and torch.equal(va, vb.cpu())
    opt_o = make_optimizer(ora)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    rng = np.random.default_rng(7)
    # a small pool of batches, so rows are revisited after idle gaps (lazy Adam catch-up)
    pool = [random_batch(rng, U, I, E, R, n_rec, n_kg, k_rec, k_kg) for _ in range(4)]
    for step in range(steps):
        b = pool[(step * step) % 4]
        want = train_step(ora, opt_o, to_cpu_batch(tile_batch(b, k_rec, k_kg)))
        got = _trainer_step(m, opt, to_device_batch(b))
        np.testing.assert_allclose(got, want, rtol=RTOL, err_msg=f"loss at step {step + 1}")
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=5e-7, err_msg=k)


def test_tiled_and_compact_negatives_agree():
    """The reference's K-negative layout (positives tiled K times) and the compact layout give
    the same loss and the same update."""
    name, U, I, E, R, d, K = "RotatE", 90, 60, 200, 6, 32, 3
    rng = np.random.default_rng(3)
    b = random_batch(rng, U, I, E, R, 40, 50, K, K)
    ma = make_product_model(name, U, I, E, R, d)
    mb = make_product_model(name, U, I, E, R, d)
    la = ma.calculate_loss(to_device_batch(b))
    lb = mb.calculate_loss(to_device_batch(tile_batch(b, K, K)))
    np.testing.assert_allclose(la.item(), lb.item(), rtol=1e-6)
    la.backward()
    lb.backward()
    for (k, va), (_, vb) in zip(ma.state_dict().items(), mb.state_dict().items()):
        np.testing.assert_allclose(va.cpu().numpy(), vb.cpu().numpy(), rtol=1e-5, atol=1e-7, err_msg=k)


def test_loss_without_backward_leaves_weights_alone():
    name, U, I, E, R, d = "DistMult", 90, 60, 200, 6, 32
    rng = np.random.default_rng(5)
    b = to_device_batch(random_batch(rng, U, I, E, R, 64, 64))
    m = make_product_model(name, U, I, E, R, d)
    before = {k: v.clone() for k, v in m.state_dict().items()}
    l1 = m.calculate_loss(b).item()          # graph built, backward never called
    with torch.no_grad():
        l2 = m.calculate_loss(b).item()      # evaluation-style call
    l3 = m.calculate_loss(b)
    assert l1 == pytest.approx(l2, rel=1e-6) and l1 == pytest.approx(l3.item(), rel=1e-6)
    for k, v in m.state_dict().items():
        assert torch.equal(v, before[k])
    l3.backward()                            # only this one updates, exactly once
    ora = make_oracle_model(name, U, I, E, R, d)
    train_step(ora, make_optimizer(ora), {k: v.cpu() for k, v in b.items()})
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=5e-7, err_msg=k)


def test_grad_output_scale_is_honoured():
    """(loss * c).backward() must equal a step with gradient c * g (trainer adds sync_loss terms)."""
    name, U, I, E, R, d = "TransE", 90, 60, 200, 6, 32
    rng = np.random.default_rng(9)
    b = random_batch(rng, U, I, E, R, 64, 64)
    m = make_product_model(name, U, I, E, R, d)
    ora = make_oracle_model(name, U, I, E, R, d)
    opt_o = make_optimizer(ora)
    for _ in range(3):
        (m.calculate_loss(to_device_batch(b)) * 0.25 + 0.0).backward()
        opt_o.zero_grad()
        (ora.calculate_loss(to_cpu_batch(b)) * 0.25).backward()
        opt_o.step()
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=5e-7, err_msg=k)


def test_long_idle_rows_follow_dense_adam():
    """A row touched once and then idle for more steps than the replay cap still lands on dense
    Adam's value (closed-form tail of the lazy catch-up)."""
    name, U, I, E, R, d = "TransE", 40, 30, 120, 5, 16
    rng = np.random.default_rng(11)

    def half_batch(lo_frac, hi_frac, n):
        def ids(size):
            return rng.integers(max(1, int(size * lo_frac)), max(2, int(size * hi_frac)), n)

        return {
            "user_id": ids(U), "item_id": ids(I), "neg_item_id": ids(I), "head_id": ids(E),
            "relation_id": rng.integers(1, R - 1, n), "tail_id": ids(E), "neg_tail_id": ids(E),
        }

    first = half_batch(0.5, 1.0, 32)   # upper half of every id range, seen once
    later = half_batch(0.0, 0.5, 32)   # lower half, seen on every later step
    m = make_product_model(name, U, I, E, R, d)   # default replay cap: 200 exact steps, then closed form
    ora = make_oracle_model(name, U, I, E, R, d)
    opt_o = make_optimizer(ora)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    for step in range(240):
        b = first if step == 0 else later
        train_step(ora, opt_o, to_cpu_batch(b))
        _trainer_step(m, opt, to_device_batch(b))
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=1e-6, err_msg=k)


def test_rows_of_inactive_triples_stay_current():
    """Rows that keep being referenced by margin-inactive triples (no gradient) must not fall behind the
    optimiser: a lagging referenced row is marked and caught up by the Adam kernel, so its lag is bounded by the
    gap between two references (otherwise every forward pass replays a growing run of skipped steps).  The
    trajectory is dense Adam's either way."""
    name, U, I, E, R, d = "DistMult", 50, 40, 200, 6, 16   # (margin_ranking_loss accepts the negative margin below)
    rng = np.random.default_rng(21)
    b = random_batch(rng, U, I, E, R, 64, 64)
    m = make_product_model(name, U, I, E, R, d, margin=1.0)
    ora = make_oracle_model(name, U, I, E, R, d, margin=1.0)
    opt_o = make_optimizer(ora)
    opt = torch.optim.Adam(m.parameters(), lr=1e-3)
    steps = 30
    for step in range(steps):
        if step == 3:   # from here on no triple is active: margin - s(pos) + s(neg) < 0 for every pair
            m.margin = -1e3
            m._struct_cache = {}
            ora.shapes.margin = -1e3
        train_step(ora, opt_o, to_cpu_batch(b))
        _trainer_step(m, opt, to_device_batch(b))
    rs = m._state["entity"]["row_state"].cpu().numpy()
    ref = np.unique(np.concatenate([b["item_id"], b["neg_item_id"], b["head_id"], b["tail_id"], b["neg_tail_id"]]))
    last = rs[ref, 0]
    assert (last[last >= 0] >= steps - 1).all(), "a referenced row lags behind the optimiser"
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=1e-6, err_msg=k)


def test_checkpoint_round_trip_continues_the_trajectory():
    name, U, I, E, R, d = "ComplEx", 60, 40, 150, 6, 16
    rng = np.random.default_rng(13)
    pool = [random_batch(rng, U, I, E, R, 48, 48) for _ in range(3)]
    a = make_product_model(name, U, I, E, R, d)
    for s in range(5):
        a.calculate_loss(to_device_batch(pool[s % 3])).backward()
    ckpt = {"state_dict": a.state_dict(), "other_parameter": a.other_parameter()}
    b = make_product_model(name, U, I, E, R, d, seed=1)
    b.load_state_dict(ckpt["state_dict"])
    b.load_other_parameter(ckpt["other_parameter"])
    for s in range(5, 9):
        la = a.calculate_loss(to_device_batch(pool[s % 3]))
        lb = b.calculate_loss(to_device_batch(pool[s % 3]))
        assert la.item() == pytest.approx(lb.item(), rel=1e-6)
        la.backward()
        lb.backward()
    for (k, va), (_, vb) in zip(a.state_dict().items(), b.state_dict().items()):
        np.testing.assert_allclose(va.cpu().numpy(), vb.cpu().numpy(), rtol=1e-6, atol=1e-8, err_msg=k)


def test_empty_batch_and_bad_arguments():
    m = make_product_model("TransE", 20, 10, 40, 5, 16)
    empty = {k: torch.zeros(0, dtype=torch.long, device="cuda") for k in BATCH_KEYS}
    assert m.calculate_loss(empty).item() == 0.0
    with pytest.raises(ValueError):
        bad = to_device_batch(random_batch(np.random.default_rng(0), 20, 10, 40, 5, 8, 8))
        bad["item_id"] = bad["item_id"][:5]
        m.calculate_loss(bad)
    with pytest.raises(RuntimeError):
        m.calculate_loss(to_cpu_batch(random_batch(np.random.default_rng(0), 20, 10, 40, 5, 8, 8)))


def test_full_size_step_properties():
    """BASELINE config 2 at the roofline batch: invariants that do not need the oracle at size:
    the update is a no-op for untouched rows, finite everywhere, and the loss of a repeated batch
    goes down."""
    U, I, E, R, d = 6041, 3001, 30001, 22, 100
    m = make_product_model("TransE", U, I, E, R, d)
    rng = np.random.default_rng(2024)
    b = random_batch(rng, U, I, E, R, 262144, 262144)
    b["head_id"] = np.minimum(b["head_id"], 20000)  # leave entities > 20000 untouched as heads
    b["tail_id"] = np.minimum(b["tail_id"], 20000)
    b["neg_tail_id"] = np.minimum(b["neg_tail_id"], 20000)
    w0 = m.entity_embedding.weight.detach().clone()
    db = to_device_batch(b)
    losses = []
    for _ in range(5):
        loss = m.calculate_loss(db)
        loss.backward()
        losses.append(loss.item())
    m.flush()
    w1 = m.entity_embedding.weight.detach()
    assert torch.isfinite(w1).all()
    assert torch.equal(w1[20001:], w0[20001:])
    assert not torch.equal(w1[3001:20001], w0[3001:20001])
    assert losses[-1] < losses[0]
    # one oracle step on the same batch (CPU, a few seconds) pins the loss value at full size
    ora = make_oracle_model("TransE", U, I, E, R, d)
    with torch.no_grad():
        want = ora.calculate_loss(to_cpu_batch(b)).item()
    np.testing.assert_allclose(losses[0], want, rtol=RTOL)


def test_device_prefetcher_preserves_batches_and_training_result():
    """Staging batches one step ahead on a copy stream changes nothing but the timing."""
    from hopwise_b200.loader import DevicePrefetcher

    U, I, E, R, d = 300, 200, 900, 7, 32
    rng = np.random.default_rng(3)
    host = [{k: torch.from_numpy(np.asarray(v)).pin_memory() for k, v in random_batch(rng, U, I, E, R, 128, 96).items()}
            for _ in range(5)]
    seen = []
    for db in DevicePrefetcher(host, "cuda"):
        assert all(t.is_cuda for t in db.values())
        seen.append({k: v.cpu() for k, v in db.items()})
    assert len(seen) == len(host)
    for a, b in zip(seen, host):
        for k in b:
            assert torch.equal(a[k], b[k])
    m1 = make_product_model("TransE", U, I, E, R, d)
    m2 = make_product_model("TransE", U, I, E, R, d)
    for b in host:
        m1.calculate_loss({k: v.cuda() for k, v in b.items()}).backward()
    from hopwise_b200.loader import pack_batch

    packed = [pack_batch(b) for b in host]   # one copy per step instead of seven
    assert packed[0].base.is_pinned() and packed[0].base.numel() == (sum(v.numel() for v in host[0].values()) + 3) // 4 * 4
    # ids staged as int32 and widened on the device (kge_widen_ids_i32): the consumer sees the same int64 vectors
    narrow = [pack_batch(b, narrow=True) for b in host]
    assert narrow[0].base.dtype == torch.int32 and narrow[0].base.nbytes * 2 == packed[0].base.nbytes
    for i, db in enumerate(DevicePrefetcher(narrow, "cuda")):
        for k in host[i]:
            assert db[k].dtype == torch.int64 and torch.equal(db[k].cpu(), host[i][k])
    for k, v in narrow[2].to("cuda").items():
        assert v.dtype == torch.int64 and torch.equal(v.cpu(), host[2][k])
    with pytest.raises(ValueError):
        pack_batch({"user_id": np.array([1, 2 ** 31])}, narrow=True)
    for db in DevicePrefetcher(packed, "cuda", depth=3):
        assert set(db) == set(host[0]) and all(t.is_cuda for t in db.values())
        m2.calculate_loss(db).backward()
    for (k1, v1), (_, v2) in zip(m1.state_dict().items(), m2.state_dict().items()):
        assert_weights_close(v2.cpu().numpy(), v1.cpu().numpy(), rtol=1e-5, atol=5e-7, err_msg=k1)


@pytest.mark.parametrize("name", MODELS)
def test_one_call_train_step_follows_the_golden_trajectory(name):
    """model.train_step(batch) -- forward + Adam in one library call, what FusedKGTrainer's epoch loop uses -- on the
    reference's golden trajectory; interleaved with the autograd route to show the two share all state."""
    g = load_golden(f"model_{name}_d20.npz")
    m = _golden_model(name, g)
    held = []
    for step, bi in enumerate(g["schedule"], start=1):
        b = _gbatch(g, int(bi))
        if step % 5 == 0:   # the two-launch route in between: same optimiser state, same step counter
            loss = m.calculate_loss(b)
            loss.backward()
        else:
            loss = m.train_step(b)
            assert loss.grad_fn is None and loss.dim() == 0
        held.append(loss.detach())
        if step in (1, 4, 12):
            for k, v in m.state_dict().items():
                assert_weights_close(v.cpu().numpy(), g[f"step{step}/{k}"], rtol=RTOL, err_msg=f"{name} {k} step {step}")
    # the losses stay valid after the fact (ring slots are never rewritten)
    np.testing.assert_allclose(torch.stack(held).cpu().numpy(), g["losses"], rtol=RTOL)


def test_train_step_loss_ring_rolls_over():
    U, I, E, R, d = 50, 40, 90, 5, 16
    rng = np.random.default_rng(3)
    m = make_product_model("TransE", U, I, E, R, d)
    ora = make_oracle_model("TransE", U, I, E, R, d)
    opt = make_optimizer(ora)
    n = m.LOSS_RING + 9
    got, want = [], []
    for _ in range(n):
        b = random_batch(rng, U, I, E, R, 8, 8)
        want.append(train_step(ora, opt, to_cpu_batch(b)))
        got.append(m.train_step(to_device_batch(b)))
    np.testing.assert_allclose(torch.stack(got).cpu().numpy(), np.array(want), rtol=1e-4)
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=1e-4, atol=2e-6, err_msg=k)


@pytest.mark.parametrize("learner,lr", [("sgd", 0.5), ("adagrad", 0.05), ("rmsprop", 1e-3), ("adamw", 1e-3)])
@pytest.mark.parametrize("name", ["TransE", "ComplEx", "TransD"])
def test_other_learners_follow_torch(name, learner, lr):
    """trainer.py:189-205: sgd / adagrad / rmsprop (and adamw, which is Adam at weight_decay 0) applied to the touched
    rows only, against torch.optim's dense versions on the oracle: rows idle for several steps in between (RMSprop's
    second moment keeps decaying on them), checkpoint flush in the middle."""
    U, I, E, R, d = 120, 80, 300, 7, 36
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d, learner=learner, lr=lr)
    assert m.learner == ("adam" if learner == "adamw" else learner)
    opt_o = make_optimizer(ora, lr=lr, learner=learner)
    rng = np.random.default_rng(11)
    pool = [random_batch(rng, U, I, E, R, 64, 48, 2, 1) for _ in range(4)]
    for step in range(14):
        b = pool[(step * step) % 4]
        want = train_step(ora, opt_o, to_cpu_batch(tile_batch(b, 2, 1)))
        got = m.train_step(to_device_batch(b)) if step % 2 else _trainer_step(m, torch.optim.SGD(m.parameters(), lr=0.1),
                                                                              to_device_batch(b))
        np.testing.assert_allclose(float(got), want, rtol=RTOL, err_msg=f"loss at step {step + 1}")
        if step == 6:
            m.state_dict()   # flushes: every row current, RMSprop's idle rows decayed
    # RMSprop / Adagrad move an element by ~lr * g / |g| on its first gradients whatever |g| is, so the rounding noise of
    # a nearly cancelled gradient becomes a visible share of one step on a few elements (like Adam, kge_helpers): more
    # of them are allowed here, none beyond a hundredth of RMSprop's ~10 * lr first step
    frac = 5e-3 if learner in ("adagrad", "rmsprop") else 5e-4
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=5e-7, outlier_frac=frac, err_msg=f"{learner} {k}")
    if learner in ("adagrad", "rmsprop"):   # the second moments too (torch keeps them per parameter)
        st = m.kge_optimizer_state
        key = "sum" if learner == "adagrad" else "square_avg"
        for fam, names in (("user", m.USER_TABLES), ("entity", m.ENTITY_TABLES), ("relation", m.RELATION_TABLES)):
            for p, tname in enumerate(names):
                want_v = opt_o.state[getattr(ora, tname).weight][key].numpy()
                np.testing.assert_allclose(st[fam]["v"][p].numpy(), want_v, rtol=2e-4, atol=1e-10, err_msg=f"{learner} v {tname}")


@pytest.mark.parametrize("name", ["TransE", "RotatE"])
def test_interleaved_and_dropped_steps_follow_the_oracle(name):
    """One-call steps (train_step) and two-launch steps (calculate_loss + backward) in any order, with a gradient
    that is dropped in between (a loss whose backward never runs: kge_grad_discard), follow the oracle's trajectory."""
    U, I, E, R, d = 150, 100, 400, 7, 32
    ora = make_oracle_model(name, U, I, E, R, d)
    m = make_product_model(name, U, I, E, R, d)
    opt_o = make_optimizer(ora)
    rng = np.random.default_rng(5)
    pool = [random_batch(rng, U, I, E, R, 96, 80) for _ in range(5)]
    plan = ["step"] * 4 + ["drop"] + ["step"] * 5 + ["drop"] + ["step"] * 2
    for step, mode in enumerate(plan):
        b = pool[step % 5]
        if mode == "drop":   # a loss whose backward never runs
            m.calculate_loss(to_device_batch(pool[(step + 2) % 5]))
            continue
        want = train_step(ora, opt_o, to_cpu_batch(b))
        if step % 2:
            got = float(m.train_step(to_device_batch(b)))
        else:
            loss = m.calculate_loss(to_device_batch(b))
            got = float(loss.item())
            loss.backward()
        np.testing.assert_allclose(got, want, rtol=RTOL, err_msg=f"loss at step {step + 1}")
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=5e-7, err_msg=k)
