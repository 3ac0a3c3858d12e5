"""Weight decay on the fused path against torch itself: AdamW's decoupled decay and SGD's L2 term reach every row of
every table in every step -- rows a batch does not touch and rows no batch has ever referenced included -- as they do
under the reference trainer's dense torch.optim.AdamW / SGD (trainer/trainer.py:189-205), whose tables all receive a
dense gradient every step."""

import os

import numpy as np
import pytest
import torch

from kge_helpers import (
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
# per-step decay lr * wd: 5e-4 (AdamW), 5e-3 (SGD) -- hundreds of times RTOL
HP = {"adamw": dict(lr=1e-3, weight_decay=0.5), "sgd": dict(lr=0.5, weight_decay=0.01)}


def _trainer_step(model, batch):
    loss = model.calculate_loss(batch)
    value = loss.item()
    loss.backward()
    return value


def _assert_model_close(m, ora, tag, frac=5e-4):
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        assert_weights_close(vp.cpu().numpy(), vo.numpy(), rtol=RTOL, atol=5e-7, outlier_frac=frac, err_msg=f"{tag} {k}")


@pytest.mark.parametrize("name,learner,d", [
    ("TransE", "adamw", 36), ("TransE", "sgd", 50), ("RotatE", "adamw", 50), ("RotatE", "sgd", 36),
    ("ComplEx", "adamw", 36), ("ComplEx", "sgd", 36), ("TransD", "adamw", 50), ("TransD", "sgd", 36),
    ("TransE", "adamw", 600), ("ComplEx", "sgd", 516),
])
def test_trajectory_follows_torch(name, learner, d):
    """Batches draw from the lower half of every table only: the upper half is never referenced and must still decay
    (checked through state_dict, which flushes).  Rows of the lower half sit idle for several steps between batches.
    One-call and two-launch steps alternate, a flush runs mid-way, and the run goes on from a checkpoint
    (state_dict + kge_optimizer_state) in a fresh model."""
    U, I, E, R = 120, 80, 300, 7
    hp = HP[learner]
    ora = make_oracle_model(name, U, I, E, R, d)
    opt_o = make_optimizer(ora, lr=hp["lr"], weight_decay=hp["weight_decay"], learner=learner)
    cfg = dict(learner=learner, lr=hp["lr"], weight_decay=hp["weight_decay"])
    m = make_product_model(name, U, I, E, R, d, **cfg)
    assert m.learner == learner
    rng = np.random.default_rng(13)
    pool = [random_batch(rng, U // 2, I // 2, E // 2, R, 48, 40, 2, 1) for _ in range(4)]
    for step in range(16):
        b = pool[(step * step) % 4]
        want = train_step(ora, opt_o, to_cpu_batch(tile_batch(b, 2, 1)))
        got = float(m.train_step(to_device_batch(b))) if step % 2 else _trainer_step(m, to_device_batch(b))
        np.testing.assert_allclose(got, want, rtol=RTOL, err_msg=f"loss at step {step + 1}")
        if step == 5:
            m.flush()
        if step == 9:   # checkpoint, then the rest of the run in a fresh model
            sd = {k: v.clone() for k, v in m.state_dict().items()}
            st = m.kge_optimizer_state
            m = make_product_model(name, U, I, E, R, d, seed=7, **cfg)
            m.load_state_dict(sd)
            m.kge_optimizer_state = st
    _assert_model_close(m, ora, f"{name} {learner} d={d}")
    # the never-referenced half moved by the decay alone (not a trivially equal untouched table)
    w0 = make_product_model(name, U, I, E, R, d, **cfg).state_dict()
    for k, v in m.state_dict().items():
        if "entity" in k:
            assert not torch.equal(v[E // 2 + 1 :], w0[k][E // 2 + 1 :]), k


@pytest.mark.parametrize("learner,lr,wd", [("adamw", 1e-3, 0.5), ("sgd", 0.05, 0.2), ("sgd", 1.0, 1.999)])
def test_idle_gaps_beyond_the_replay_cap(learner, lr, wd):
    """kge_replay_cap 3 and rows idle for ~5,000 steps: the tail beyond the cap is f^n in closed form, f = 1 - lr * wd,
    against torch's product of 5,000 rounded steps; f = -0.999 (lr * wd >= 1, where powf would give NaN) included.

    Between the first and the last step every batch pairs each positive with itself as the negative: the hinge is open
    but the gradient cancels exactly (under autograd and in the kernel alike), so the rows it names are touched in every
    step and move by the decay alone, one step at a time, while every other row lags.  The decay is then all that moves
    the model for 5,000 steps -- no trained trajectory whose rounding grows with the run.  Rows given a gradient at step
    1 (SGD) lag for ~5,000 steps and take the closed-form tail on their next touch; rows first touched at the last step
    are caught up from step 0 in the forward pass and the optimiser kernel; the rest decay in the final flush.  (AdamW
    has no rows with moments that lag: the cap bounds its Adam replay, exact only to ~200 steps; a row with zero moments
    decays alone, exactly.)"""
    U, I, E, R, d, N = 40, 20, 60, 4, 8, 5000
    ora = make_oracle_model("TransE", U, I, E, R, d)
    opt_o = make_optimizer(ora, lr=lr, weight_decay=wd, learner=learner)
    m = make_product_model("TransE", U, I, E, R, d, learner=learner, lr=lr, weight_decay=wd, kge_replay_cap=3)

    def batch(users, items, ents, self_negative=False):
        items, ents = np.array(items), np.array(ents)
        tails = ents[::-1].copy()
        return {"user_id": np.array(users), "item_id": items,
                "neg_item_id": items if self_negative else items[::-1].copy(),
                "head_id": ents, "relation_id": np.arange(len(ents)) % (R - 2) + 1, "tail_id": tails,
                "neg_tail_id": tails if self_negative else np.roll(ents, 1)}

    # (each row is the tail of at most one pair per half: its two opposite gradient terms sum to exactly zero)
    idle = batch(list(range(1, 10)), list(range(1, 10)), list(range(10, 20)), self_negative=True)
    first = batch(list(range(10, 15)), list(range(10, 15)), list(range(20, 30)))    # step 1 (SGD), then idle
    late = batch(list(range(15, 20)), list(range(15, 20)), list(range(30, 40)))     # first touched at the last step
    plan = ([first] if learner == "sgd" else []) + [idle] * (N - 2) + [{k: np.concatenate([idle[k], late[k], first[k]])
                                                                       for k in idle}]
    for i, b in enumerate(plan):
        want = train_step(ora, opt_o, to_cpu_batch(b))
        got = float(m.train_step(to_device_batch(b)))
        if i in (0, 1, len(plan) - 1):
            np.testing.assert_allclose(got, want, rtol=1e-5, err_msg=f"loss at step {i + 1}")
    # 5,000 roundings of torch's per-step product against one closed form: a few ulp per thousand steps
    for (k, vo), (_, vp) in zip(ora.state_dict().items(), m.state_dict().items()):
        vo = vo.numpy()
        assert np.isfinite(vp.cpu().numpy()).all(), k
        assert_weights_close(vp.cpu().numpy(), vo, rtol=1e-4, atol=1e-7, outlier_frac=0, outlier_atol=1e-5,
                             err_msg=f"{learner} {k}")


def test_ml100k_epoch_under_adamw():
    """The ml-100k epoch of test_ml100k_epoch (TransE, d = 64, batch 2048, DeviceKGLoader) with AdamW(weight_decay):
    all 39 losses and the final weights against the oracle's dense torch.optim.AdamW."""
    from conftest import load_golden
    from test_loader_cpu import _loader

    from hopwise_b200.loader import DeviceKGLoader
    from hopwise_b200.sampler import KGSampler, MTStream, RecSampler

    g = load_golden("loader_ml100k.npz")
    U, I, E, R = (int(g[k]) for k in ("n_users", "n_items", "n_entities", "n_relations"))
    D, lr, wd = 64, 1e-3, 0.1
    loader_o, _ = _loader(g)
    ora = make_oracle_model("TransE", U, I, E, R, D)
    opt = make_optimizer(ora, lr=lr, weight_decay=wd, learner="adamw")
    want = np.array([float(train_step(ora, opt, b)) for b in loader_o])
    stream = MTStream(state=("MT19937", g["mt_key"], int(g["mt_pos"])))
    rec = RecSampler(g["used_user"].astype(np.int64), g["used_item"].astype(np.int64), U, I, stream=stream)
    kg = KGSampler(heads=g["kg_head"].astype(np.int64), tails=g["kg_tail"].astype(np.int64), entity_num=E,
                   stream=stream)
    loader = DeviceKGLoader(g["inter_user"], g["inter_item"], g["kg_head"], g["kg_rel"], g["kg_tail"], rec, kg,
                            batch_size=int(g["batch"]), seed=int(g["seed"]), device="cuda")
    m = make_product_model("TransE", U, I, E, R, D, learner="adamw", lr=lr, weight_decay=wd)
    got = np.array([float(m.train_step(b)) for b in loader])
    assert len(got) == len(want) == 39
    np.testing.assert_allclose(got, want, rtol=1e-5)
    _assert_model_close(m, ora, "ml-100k AdamW")


# ---- two GPUs (skipped with fewer) ------------------------------------------------------------------------------------
def _worker(rank, world, port, name, route, out_dir, owner, learner):
    import torch.distributed as dist

    from hopwise_b200.distributed import broadcast_weights, enable_row_sparse_data_parallel
    from test_gpu_distributed import SHAPES, _batches, _shard

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        dev = f"cuda:{rank}"
        m = make_product_model(name, device=dev, seed=2024 + rank, **HP[learner], learner=learner, **SHAPES[route])
        broadcast_weights(m)
        enable_row_sparse_data_parallel(m, multimem=owner, owner_adam=owner)
        batches, k = _batches(name, SHAPES[route])
        losses = []
        for b in batches:
            loss = m.calculate_loss(to_device_batch(_shard(b, rank, k), dev))
            loss.backward()
            losses.append(float(loss.item()))
        sd = {key: v.cpu().numpy() for key, v in m.state_dict().items()}
        np.savez(os.path.join(out_dir, f"rank{rank}.npz"), losses=np.array(losses), **sd)
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("name,route,owner,learner", [("TransE", "sparse", False, "adamw"), ("ComplEx", "dense", False, "adamw"),
                                                      ("TransE", "sparse", False, "sgd"), ("RotatE", "dense", False, "sgd"),
                                                      ("TransE", "dense", True, "adamw"), ("ComplEx", "sparse", True, "adamw")])
def test_two_rank_step_with_weight_decay_matches_single_gpu(name, route, owner, learner, tmp_path):
    """Row-sparse and dense exchange routes, and the owner-sharded AdamW step: replicas bit-identical, and equal to the
    single-GPU step on the concatenated batch."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp

    from test_gpu_distributed import SHAPES, _batches, _free_port

    mp.spawn(_worker, args=(2, _free_port(), name, route, str(tmp_path), owner, learner), nprocs=2, join=True)
    r0, r1 = np.load(tmp_path / "rank0.npz"), np.load(tmp_path / "rank1.npz")
    for key in (k_ for k_ in r0.files if k_ != "losses"):
        np.testing.assert_array_equal(r0[key], r1[key], err_msg=key)
    m = make_product_model(name, device="cuda:0", seed=2024, **HP[learner], learner=learner, **SHAPES[route])
    batches, k = _batches(name, SHAPES[route])
    losses = []
    for b in batches:
        loss = m.calculate_loss(to_device_batch(b, "cuda:0"))
        loss.backward()
        losses.append(float(loss.item()))
    np.testing.assert_allclose(0.5 * (r0["losses"] + r1["losses"]), losses, rtol=1e-5)
    for key, v in m.state_dict().items():
        assert_weights_close(r0[key], v.cpu().numpy(), rtol=1e-5, atol=5e-7, err_msg=f"{name} {key}")
