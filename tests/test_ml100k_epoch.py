"""BASELINE config 1's first training epoch -- TransE, d = 64, batch 2048, seed 2024 on ml-100k -- without hopwise.

The reference's 39 batches of epoch 0 are rebuilt from tests/golden/loader_ml100k.npz (the CPU replay of
test_loader_cpu for the oracle, DeviceKGLoader with the device MT19937 samplers for the product; both are checked
batch for batch against the reference's own batches by the loader tests).  The epoch loss is compared with the one
hopwise's own KGTrainer logged for this epoch, and every step of the fused model -- driven the way FusedKGTrainer
drives it (train_step) and the way hopwise's unchanged KGTrainer drives it (calculate_loss, backward) -- with the
oracle's step."""

import numpy as np
import pytest
import torch

from conftest import load_golden
from kge_helpers import make_oracle_model, make_product_model
from oracle.kge_torch import make_optimizer, train_step
from test_loader_cpu import _loader

# hopwise 0.9.1.post1: KGTrainer._train_epoch(train_data, 0) of TransE on the CPU, through hopwise's Config /
# create_dataset / data_preparation on its bundled ml-100k with the config above (bench.py --impl reference,
# extras.cfg1_ml100k_pipeline.epoch_loss in profiles/r2_bench_reference_n1.json)
REF_EPOCH_LOSS = 36.800033152103424
D = 64


@pytest.fixture(scope="module")
def g():
    return load_golden("loader_ml100k.npz")


def _shapes(g):
    return tuple(int(g[k]) for k in ("n_users", "n_items", "n_entities", "n_relations"))


@pytest.fixture(scope="module")
def oracle_losses(g):
    loader, _ = _loader(g)
    ora = make_oracle_model("TransE", *_shapes(g), D)
    opt = make_optimizer(ora)
    return np.array([float(train_step(ora, opt, b)) for b in loader])


def test_oracle_epoch_loss_matches_the_reference(oracle_losses):
    assert len(oracle_losses) == 39
    np.testing.assert_allclose(oracle_losses.sum(), REF_EPOCH_LOSS, rtol=1e-6)


@pytest.mark.gpu
@pytest.mark.parametrize("drive", ["train_step", "calculate_loss"])
def test_fused_epoch_matches_the_oracle_and_the_reference(g, oracle_losses, drive):
    from hopwise_b200.loader import DeviceKGLoader
    from hopwise_b200.sampler import KGSampler, MTStream, RecSampler

    U, I, E, R = _shapes(g)
    stream = MTStream(state=("MT19937", g["mt_key"], int(g["mt_pos"])))
    rec = RecSampler(g["used_user"].astype(np.int64), g["used_item"].astype(np.int64), U, I, stream=stream)
    kg = KGSampler(heads=g["kg_head"].astype(np.int64), tails=g["kg_tail"].astype(np.int64), entity_num=E,
                   stream=stream)
    loader = DeviceKGLoader(g["inter_user"], g["inter_item"], g["kg_head"], g["kg_rel"], g["kg_tail"], rec, kg,
                            batch_size=int(g["batch"]), seed=int(g["seed"]), device="cuda")
    m = make_product_model("TransE", U, I, E, R, D)
    got = []
    for b in loader:
        if drive == "train_step":
            loss = m.train_step(b)
        else:
            loss = m.calculate_loss(b)
            loss.backward()
        got.append(float(loss.detach()))
    got = np.array(got)
    assert len(got) == 39
    np.testing.assert_allclose(got, oracle_losses, rtol=1e-5)
    np.testing.assert_allclose(got.sum(), REF_EPOCH_LOSS, rtol=1e-5)
    assert m._step == 39 and all(p.is_cuda for p in m.parameters())
    torch.cuda.synchronize()
