"""DeviceKGLoader on the GPU (MT19937 sampler kernels, device-side gathers) against the reference's batches:
every id vector of two ml-100k epochs bit-exact, final sampler state equal to numpy's."""

import zlib

import numpy as np
import pytest
import torch

from conftest import load_golden

pytestmark = pytest.mark.gpu


def test_device_kg_loader_gpu_matches_reference_epochs():
    from hopwise_b200.loader import DeviceKGLoader
    from hopwise_b200.sampler import KGSampler, MTStream, RecSampler

    g = load_golden("loader_ml100k.npz")
    stream = MTStream(state=("MT19937", g["mt_key"], int(g["mt_pos"])))
    n_users, n_items, n_ent = int(g["n_users"]), int(g["n_items"]), int(g["n_entities"])
    rec = RecSampler(g["used_user"].astype(np.int64), g["used_item"].astype(np.int64), n_users, n_items, stream=stream)
    kg = KGSampler(heads=g["kg_head"].astype(np.int64), tails=g["kg_tail"].astype(np.int64), entity_num=n_ent,
                   stream=stream)
    loader = DeviceKGLoader(g["inter_user"], g["inter_item"], g["kg_head"], g["kg_rel"], g["kg_tail"], rec, kg,
                            batch_size=int(g["batch"]), seed=int(g["seed"]), device="cuda")
    for ep in range(2):
        steps = 0
        for i, b in enumerate(loader):
            for c, key in enumerate(DeviceKGLoader.KEYS):
                assert b[key].is_cuda and b[key].dtype == torch.int64
                v = b[key].cpu().numpy()
                assert zlib.crc32(v.tobytes()) == int(g["crc"][ep, i, c]), (ep, i, key)
            steps += 1
        assert steps == 39
    state = stream.get_state()
    np.testing.assert_array_equal(state[1], g["mt_key_end"])
    assert state[2] == int(g["mt_pos_end"])


def test_device_kg_loader_feeds_the_fused_step():
    """A short training run driven by the device loader: finite, decreasing loss."""
    from hopwise_b200.loader import DeviceKGLoader
    from hopwise_b200.sampler import KGSampler, MTStream, RecSampler
    from kge_helpers import make_product_model

    g = load_golden("loader_ml100k.npz")
    stream = MTStream(seed=2024)
    n_users, n_items, n_ent, n_rel = (int(g[k]) for k in ("n_users", "n_items", "n_entities", "n_relations"))
    rec = RecSampler(g["used_user"].astype(np.int64), g["used_item"].astype(np.int64), n_users, n_items, stream=stream)
    kg = KGSampler(heads=g["kg_head"].astype(np.int64), tails=g["kg_tail"].astype(np.int64), entity_num=n_ent,
                   stream=stream)
    loader = DeviceKGLoader(g["inter_user"], g["inter_item"], g["kg_head"], g["kg_rel"], g["kg_tail"], rec, kg,
                            batch_size=2048, seed=2024)
    m = make_product_model("TransE", n_users, n_items, n_ent, n_rel, 64, lr=1e-2)   # relation_num counts [UI-Relation]
    epoch_loss = []
    for _ in range(3):
        tot = 0.0
        for b in loader:
            loss = m.calculate_loss(b)
            tot += float(loss.item())
            loss.backward()
        epoch_loss.append(tot)
    assert np.isfinite(epoch_loss).all() and epoch_loss[-1] < epoch_loss[0]


def test_dynamic_negative_sampling_matches_oracle():
    """train_neg_sample_args = {dynamic: True, candidate_num: 3, sample_num: 2} (abstract_dataloader.py:166-183):
    candidates from the shared stream (KG draw first), scored by the model, best one kept per row; positives
    repeat once per negative.  Checked against the oracle sampler + oracle model on the same index stream."""
    from hopwise_b200.loader import DeviceKGLoader, EpochOrder
    from hopwise_b200.sampler import KGSampler, MTStream, RecSampler
    from kge_helpers import make_oracle_model, make_product_model
    from oracle import mt19937 as omt

    U, I, E, R, d, B, num, cn = 300, 200, 500, 6, 32, 512, 2, 3
    rng = np.random.default_rng(17)
    iu, ii = rng.integers(1, U, 1800), rng.integers(1, I, 1800)
    kh, kr, kt = rng.integers(1, E, 2500), rng.integers(1, R - 1, 2500), rng.integers(1, E, 2500)
    stream = MTStream(seed=5)
    rec = RecSampler(iu, ii, U, I, stream=stream)
    kg = KGSampler(heads=kh, tails=kt, entity_num=E, stream=stream)
    loader = DeviceKGLoader(iu, ii, kh, kr, kt, rec, kg, batch_size=B, seed=7, neg_sample_num=num, dynamic=True,
                            candidate_num=cn)
    m = make_product_model("TransE", U, I, E, R, d)
    ora = make_oracle_model("TransE", U, I, E, R, d)
    with pytest.raises(RuntimeError):
        next(iter(loader))
    loader = DeviceKGLoader(iu, ii, kh, kr, kt, rec, kg, batch_size=B, seed=7, neg_sample_num=num, dynamic=True,
                            candidate_num=cn)
    stream.seed(5)
    loader.get_model(m)

    gen = omt.MT19937(5)
    kg_off, kg_vals = omt.build_used_csr(kh, kt, E)
    rec_off, rec_vals = omt.build_used_csr(iu, ii, U)
    rec_o, kg_o = EpochOrder(len(iu), B, 7, True), EpochOrder(len(kh), B, 7, True)
    kg_o.start()
    rec_o.start()
    steps, exact, rows = 0, 0, 0
    for b in loader:
        kidx = kg_o.next_indices().numpy()
        np.testing.assert_array_equal(b["neg_tail_id"].cpu().numpy(),
                                      omt.sample_by_key_ids(gen, kh[kidx], 1, kg_off, kg_vals, 1, E))
        ridx = rec_o.next_indices().numpy()
        n = len(ridx)
        cand = omt.sample_by_key_ids(gen, iu[ridx], num * cn, rec_off, rec_vals, 1, I)
        with torch.no_grad():
            sc = ora.predict({"user_id": torch.from_numpy(np.tile(iu[ridx], num * cn)),
                              "item_id": torch.from_numpy(cand)}).numpy().reshape(cn, -1)
        want = cand.reshape(cn, -1)[sc.argmax(0), np.arange(num * n)]
        got = b["neg_item_id"].cpu().numpy()
        assert got.shape == (num * n,)
        np.testing.assert_array_equal(b["user_id"].cpu().numpy(), np.tile(iu[ridx], num))
        np.testing.assert_array_equal(b["item_id"].cpu().numpy(), np.tile(ii[ridx], num))
        same = got == want
        # a row may pick another candidate only when the two score within fp32 rounding of each other
        for j in np.flatnonzero(~same):
            col = cand.reshape(cn, -1)[:, j]
            pick = np.flatnonzero(col == got[j])
            assert len(pick) and sc[pick[0], j] >= sc[:, j].max() - 1e-5 * np.abs(sc[:, j]).max()
        exact += int(same.sum())
        rows += num * n
        steps += 1
    assert steps == 4 and exact >= 0.99 * rows
    # like the reference (knowledge_dataloader.py:137-145) the loader draws a KG batch before it finds the
    # recommendation side exhausted: one more KG draw on the stream
    omt.sample_by_key_ids(gen, kh[kg_o.next_indices().numpy()], 1, kg_off, kg_vals, 1, E)
    st = stream.get_state()
    np.testing.assert_array_equal(st[1], gen.key)
    assert st[2] == gen.pos


def test_gather_columns_kernel():
    """kge_gather_columns against numpy fancy indexing: 1..8 columns, empty index, repeated and boundary rows, and the
    out-of-range flag."""
    import ctypes as C

    from hopwise_b200 import _abi

    lib = _abi.lib()
    rng = np.random.default_rng(0)
    rows = 100_003
    for nc, n in ((1, 1), (3, 2048), (8, 70_001), (2, 0)):
        cols = [torch.from_numpy(rng.integers(0, 1 << 40, rows)).cuda() for _ in range(nc)]
        idx = rng.integers(0, rows, n)
        if n > 2:
            idx[0], idx[1], idx[2] = 0, rows - 1, rows - 1
        idx_d = torch.from_numpy(idx).cuda()
        out = torch.full((nc, n), -1, dtype=torch.int64, device="cuda")
        src = (C.c_void_p * nc)(*[c.data_ptr() for c in cols])
        dst = (C.c_void_p * nc)(*[out.data_ptr() + 8 * n * c for c in range(nc)])
        status = torch.zeros(1, dtype=torch.int32, device="cuda")
        _abi.check(lib.kge_gather_columns(src, nc, rows, idx_d.data_ptr(), n, dst, status.data_ptr(), _abi.stream_ptr()),
                   "kge_gather_columns")
        for c in range(nc):
            np.testing.assert_array_equal(out[c].cpu().numpy(), cols[c].cpu().numpy()[idx])
        assert status.item() == 0
    bad = torch.tensor([5, rows, -1, 7], device="cuda")
    out = torch.full((1, 4), -1, dtype=torch.int64, device="cuda")
    src = (C.c_void_p * 1)(cols[0].data_ptr())
    dst = (C.c_void_p * 1)(out.data_ptr())
    _abi.check(lib.kge_gather_columns(src, 1, rows, bad.data_ptr(), 4, dst, status.data_ptr(), _abi.stream_ptr()), "gather")
    assert status.item() == 1 and out[0, 1].item() == -1 and out[0, 0].item() == cols[0][5].item()
    assert lib.kge_gather_columns(src, 9, rows, bad.data_ptr(), 4, dst, None, _abi.stream_ptr()) != 0


def test_one_call_batch_assembly_equals_the_piecewise_path():
    """kge_assemble_batch (one library call per batch) against the loader's piecewise path (gather hook + separate
    sampler calls): same batches, 2 negatives per interaction, KG wrap-around, same final sampler state."""
    from hopwise_b200.loader import DeviceKGLoader
    from hopwise_b200.sampler import KGSampler, MTStream, RecSampler

    U, I, E, R, B, num = 300, 200, 500, 6, 256, 2
    rng = np.random.default_rng(23)
    iu, ii = rng.integers(1, U, 3000), rng.integers(1, I, 3000)
    kh, kr, kt = rng.integers(1, E, 1100), rng.integers(1, R - 1, 1100), rng.integers(1, E, 1100)   # 5 KG batches < 12 rec

    def run(fast):
        stream = MTStream(seed=9)
        rec = RecSampler(iu, ii, U, I, stream=stream)
        kg = KGSampler(heads=kh, tails=kt, entity_num=E, stream=stream)
        hook = None if fast else (lambda table, idx: table.index_select(0, idx))
        loader = DeviceKGLoader(iu, ii, kh, kr, kt, rec, kg, batch_size=B, seed=3, neg_sample_num=num, gather=hook)
        assert loader._fast_path() == fast
        out = []
        for _ in range(2):
            out += [{k: v.cpu().numpy().copy() for k, v in b.items()} for b in loader]
        return out, stream.get_state()

    a, sa = run(True)
    b, sb = run(False)
    assert len(a) == len(b) == 24
    for x, y in zip(a, b):
        assert set(x) == set(y) == set(DeviceKGLoader.KEYS)
        for k in x:
            np.testing.assert_array_equal(x[k], y[k], err_msg=k)
        assert len(x["user_id"]) == len(x["neg_item_id"]) == num * (len(x["neg_item_id"]) // num)
    np.testing.assert_array_equal(sa[1], sb[1])
    assert sa[2] == sb[2]
