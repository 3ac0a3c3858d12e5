"""The training loader's batch order against the reference's own batches (no GPU).

`DeviceKGLoader` is driven on the CPU with the oracle's MT19937 samplers standing in for the two GPU
samplers: what is under test is the product's host logic -- the draw-for-draw replay of the reference's two
torch generators (EpochOrder, SURVEY.md H10), the KG-first / rec-second order, the phantom KG batch at the end
of an epoch and the epoch length -- against golden batches frozen from the unmodified reference pipeline
on ml-100k (tests/golden/make_golden_loader.py).  All 78 steps of two epochs are compared by CRC, five steps
element by element, and the sampler stream must end in the reference's final numpy state."""

import zlib

import numpy as np
import pytest
import torch

from conftest import load_golden
from hopwise_b200.loader import DeviceKGLoader, EpochOrder
from oracle import mt19937 as omt


class _OracleSampler:
    def __init__(self, gen, keys, values, n_keys, high):
        self.gen, self.high = gen, int(high)
        self.off, self.vals = omt.build_used_csr(keys, values, n_keys)

    def _draw(self, keys, num):
        out = omt.sample_by_key_ids(self.gen, keys.numpy(), num, self.off, self.vals, 1, self.high)
        return torch.from_numpy(out)

    def sample_by_entity_ids(self, heads, num=1):
        return self._draw(heads, num)

    def sample_by_user_ids(self, users, items=None, num=1):
        return self._draw(users, num)


def _loader(g):
    gen = omt.MT19937()
    gen.set_state(("MT19937", g["mt_key"], int(g["mt_pos"])))
    n_users, n_items, n_ent = int(g["n_users"]), int(g["n_items"]), int(g["n_entities"])
    rec = _OracleSampler(gen, g["used_user"], g["used_item"], n_users, n_items)
    kg = _OracleSampler(gen, g["kg_head"], g["kg_tail"], n_ent, n_ent)
    loader = DeviceKGLoader(g["inter_user"], g["inter_item"], g["kg_head"], g["kg_rel"], g["kg_tail"], rec, kg,
                            batch_size=int(g["batch"]), seed=int(g["seed"]), device="cpu", gather=lambda table, idx: table.index_select(0, idx))
    return loader, gen


def test_device_kg_loader_replays_reference_batches():
    g = load_golden("loader_ml100k.npz")
    loader, gen = _loader(g)
    assert len(loader) == g["crc"].shape[1] == 39
    for ep in range(2):
        n = 0
        for i, b in enumerate(loader):
            for c, key in enumerate(DeviceKGLoader.KEYS):
                v = b[key].numpy().astype(np.int64)
                assert v.shape[0] == int(g["lens"][ep, i, c]), (ep, i, key)
                assert zlib.crc32(v.tobytes()) == int(g["crc"][ep, i, c]), (ep, i, key)
                full = f"full_{ep}_{i}_{key}"
                if full in g.files:
                    np.testing.assert_array_equal(v, g[full].astype(np.int64), err_msg=full)
            n += 1
        assert n == 39
    # the shared stream ends where numpy's global generator ended in the reference run
    state = gen.get_state()
    np.testing.assert_array_equal(state[1], g["mt_key_end"])
    assert state[2] == int(g["mt_pos_end"])


def test_epoch_order_matches_torch_dataloader():
    """EpochOrder against a live torch DataLoader built like abstract_dataloader.py:47-73, including an
    epoch abandoned half way (the KG loader's situation) and an unshuffled loader."""
    from torch.utils.data import DataLoader

    for shuffle in (True, False):
        n, step, seed = 1000, 64, 7
        gen = torch.Generator()
        gen.manual_seed(seed)
        dl = DataLoader(list(range(n)), batch_size=step, shuffle=shuffle, generator=gen, collate_fn=lambda x: x)
        order = EpochOrder(n, step, seed, shuffle)
        for take in (None, 5, None):
            it = iter(dl)
            order.start()
            k = 0
            while take is None or k < take:
                want = next(it, None)
                got = order.next_indices()
                if want is None:
                    assert got is None
                    break
                assert got.tolist() == want
                k += 1


@pytest.mark.parametrize("n,step,world,shuffle", [(103, 16, 2, True), (103, 16, 4, False), (10, 64, 4, True),
                                                  (3, 8, 8, True), (2049, 2048, 8, True)])
def test_epoch_order_matches_torch_distributed_sampler(n, step, world, shuffle):
    """abstract_dataloader.py:59-64: DistributedSampler(list(range(n)), shuffle, drop_last=False) + step // world.
    No process group is needed to build the sampler when num_replicas and rank are given."""
    from torch.utils.data import DataLoader
    from torch.utils.data.distributed import DistributedSampler

    from hopwise_b200.loader import EpochOrder

    for rank in range(world):
        sampler = DistributedSampler(list(range(n)), num_replicas=world, rank=rank, shuffle=shuffle, drop_last=False)
        ref = DataLoader(list(range(n)), batch_size=max(1, step // world), sampler=sampler,
                         collate_fn=lambda b: torch.tensor(b))
        mine = EpochOrder(n, step, seed=2024, shuffle=shuffle, rank=rank, world=world)
        assert len(mine) == len(ref)
        for epoch in (0, 1, 5):
            sampler.set_epoch(epoch)
            mine.set_epoch(epoch)
            mine.start()
            want = list(ref)
            got = []
            while True:
                idx = mine.next_indices()
                if idx is None:
                    break
                got.append(idx)
            assert len(got) == len(want)
            for a, b in zip(got, want):
                assert torch.equal(a, b)


def test_pack_batch_layouts_on_the_host():
    """pack_batch: one contiguous buffer (int64, or int32 with narrow=True), padded to a multiple of four ids, named
    views at their offsets; ids beyond 32 bits are refused for the narrow layout."""
    from hopwise_b200.loader import pack_batch

    rng = np.random.default_rng(0)
    batch = {"user_id": rng.integers(0, 1000, 7), "item_id": rng.integers(0, 2 ** 31 - 1, 7), "neg_item_id": rng.integers(0, 9, 14)}
    for narrow in (False, True):
        pb = pack_batch(batch, pin=False, narrow=narrow)
        assert pb.narrow == narrow and pb.base.dtype == (torch.int32 if narrow else torch.int64)
        assert pb.base.numel() == 28 and pb.base.numel() % 4 == 0
        views = pb.views()
        assert list(views) == list(batch)
        for k, v in batch.items():
            np.testing.assert_array_equal(views[k].numpy().astype(np.int64), v)
        off = [pb.slices[k][0] for k in batch]
        assert off == [0, 7, 14]
    with pytest.raises(ValueError):
        pack_batch({"user_id": np.array([3, 2 ** 31])}, pin=False, narrow=True)
    assert pack_batch({"user_id": np.array([3, 2 ** 31])}, pin=False).base[1].item() == 2 ** 31


def test_device_loader_refuses_the_cpu_without_a_gather_hook():
    from hopwise_b200.loader import DeviceKGLoader

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        DeviceKGLoader([1], [1], [1], [1], [1], None, None, batch_size=1, seed=0, device="cpu")
    with pytest.raises(ValueError, match="candidate_num"):
        DeviceKGLoader([1], [1], [1], [1], [1], None, None, batch_size=1, seed=0, device="cpu", dynamic=True,
                       gather=lambda t, i: t.index_select(0, i))
