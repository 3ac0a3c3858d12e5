"""CPU-side checks of the sampled-evaluation entry point: exported, sized from the candidate count, and refusing
bad arguments with an error code (C ABI) or a ValueError (model API) before any device work."""

import numpy as np
import pytest
import torch


def test_candidate_select_is_exported_and_sized_from_the_candidates():
    from hopwise_b200 import _abi

    lib = _abi.lib()
    assert lib.kge_abi_version() == 8
    assert lib.kge_candidate_select_workspace_bytes(10, 1000) == 8000
    assert lib.kge_candidate_select_workspace_bytes(0, 0) == 0
    assert lib.kge_candidate_select_workspace_bytes(-1, 10) == -1
    assert lib.kge_candidate_select_workspace_bytes(10, -1) == -1


def _call(lib, **kw):
    args = dict(scores=None, items=None, n_cand=4, off=None, n=2, n_targets=100, pos_off=None, pos_items=None, k=10,
                ids=None, top=None, greater=None, equal=None, n_unmasked=None, ws=None, ws_bytes=32)
    args.update(kw)
    return lib.kge_candidate_select(*args.values(), None)


def test_candidate_select_refuses_bad_arguments():
    from hopwise_b200 import _abi

    lib = _abi.lib()
    fake = 0x1000   # never dereferenced: every refusal below happens on the host
    ok = dict(scores=fake, items=fake, off=fake, ws=fake)
    cases = {
        "NULL cand_off": dict(ok, off=None),
        "NULL scores": dict(ok, scores=None),
        "NULL cand_items": dict(ok, items=None),
        "NULL workspace": dict(ok, ws=None),
        "workspace too small": dict(ok, ws_bytes=31),
        "k below 1": dict(ok, k=0),
        "negative k": dict(ok, k=-3),
        "k above n_targets": dict(ok, k=101),
        "NULL positives with rank outputs": dict(ok, greater=fake, equal=fake),
        "greater without equal": dict(ok, greater=fake, pos_off=fake, pos_items=fake),
        "negative n": dict(ok, n=-1),
        "no targets": dict(ok, n_targets=0),
    }
    for what, kw in cases.items():
        assert _call(lib, **kw) == -1, what   # KGE_E_ARG
        assert lib.kge_last_error(), what
    assert _call(lib, n=0, k=0) == -1        # k is checked for an empty call too
    assert _call(lib, n=0) == 0              # nothing to do: no pointer is needed


def test_model_api_checks_offsets_and_k_before_device_work():
    from kge_helpers import make_product_model

    m = make_product_model("DistMult", 10, 50, 60, 4, 16, device="cpu")
    users, items = torch.tensor([1, 1, 2, 2, 2]), torch.tensor([3, 4, 5, 6, 3])
    with pytest.raises(ValueError, match="cand_off"):
        m.candidate_topk(users, items, torch.tensor([0, 2, 4]), 3)          # ends at 4, 5 candidates
    with pytest.raises(ValueError, match="cand_off"):
        m.candidate_topk(users, items, torch.tensor([1, 2, 5]), 3)          # does not start at 0
    with pytest.raises(ValueError, match="cand_off"):
        m.candidate_meanrank(users, items, np.array([[0, 5]]), [0, 1], [3])
    with pytest.raises(ValueError, match="k=0"):
        m.candidate_topk(users, items, torch.tensor([0, 2, 5]), 0)
    with pytest.raises(ValueError, match="k=51"):
        m.candidate_topk(users, items, torch.tensor([0, 2, 5]), 51)
    with pytest.raises(ValueError, match="one entry per candidate"):
        m.candidate_topk(users[:4], items, torch.tensor([0, 2, 5]), 3)
    # well-formed arguments reach the device check: no CPU fallback
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.candidate_topk(users, items, torch.tensor([0, 2, 5]), 3)


def test_collect_sampled_refuses_ungrouped_candidate_rows():
    from hopwise_b200 import evaluator as ev
    from kge_helpers import make_product_model

    m = make_product_model("DistMult", 10, 50, 60, 4, 16, device="cpu")
    inter = {"user_id": torch.tensor([1, 2, 1]), "item_id": torch.tensor([3, 4, 5])}
    with pytest.raises(ValueError, match="grouped by user"):
        ev.collect_sampled(m, [(inter, [0, 1, 0], torch.tensor([0, 1]), torch.tensor([3, 4]))], 2)
