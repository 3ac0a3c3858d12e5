"""CPU-side checks of the boundary: the library builds for sm_100a, loads without a GPU and
exports every symbol include/kge_b200.h declares; the ctypes structs match the header."""

import ctypes as C
import os
import re

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "kge_b200.h")


def _declared_functions():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(kge_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from hopwise_b200 import _abi, _build

    _build.build()
    lib = _abi.lib()
    names = _declared_functions()
    assert len(names) >= 15
    for n in names:
        assert hasattr(lib, n), f"{n} declared in kge_b200.h but not exported"
    assert set(names) == set(_abi.PROTOTYPES), "ctypes prototypes and header disagree"
    assert lib.kge_abi_version() == _abi.KGE_ABI_VERSION


def test_struct_sizes_match_header_field_lists():
    from hopwise_b200 import _abi

    # sizes computed from the header's field lists (LP64)
    assert C.sizeof(_abi.kge_table_t) == 8 + 4 + 4 + 4 * 16 + 8
    assert C.sizeof(_abi.kge_model_t) == 4 * 6 + 8 + 3 * C.sizeof(_abi.kge_table_t) + 8 + 8
    assert C.sizeof(_abi.kge_batch_t) == 3 * 8 + 8 + 4 * 8 + 8 + 8
    assert C.sizeof(_abi.kge_adam_t) == 32


def test_host_only_entry_points():
    from hopwise_b200 import _abi

    lib = _abi.lib()
    n = lib.kge_adam_table_fill(1e-3, 0.9, 0.999, None, 0)
    assert n > 20000
    buf = (C.c_float * (2 * n))()
    lib.kge_adam_table_fill(1e-3, 0.9, 0.999, buf, n)
    assert abs(buf[2] - 1e-3 / (1 - 0.9)) < 1e-8  # lr / (1 - b1^1)
    assert abs(buf[3] - 1 / (1 - 0.999) ** 0.5) < 1e-3
    assert abs(buf[2 * (n - 1)] - 1e-3) < 1e-10 and abs(buf[2 * (n - 1) + 1] - 1.0) < 1e-6
    assert lib.kge_sample_workspace_bytes(100) == 800
    assert lib.kge_sample_alias_workspace_bytes(100) == 2000       # two open-slot lists, round indices, 2 words / slot
    assert lib.kge_assemble_batch_workspace_bytes(2048, 2048, 3) == lib.kge_sample_workspace_bytes(2048 * 3)
    assert lib.kge_assemble_batch_workspace_bytes(-1, 0, 1) == -1
    # the entry points added in round 2 refuse bad arguments the same way
    assert lib.kge_gather_columns(None, 9, 10, None, 4, None, None, None) < 0
    assert lib.kge_widen_ids_i32(None, None, 8, None) < 0
    assert lib.kge_transd_project(None, None, None, 4, 16, None, None, 0, None, None) < 0
    assert lib.kge_transh_project(None, None, 4, 16, None, None, 0, None, None) < 0
    assert lib.kge_sample_negatives_alias(None, None, 4, 1, None, None, 0, None, None, None, None, None, None) < 0
    assert lib.kge_owner_adam_step(None, None, None, None, None, None, 16, 0, 2, None, 1.0, None, 0, None, 1, None) < 0
    # argument errors come back as codes + message, never exceptions or crashes
    assert lib.kge_train_forward(None, None, None, 1, None, None) < 0
    assert b"NULL" in lib.kge_last_error()


def _model_struct(kind, d, rows=1000):
    from hopwise_b200 import _abi

    m = _abi.kge_model_t()
    m.model = _abi.MODEL_KINDS[kind]
    m.d = d
    parts = 2 if kind in ("RotatE", "ComplEx") else 1
    for fam in ("user", "entity", "relation"):
        t = getattr(m, fam)
        t.rows, t.parts = rows, parts
    m.relation.parts = 2 if kind == "ComplEx" else 1
    return m


@pytest.mark.parametrize("kind,d,tn", [("DistMult", 64, 128), ("ComplEx", 64, 128), ("TransE", 100, 128),
                                       ("RotatE", 120, 64), ("ComplEx", 128, 64)])
def test_sweep_plan_sizes(kind, d, tn):
    """plan_mma (csrc/mma_topk.cu) without a GPU: the operand image is tiles of TN rows of the padded K (fp16), the
    workspace holds one 128-entry list per (row, split, slice), the per-row scalars and bitmap, the row map and
    the partial lists of the device-gated exact fallback; K > 640 and k > 32 are refused."""
    from hopwise_b200 import _abi

    lib = _abi.lib()
    m = _model_struct(kind, d)
    n_targets = 200_001
    parts = 2 if kind in ("RotatE", "ComplEx") else 1
    kd = parts * d + (3 if kind in ("TransE", "RotatE") else 0)
    kp = (kd + 15) // 16 * 16
    tiles = (n_targets + tn - 1) // tn
    tiles128 = (n_targets + 127) // 128
    img = lib.kge_mma_image_bytes(C.byref(m), n_targets, 0)
    assert img == 128 + tiles * tn * kp * 2 + (n_targets * 4 + 127) // 128 * 128
    n, k = 75_776, 20
    ws = lib.kge_full_sort_topk_mma_workspace_bytes(C.byref(m), n, n_targets, k, 0)
    rows_pad = (n + 255) // 256 * 256
    wpr = (tiles * (tn // 32) + 31) // 32
    ncol = 2 if (tn == 128 and kp > 80) else 1           # shape (f): two column slices per tile
    a16 = lambda x: (x + 15) // 16 * 16                  # noqa: E731
    lists = ncol * rows_pad                              # one split at this size
    exact_tiles = (n_targets + 127) // 128               # the fallback: 1024 rows x 48 target splits, the rest 1 list
    tps = (exact_tiles + 47) // 48
    exact = (1024 * ((exact_tiles + tps - 1) // tps) * k + (n - 1024) * k) * 8
    want = (a16(lists * 128 * 8) + 2 * a16(lists * 4) + 2 * a16(rows_pad * 4) + a16(rows_pad * wpr * 4)
            + a16(rows_pad * 4) + a16(exact))
    assert ws == want
    assert lib.kge_full_sort_topk_mma_workspace_bytes(C.byref(m), n, n_targets, 64, 0) == -1    # k > 32
    big = _model_struct("ComplEx", 160)                                                     # K = 320: shape (k)
    assert lib.kge_mma_image_bytes(C.byref(big), n_targets, 0) == 128 + tiles128 * 128 * 320 * 2 + (n_targets * 4 + 127) // 128 * 128
    huge = _model_struct("ComplEx", 330)
    assert lib.kge_mma_image_bytes(C.byref(huge), n_targets, 0) == -1                         # K = 672 > 640
    # a forced shape is accepted ('c' always fits), an unknown one is refused
    assert lib.kge_mma_image_bytes(C.byref(m), n_targets, ord("c")) > 0
    assert lib.kge_mma_image_bytes(C.byref(m), n_targets, ord("x")) == -1


@pytest.mark.parametrize("kind,project", [("TransH", b"kge_transh_project"), ("TransD", b"kge_transd_project")])
def test_projected_models_are_refused_by_the_scorers(kind, project):
    """TransH and TransD score as TransE over the rows their projection entry point writes: every scoring entry
    point refuses the model kind itself (KGE_E_UNSUPPORTED, naming that entry point) before it looks at a table."""
    from hopwise_b200 import _abi

    lib = _abi.lib()
    m = C.byref(_model_struct(kind, 16))
    calls = {
        "kge_predict": lambda: lib.kge_predict(m, None, None, None, 4, 1, None, None),
        "kge_full_sort_scores": lambda: lib.kge_full_sort_scores(m, None, None, 4, 1, 100, None, None),
        "kge_full_sort_topk": lambda: lib.kge_full_sort_topk(m, None, None, 4, 1, 100, None, None, 1, 10, None, None,
                                                             None, 0, None),
        "kge_full_sort_rank_counts": lambda: lib.kge_full_sort_rank_counts(m, None, None, 4, 1, 100, None, None, 1, None,
                                                                           None, None, None, None, None, 0, None),
    }
    for name, call in calls.items():
        assert call() == -2, name   # KGE_E_UNSUPPORTED
        assert project in lib.kge_last_error(), name


def test_product_has_no_cpu_fallback_and_no_oracle_import():
    import torch

    from kge_helpers import make_product_model, random_batch, to_cpu_batch
    import numpy as np

    m = make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu")
    b = to_cpu_batch(random_batch(np.random.default_rng(0), 10, 8, 20, 5, 4, 4))
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.calculate_loss(b)
    with pytest.raises(RuntimeError, match="CUDA only"):
        m.full_sort_predict({"user_id": torch.arange(1, 3)})
    pkg = os.path.join(ROOT, "hopwise_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle\b", src, flags=re.M), f"{f} imports the oracle"


def test_state_dict_keys_match_reference_names(golden):
    from kge_helpers import make_product_model

    for name in ("TransE", "RotatE", "DistMult", "ComplEx", "TorusE", "TransH", "TransD"):
        g = golden(f"model_{name}_d10.npz")
        U, I, E, R, d = (int(x) for x in g["shape"])
        m = make_product_model(name, U, I, E, R, d, device="cpu")
        want = sorted(k[5:] for k in g.files if k.startswith("init/"))
        assert sorted(m.state_dict().keys()) == want
        # same seed, same constructor order => the reference's initial weights, bit for bit
        for k, v in m.state_dict().items():
            assert (v.numpy() == g["init/" + k]).all(), (name, k)


def test_unsupported_configs_are_refused():
    from kge_helpers import ShapeDataset, make_product_model
    import hopwise_b200
    from kge_helpers import BASE_CONFIG

    # TransH reads relation_embedding.weight[-1] but norm_vec(ui_relation): one row only when the token is last
    cfg = dict(BASE_CONFIG, embedding_size=16, margin=1.0, device=torch.device("cpu"))
    with pytest.raises(NotImplementedError, match="UI-Relation"):
        hopwise_b200.TransH(cfg, ShapeDataset(10, 8, 20, 5, ui_token_id=2))
    hopwise_b200.TransH(cfg, ShapeDataset(10, 8, 20, 5))

    with pytest.raises(NotImplementedError):
        make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu", learner="sparse_adam")
    for learner, want in (("sgd", "sgd"), ("Adagrad", "adagrad"), ("rmsprop", "rmsprop"), ("adamw", "adam")):
        assert make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu", learner=learner).learner == want
    with pytest.warns(UserWarning, match="unrecognized learner"):
        assert make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu", learner="lion").learner == "adam"
    with pytest.raises(NotImplementedError):
        make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu", weight_decay=0.1)
    with pytest.raises(NotImplementedError):
        make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu", clip_grad_norm={"max_norm": 5})


def test_entry_points_the_reference_does_not_offer_are_refused_before_any_device_work():
    """TransH has no KG scoring in the reference (transh.py); TransD's dense KG full-sort is not mirrored
    (transd.py:192-217).  Both refuse by name, on any device."""
    from kge_helpers import make_product_model

    h = make_product_model("TransH", 10, 8, 20, 5, 16, device="cpu")
    d = make_product_model("TransD", 10, 8, 20, 5, 16, device="cpu")
    b = {"head_id": torch.tensor([1]), "relation_id": torch.tensor([1]), "tail_id": torch.tensor([2])}
    for call in (lambda: h.predict_kg(b), lambda: h.full_sort_predict_kg(b), lambda: d.full_sort_predict_kg(b),
                 lambda: d.full_sort_topk(torch.tensor([1]), 3, relation_ids=torch.tensor([1]))):
        with pytest.raises(NotImplementedError):
            call()
    # and the compute paths of every model refuse CPU tensors instead of falling back
    for m in (h, d):
        with pytest.raises(RuntimeError, match="CUDA only"):
            m.predict({"user_id": torch.tensor([1]), "item_id": torch.tensor([2])})
