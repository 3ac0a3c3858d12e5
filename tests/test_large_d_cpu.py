"""Embedding sizes 513 to 1,024 without a GPU: the row geometry's Python mirror and the bounds of the C ABI.

kge_pick_rowcfg (csrc/common.cuh) maps every d from 1 to 1,024 to a row layout (VEC, G, NCH); the three layouts past
the old bound are (4, 32, 8) for d % 4 == 0 above 128 float4s and (1, 32, 16) / (1, 32, 32) for the other d above 256.
Every d the old geometry accepted keeps its layout.  LARGE_D_LADDER is the ladder tests/test_gpu_large_d.py runs."""

import ctypes as C

import pytest

from test_gpu_row_layouts import pick_rowcfg as pick_rowcfg_512

MAX_D = 1024
NEW_LAYOUTS = ((4, 32, 8), (1, 32, 16), (1, 32, 32))
LARGE_D_LADDER = (257, 301, 511, 513, 516, 600, 640, 767, 1000, 1021, 1024)
ALL_KINDS = ("TransE", "DistMult", "RotatE", "ComplEx", "TorusE", "TransH", "TransD")


def pick_rowcfg(d):
    """kge_pick_rowcfg (csrc/common.cuh): the (VEC, G, NCH) of a row of d floats, None outside 1 .. 1,024."""
    if d <= 0 or d > MAX_D:
        return None
    if d % 4 == 0:
        nv = d // 4
        if nv <= 8:
            return (4, 8, 1)
        if nv <= 16:
            return (4, 16, 1)
        n = (nv + 31) // 32
        return (4, 32, next(c for c in (1, 2, 4, 8) if n <= c))
    n = (d + 31) // 32
    return (1, 32, next(c for c in (1, 2, 4, 8, 16, 32) if n <= c))


def test_mirror_keeps_every_old_layout():
    """Every d the old geometry accepted maps to the layout it had; the rest of 1 .. 1,024 to a new layout."""
    for d in range(-1, MAX_D + 8):
        old, new = pick_rowcfg_512(d), pick_rowcfg(d)
        if old is not None:
            assert new == old, d
        elif 1 <= d <= MAX_D:
            assert new in NEW_LAYOUTS, d
        else:
            assert new is None, d
    assert {pick_rowcfg(d) for d in range(1, MAX_D + 1)} - {pick_rowcfg_512(d) for d in range(1, 513)} == set(NEW_LAYOUTS)


def test_ladder_reaches_every_new_layout_with_partial_and_empty_chunks():
    """Each new layout is reached at its first and its last chunk count, with a partial last chunk (fewer than 32
    units in the last used chunk) and with chunks no lane uses (the chunk count rounds up to a power of two)."""
    assert {pick_rowcfg(d) for d in LARGE_D_LADDER} == set(NEW_LAYOUTS)
    for vec, g, nch in NEW_LAYOUTS:
        ds = [d for d in LARGE_D_LADDER if pick_rowcfg(d) == (vec, g, nch)]
        units = [d // vec for d in ds]   # float4s or floats per row; lane l holds units l + 32 j
        chunks = [(u + 31) // 32 for u in units]
        assert min(chunks) == nch // 2 + 1 and max(chunks) == nch, (vec, nch)   # the first and the last chunk count
        assert any(u % 32 for u in units), (vec, nch)
        assert any((u + 31) // 32 < nch for u in units), (vec, nch)


def _model_struct(kind, d, rows=1000, weights=False):
    from hopwise_b200 import _abi

    m = _abi.kge_model_t()
    m.model = _abi.MODEL_KINDS[kind]
    m.d = d
    ph = 2 if kind in ("RotatE", "ComplEx", "TransD") else 1
    pr = 2 if kind in ("ComplEx", "TransH", "TransD") else 1
    for fam, parts in (("user", ph), ("entity", ph), ("relation", pr)):
        t = getattr(m, fam)
        t.rows, t.parts = rows, parts
        for p in range(parts):
            t.w[p] = 16 if weights else None   # (a refused call never dereferences them)
    return m


@pytest.mark.parametrize("kind", ALL_KINDS)
def test_full_sort_workspaces_accept_1_to_1024(kind):
    """The top-k (k = 20, 128 and the large-k buffers of 300) and rank workspace functions size a call at d = 1,024
    and at 1 and refuse 0 and 1,025, for every model kind."""
    from hopwise_b200 import _abi

    lib = _abi.lib()
    n, n_targets = 4096, 200_001
    for d, ok in ((1, True), (513, True), (1000, True), (1024, True), (0, False), (1025, False), (2048, False)):
        m = C.byref(_model_struct(kind, d))
        for k in (20, 128, 300):
            ws = lib.kge_full_sort_topk_workspace_bytes(m, n, n_targets, k)
            assert (ws >= 0) == ok, (kind, d, k, ws)
        ws = lib.kge_full_sort_rank_workspace_bytes(m, n, n_targets, 5 * n)
        assert (ws >= 0) == ok, (kind, d, ws)


@pytest.mark.parametrize("kind", ("TransE", "DistMult", "RotatE", "ComplEx"))
def test_tensor_core_path_keeps_its_k_bound(kind):
    """kge_mma_image_bytes keeps K = parts * d (+3 for the distance models), padded to 16, at most 640, whatever the
    CUDA-core bound: DistMult up to d = 640, TransE up to 637, RotatE / ComplEx up to 318 / 320."""
    from hopwise_b200 import _abi

    lib = _abi.lib()
    last = {"TransE": 637, "DistMult": 640, "RotatE": 318, "ComplEx": 320}[kind]
    for d in (last - 1, last, last + 1, 1000, 1024):
        m = C.byref(_model_struct(kind, d))
        img = lib.kge_mma_image_bytes(m, 200_001, 0)
        ws = lib.kge_full_sort_topk_mma_workspace_bytes(m, 4096, 200_001, 10, 0)
        assert (img >= 0) == (d <= last), (kind, d, img)
        assert (ws >= 0) == (d <= last), (kind, d, ws)


def test_entry_points_name_the_bound():
    """A model past 1,024 is refused with KGE_E_UNSUPPORTED before any device work, and the message names the
    bound: training, predict, the full-sort scorers and the projections."""
    from hopwise_b200 import _abi

    lib = _abi.lib()
    calls = {
        "kge_train_forward": lambda m: lib.kge_train_forward(m, None, None, 0, None, None),
        "kge_predict": lambda m: lib.kge_predict(m, None, None, None, 4, 1, None, None),
        "kge_full_sort_scores": lambda m: lib.kge_full_sort_scores(m, None, None, 4, 1, 100, None, None),
        "kge_full_sort_topk": lambda m: lib.kge_full_sort_topk(m, None, None, 4, 1, 100, None, None, 1, 10, None, None,
                                                               None, 0, None),
        "kge_full_sort_rank_counts": lambda m: lib.kge_full_sort_rank_counts(m, None, None, 4, 1, 100, None, None, 1,
                                                                             None, None, None, None, None, None, 0,
                                                                             None),
    }
    for kind in ("TransE", "ComplEx"):
        m = C.byref(_model_struct(kind, 1025, weights=True))
        for name, call in calls.items():
            assert call(m) == -2, (kind, name)
            assert b"embedding_size 1025 unsupported (1 to 1024)" in lib.kge_last_error(), (kind, name)
    buf = C.c_void_p(16)
    assert lib.kge_transh_project(buf, None, 4, 1025, buf, None, 0, buf, None) == -2
    assert b"(1 to 1024)" in lib.kge_last_error()
    assert lib.kge_transd_project(buf, buf, None, 4, 1025, buf, None, 0, buf, None) == -2
    assert b"(1 to 1024)" in lib.kge_last_error()
