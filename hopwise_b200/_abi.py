"""ctypes binding of include/kge_b200.h -- the thin C-ABI boundary.

Nothing here computes: it marshals device pointers (``tensor.data_ptr()``), sizes and the
current CUDA stream into the plain-C entry points of libkge_b200.so and turns error codes
into Python exceptions.  There is no CPU fallback: if the library cannot be loaded the
import of any product path fails loudly.
"""

from __future__ import annotations

import ctypes as C
import os

from . import _build

KGE_ABI_VERSION = 8
MODEL_KINDS = {"TransE": 0, "DistMult": 1, "RotatE": 2, "ComplEx": 3, "TorusE": 4, "TransH": 5, "TransD": 6}


class KgeError(RuntimeError):
    pass


class kge_table_t(C.Structure):
    _fields_ = [
        ("rows", C.c_int64),
        ("parts", C.c_int32),
        ("_pad", C.c_int32),
        ("w", C.c_void_p * 2),
        ("m", C.c_void_p * 2),
        ("v", C.c_void_p * 2),
        ("g", C.c_void_p * 2),
        ("row_state", C.c_void_p),
    ]


class kge_model_t(C.Structure):
    _fields_ = [
        ("model", C.c_int32),
        ("d", C.c_int32),
        ("margin", C.c_float),
        ("ui_relation", C.c_int32),
        ("ui_relation_fullsort", C.c_int32),
        ("_pad", C.c_int32),
        ("n_items", C.c_int64),
        ("user", kge_table_t),
        ("entity", kge_table_t),
        ("relation", kge_table_t),
        ("adam_table", C.c_void_p),
        ("adam_table_len", C.c_int32),
        ("_pad2", C.c_int32),
    ]


class kge_batch_t(C.Structure):
    _fields_ = [
        ("user", C.c_void_p),
        ("item", C.c_void_p),
        ("neg_item", C.c_void_p),
        ("n_rec", C.c_int64),
        ("head", C.c_void_p),
        ("relation", C.c_void_p),
        ("tail", C.c_void_p),
        ("neg_tail", C.c_void_p),
        ("n_kg", C.c_int64),
        ("k_rec", C.c_int32),
        ("k_kg", C.c_int32),
    ]


class kge_adam_t(C.Structure):
    _fields_ = [
        ("lr", C.c_float),
        ("beta1", C.c_float),
        ("beta2", C.c_float),
        ("eps", C.c_float),
        ("step", C.c_int32),
        ("replay_cap", C.c_int32),
        ("optimizer", C.c_int32),
        ("reserved", C.c_int32),
    ]


OPTIMIZERS = {"adam": 0, "sgd": 1, "adagrad": 2, "rmsprop": 3}   # enum kge_optimizer


_P = C.c_void_p
_MP = C.POINTER(kge_model_t)
_BP = C.POINTER(kge_batch_t)
_AP = C.POINTER(kge_adam_t)

# name -> (restype, argtypes); every symbol include/kge_b200.h declares
PROTOTYPES = {
    "kge_abi_version": (C.c_int, []),
    "kge_last_error": (C.c_char_p, []),
    "kge_adam_table_fill": (C.c_int, [C.c_float, C.c_float, C.c_float, C.POINTER(C.c_float), C.c_int32]),
    "kge_train_forward": (C.c_int, [_MP, _BP, _AP, C.c_int, _P, _P]),
    "kge_adam_apply": (C.c_int, [_MP, _AP, C.c_float, _P, _P]),
    "kge_train_step": (C.c_int, [_MP, _BP, _AP, C.c_float, _P, _P]),
    "kge_adam_flush": (C.c_int, [_MP, _AP, _P]),
    "kge_grad_discard": (C.c_int, [_MP, C.c_int32, _P]),
    "kge_grad_pack": (C.c_int, [_MP, C.c_int32, C.c_int32, _P, _P, _P, _P]),
    "kge_grad_add": (C.c_int, [_MP, C.c_int32, C.c_int32, _P, _P, _P, C.c_int64, _P]),
    "kge_transh_project": (C.c_int, [_P, _P, C.c_int64, C.c_int32, _P, _P, C.c_int64, _P, _P]),
    "kge_transd_project": (C.c_int, [_P, _P, _P, C.c_int64, C.c_int32, _P, _P, C.c_int64, _P, _P]),
    "kge_predict": (C.c_int, [_MP, _P, _P, _P, C.c_int64, C.c_int, _P, _P]),
    "kge_full_sort_scores": (C.c_int, [_MP, _P, _P, C.c_int64, C.c_int, C.c_int64, _P, _P]),
    "kge_full_sort_topk_workspace_bytes": (C.c_int64, [_MP, C.c_int64, C.c_int64, C.c_int32]),
    "kge_full_sort_topk": (
        C.c_int,
        [_MP, _P, _P, C.c_int64, C.c_int, C.c_int64, _P, _P, C.c_int, C.c_int32, _P, _P, _P, C.c_int64, _P],
    ),
    "kge_full_sort_rank_workspace_bytes": (C.c_int64, [_MP, C.c_int64, C.c_int64, C.c_int64]),
    "kge_full_sort_rank_counts": (
        C.c_int,
        [_MP, _P, _P, C.c_int64, C.c_int, C.c_int64, _P, _P, C.c_int, _P, _P, _P, _P, _P, _P, C.c_int64, _P],
    ),
    "kge_copy_h2d_async": (C.c_int, [_P, _P, C.c_int64, _P]),
    "kge_multimem_all_reduce_f32": (C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P]),
    "kge_owner_adam_step": (
        C.c_int,
        [_P, _P, _P, _P, _P, _P, C.c_int64, C.c_int32, C.c_int32, _AP, C.c_float, _P, C.c_int32, _P, C.c_uint32, _P],
    ),
    "kge_multimem_all_reduce_fused_f32": (
        C.c_int, [_P, C.c_int64, C.c_int32, C.c_int32, _P, C.c_int32, _P, C.c_uint32, _P, C.c_int64, C.c_int32, _P]),
    "kge_mma_image_bytes": (C.c_int64, [_MP, C.c_int64, C.c_int32]),
    "kge_mma_prepare_targets": (C.c_int, [_MP, C.c_int64, _P, C.c_int64, C.c_int32, _P]),
    "kge_full_sort_topk_mma_workspace_bytes": (C.c_int64, [_MP, C.c_int64, C.c_int64, C.c_int32, C.c_int32]),
    "kge_full_sort_topk_mma": (
        C.c_int,
        [_MP, _P, _P, C.c_int64, C.c_int, C.c_int64, _P, _P, _P, C.c_int, C.c_int32, _P, _P, _P, _P, _P, C.c_int64, _P,
         C.c_int32, _P],
    ),
    "kge_topk_hits": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P, _P, _P]),
    "kge_topk_metric_sums": (C.c_int, [_P, C.c_int64, C.c_int32, _P, _P]),
    "kge_candidate_select_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64]),
    "kge_candidate_select": (
        C.c_int,
        [_P, _P, C.c_int64, _P, C.c_int64, C.c_int64, _P, _P, C.c_int32, _P, _P, _P, _P, _P, _P, C.c_int64, _P],
    ),
    "kge_gather_columns": (C.c_int, [_P, C.c_int32, C.c_int64, _P, C.c_int64, _P, _P, _P]),
    "kge_widen_ids_i32": (C.c_int, [_P, _P, C.c_int64, _P]),
    "kge_assemble_batch_workspace_bytes": (C.c_int64, [C.c_int64, C.c_int64, C.c_int32]),
    "kge_assemble_batch": (
        C.c_int,
        [_P, _P, _P, _P, C.c_int64, _P, C.c_int64, _P, _P, C.c_int64, _P, _P, C.c_int64, _P, C.c_int64, C.c_int32,
         _P, _P, C.c_int64, _P, _P, _P],
    ),
    "kge_sample_workspace_bytes": (C.c_int64, [C.c_int64]),
    "kge_sample_negatives": (
        C.c_int,
        [_P, _P, C.c_int64, C.c_int32, _P, _P, C.c_int64, C.c_int64, _P, _P, _P],
    ),
    "kge_sample_alias_workspace_bytes": (C.c_int64, [C.c_int64]),
    "kge_sample_negatives_alias": (
        C.c_int,
        [_P, _P, C.c_int64, C.c_int32, _P, _P, C.c_int64, _P, _P, _P, _P, _P, _P],
    ),
    "kge_mt19937_seed": (C.c_int, [_P, C.c_uint32, _P]),
}

_lib = None


def lib():
    """Load libkge_b200.so (building it in-tree first when nvcc is available and it is stale)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("KGE_B200_LIB")   # an experimental build (scripts/build_variant.sh)
    if not path:
        path = _build.LIB_PATH
        if not os.path.exists(path):
            path = _build.build()  # raises when nvcc is missing: no fallback
        elif _build.needs_build() and _build.have_nvcc():
            path = _build.build()  # a source is newer than the library: never test or time stale kernels
    handle = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(handle, name)  # AttributeError = ABI mismatch, deliberately loud
        fn.restype = res
        fn.argtypes = args
    if handle.kge_abi_version() != KGE_ABI_VERSION:
        raise KgeError(f"libkge_b200.so ABI {handle.kge_abi_version()} != binding {KGE_ABI_VERSION}")
    _lib = handle
    return _lib


def check(rc: int, what: str = "") -> None:
    if rc != 0:
        msg = lib().kge_last_error().decode(errors="replace")
        kind = "CUDA error" if rc > 0 else "argument error"
        raise KgeError(f"{what or 'libkge_b200'}: {kind} {rc}: {msg}")


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


class on_device:
    """``with on_device(dev):`` like torch.cuda.device(dev), but free when `dev` is already current (the usual case;
    torch's guard costs ~5 us of host time per use, which the reference-batch loop pays several times per step)."""

    __slots__ = ("idx", "prev")

    def __init__(self, device):
        import torch

        idx = getattr(device, "index", device)
        self.idx = torch.cuda.current_device() if idx is None else int(idx)

    def __enter__(self):
        import torch

        self.prev = torch.cuda.current_device()
        if self.prev != self.idx:
            torch.cuda.set_device(self.idx)

    def __exit__(self, *exc):
        if self.prev != self.idx:
            import torch

            torch.cuda.set_device(self.prev)
        return False


def stream_ptr():
    """cudaStream_t of torch's current stream on the current device (the raw getter: torch.cuda.current_stream()
    builds a Stream object, ~10 us of host time per call on the step's critical path)."""
    import torch

    raw = getattr(torch._C, "_cuda_getCurrentRawStream", None)
    if raw is not None:
        return raw(torch.cuda.current_device())
    return torch.cuda.current_stream().cuda_stream
