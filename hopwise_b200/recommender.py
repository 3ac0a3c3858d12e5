"""KnowledgeRecommender-compatible TransE / DistMult / RotatE / ComplEx on the fused CUDA path.

Host-side mirror of hopwise's model API (paths under /root/reference/hopwise/):
  model/abstract_recommender.py:36-108, 197-223   AbstractRecommender / KnowledgeRecommender
  model/knowledge_graph_embedding_recommender/transe.py:22-154, distmult.py:22-146,
      rotate.py:24-220, complex.py:22-219          (constructor, calculate_loss, predict,
                                                    full_sort_predict and the _kg twins)
  model/init.py:13-29                              xavier_normal_ on every nn.Embedding
  trainer/trainer.py:165-206, 243-265              optimiser choice and the step loop

Same class names, constructor signature ``(config, dataset)``, attribute names and
``state_dict`` keys as the reference, so the unchanged ``KGTrainer`` drives these models:

  optimizer.zero_grad(); loss = model.calculate_loss(batch); loss.backward(); optimizer.step()

What differs underneath: ``calculate_loss`` launches one kernel that gathers the rows, scores,
accumulates the scalar loss and scatters analytic gradients; ``loss.backward()`` launches the
exact row-lazy Adam on the touched rows (scaled by the incoming grad).  The embedding
parameters never receive a ``.grad``, so the trainer's ``torch.optim.Adam.step()`` is a no-op
by construction.  Rows a step did not touch are caught up lazily (dense Adam keeps moving a row
after its last gradient); ``flush()`` brings every row up to date and runs automatically before
the weights are read (``state_dict``, ``eval``, ``predict*``).

All compute goes through the C ABI in include/kge_b200.h.  There is no CPU fallback: calling a
compute method on CPU tensors raises.
"""

from __future__ import annotations

import ctypes as C
import enum
import math
import os

import torch
from torch import nn

from . import _abi

try:  # use hopwise's own enums when it is importable so Config(model=cls) accepts the classes
    from hopwise.utils import InputType, ModelType  # type: ignore
except Exception:  # pragma: no cover - exercised on boxes without hopwise

    class ModelType(enum.Enum):
        GENERAL = 1
        SEQUENTIAL = 2
        CONTEXT = 3
        KNOWLEDGE = 4
        TRADITIONAL = 5
        DECISIONTREE = 6

    class InputType(enum.Enum):
        POINTWISE = 1
        PAIRWISE = 2
        LISTWISE = 3


TOPK_LIST_MAX = 128                 # largest k of the sorted-list top-k epilogue; larger k take per-row buffers
TOPK_WORKSPACE_BUDGET = 2 << 30     # default workspace bound of a k > TOPK_LIST_MAX full_sort_topk call (bytes)


def _cfg_get(config, key, default=None):
    try:
        if key in config:
            return config[key]
    except TypeError:
        pass
    try:
        v = config[key]
        return default if v is None else v
    except (KeyError, AttributeError):
        return default


class KnowledgeRecommender(nn.Module):
    """Field names and entity counts, as abstract_recommender.py:197-223."""

    type = ModelType.KNOWLEDGE

    def __init__(self, config, dataset):
        super().__init__()
        self.USER_ID = config["USER_ID_FIELD"]
        self.ITEM_ID = config["ITEM_ID_FIELD"]
        self.NEG_ITEM_ID = config["NEG_PREFIX"] + self.ITEM_ID
        self.ENTITY_ID = config["ENTITY_ID_FIELD"]
        self.RELATION_ID = config["RELATION_ID_FIELD"]
        self.HEAD_ENTITY_ID = config["HEAD_ENTITY_ID_FIELD"]
        self.TAIL_ENTITY_ID = config["TAIL_ENTITY_ID_FIELD"]
        self.NEG_TAIL_ENTITY_ID = config["NEG_PREFIX"] + self.TAIL_ENTITY_ID
        self.n_users = dataset.num(self.USER_ID)
        self.n_items = dataset.num(self.ITEM_ID)
        self.n_entities = dataset.num(self.ENTITY_ID)
        self.n_relations = dataset.num(self.RELATION_ID)
        self.device = config["device"]

    # abstract_recommender.py:93-102
    def other_parameter(self):
        if hasattr(self, "other_parameter_name"):
            return {key: getattr(self, key) for key in self.other_parameter_name}
        return dict()

    def load_other_parameter(self, para):
        if para is None:
            return
        for key, value in para.items():
            setattr(self, key, value)

    def __str__(self):
        params = sum(p.numel() for p in self.parameters() if p.requires_grad)
        return super().__str__() + f"\nTrainable parameters: {params}"


# per-step bookkeeping attributes are plain Python values: nn.Module.__setattr__ costs ~5 us per store
_plain_set = object.__setattr__


class _FusedStep(torch.autograd.Function):
    """loss = forward kernel; backward = Adam on the touched rows, scaled by grad_output."""

    @staticmethod
    def forward(ctx, anchor, model, batch):
        ctx.model = model
        return model._launch_forward(batch, with_grad=True, device=anchor.device)

    @staticmethod
    def backward(ctx, grad_out):
        ctx.model._launch_apply(grad_out)
        return None, None, None   # the anchor only exists to give the loss a grad_fn


class _FusedLoss(torch.Tensor):
    """The 0-dim loss `calculate_loss` returns.  It carries the `_FusedStep` grad_fn, so anything built on it
    (`loss + sync_loss`, `scaler.scale(loss)`, `torch.autograd.backward`) runs the fused update through autograd
    as usual; a direct `loss.backward()` -- what the reference trainer calls (trainer/trainer.py:261) -- launches
    the same update without the autograd engine's round trip (~40 us of host time per step, which the trainer's
    per-step `loss.item()` sync otherwise exposes as GPU idle time)."""

    __torch_function__ = torch._C._disabled_torch_function_impl   # ops on the loss give plain tensors, no dispatch cost

    def backward(self, gradient=None, retain_graph=None, create_graph=False, inputs=None):
        model = self.__dict__.get("_kge_model")
        if (model is not None and gradient is None and not create_graph and inputs is None
                and model._pending and model.__dict__.get("_pending_loss") is self):
            model._launch_apply(None)   # d(loss)/d(loss) = 1
            return None
        return super().backward(gradient, retain_graph, create_graph, inputs)


class FusedKGEModel(KnowledgeRecommender):
    """Shared machinery; the four public classes only name their tables."""

    input_type = InputType.PAIRWISE
    KIND: str = ""
    USER_TABLES: tuple = ()
    ENTITY_TABLES: tuple = ()
    RELATION_TABLES: tuple = ()
    HAS_MARGIN = True
    CREATION_ORDER: tuple = ()    # table names in the reference constructor's order when it is not user, entity, relation
    # rotate.py:43 / complex.py:38 look the [UI-Relation] token up; transe/distmult take weight[-1]
    UI_BY_TOKEN = False
    UI_FULLSORT_BY_TOKEN = False
    # extra state the reference checkpoints through other_parameter() (trainer.py:296-304)
    other_parameter_name = ["kge_optimizer_state"]

    def __init__(self, config, dataset):
        super().__init__(config, dataset)
        self.embedding_size = int(config["embedding_size"])
        self.margin = float(config["margin"]) if self.HAS_MARGIN else 0.0
        if self.UI_BY_TOKEN or self.UI_FULLSORT_BY_TOKEN:
            self.ui_relation = int(dataset.field2token_id["relation_id"][dataset.ui_relation])
        # tables in the reference's creation order (fixes the RNG stream of the initialisation)
        d = self.embedding_size
        rows = {**{n: self.n_users for n in self.USER_TABLES}, **{n: self.n_entities for n in self.ENTITY_TABLES},
                **{n: self.n_relations for n in self.RELATION_TABLES}}
        for name in (self.CREATION_ORDER or self.USER_TABLES + self.ENTITY_TABLES + self.RELATION_TABLES):
            setattr(self, name, nn.Embedding(rows[name], d))
        self.apply(_xavier_normal_initialization)
        if self.KIND == "RotatE":
            nn.init.uniform_(self.relation_embedding.weight, 0, 2 * math.pi)  # rotate.py:59

        # optimiser hyper-parameters: the trainer's (trainer.py:165-206); anything the fused
        # update does not reproduce is refused instead of silently diverging
        # (trainer.py:189-205: adam, adamw, sgd, adagrad, rmsprop; an unrecognised name falls back to Adam there too.
        # AdamW with weight_decay 0 IS Adam; sparse_adam needs sparse gradients, which these dense tables never give
        # the reference either)
        learner = str(_cfg_get(config, "learner", "adam")).lower()
        if learner == "sparse_adam":
            raise NotImplementedError("learner 'sparse_adam' needs sparse embedding gradients (nn.Embedding(sparse=True))")
        if learner == "adamw":
            learner = "adam"
        if learner not in _abi.OPTIMIZERS:
            import warnings

            warnings.warn(f"unrecognized learner {learner!r}: Adam, as the reference trainer does (trainer.py:203-205)")
            learner = "adam"
        self.learner = learner
        if float(_cfg_get(config, "weight_decay", 0.0) or 0.0) != 0.0:
            raise NotImplementedError("fused KGE step implements weight_decay 0.0 only")
        if _cfg_get(config, "clip_grad_norm", None):
            raise NotImplementedError("clip_grad_norm is not supported by the fused KGE step")
        if _cfg_get(config, "enable_amp", False) or _cfg_get(config, "enable_scaler", False):
            raise NotImplementedError("AMP / GradScaler are not supported: the kernels are fp32")
        self.learning_rate = float(_cfg_get(config, "learning_rate", 1e-3))
        # torch's defaults for the learner (the trainer passes lr and weight_decay only): Adam betas (0.9, 0.999) eps
        # 1e-8; Adagrad eps 1e-10; RMSprop alpha 0.99 (carried in the beta2 slot) eps 1e-8
        self.betas = (0.9, 0.99) if learner == "rmsprop" else (0.9, 0.999)
        self.adam_eps = 1e-10 if learner == "adagrad" else 1e-8
        self.replay_cap = int(_cfg_get(config, "kge_replay_cap", 200))

        self._step = 0          # optimiser steps applied so far
        self._pending = False   # a gradient was accumulated and not yet applied
        self._dirty = False     # some rows lag behind self._step (lazy Adam)
        self._state = None      # device-side optimiser state, allocated on first training step
        self._anchor = None
        self._grad_sync = None  # optional callable(model) run between forward and apply (multi-GPU)
        self._owner_adam = False  # distributed.py: dense Adam, owner-sharded over the switch (no row-lazy state)
        self._grad_scale = 1.0  # 1 / world_size under data parallelism (DDP averages gradients)
        self._keepalive = None
        self._touch_bounds = (0, 0, 0)
        self._mma_cache = None
        self._mma_ws = {}             # (n, n_targets, k, shape) -> (workspace, row flags, exact-row counter)
        self._mma_counters = []       # device counters of the calls since the last read of the diagnostics
        self._mma_total = 0
        self._ready_key = None
        self._struct_cache = {}

    # ------------------------------------------------------------------ tables
    def _tables(self, names):
        return [getattr(self, n).weight for n in names]

    def _check_ready(self):
        # (the Parameter objects are looked up once: nn.Module.__getattr__ is slow, and this runs every step; code
        # that swaps a Parameter object -- not its .data -- drops the cache through _apply / load_state_dict)
        plist = self.__dict__.get("_table_params")
        if plist is None:
            plist = [t for names in (self.USER_TABLES, self.ENTITY_TABLES, self.RELATION_TABLES)
                     for t in self._tables(names)]
            self.__dict__["_table_params"] = plist
            self.__dict__["_entity0"] = self._tables(self.ENTITY_TABLES)[0]
        w = self.__dict__["_entity0"]
        key = tuple([t.data_ptr() for t in plist])
        if key == self._ready_key:   # same storages as the last (successful) check: nothing can have changed
            return w.device
        if not w.is_cuda:
            raise RuntimeError(
                f"{type(self).__name__}: the fused KGE path runs on CUDA only (weights are on {w.device}); "
                "there is no CPU fallback"
            )
        for names in (self.USER_TABLES, self.ENTITY_TABLES, self.RELATION_TABLES):
            for t in self._tables(names):
                if t.dtype != torch.float32 or not t.is_contiguous():
                    raise RuntimeError("the fused KGE kernels need contiguous float32 tables (weight_precision float32)")
        self._ready_key = key
        self._struct_cache = {}
        return w.device

    def _ui_row(self, full_sort: bool) -> int:
        by_token = self.UI_FULLSORT_BY_TOKEN if full_sort else self.UI_BY_TOKEN
        return self.ui_relation if by_token else self.n_relations - 1

    def _ensure_state(self, device):
        if self._state is not None and self._state["device"] == device:
            return self._state
        old = self._state   # the model moved: the moments move with it (re-zeroing them would keep _step and
        #                     silently restart Adam's bias correction from a wrong state)
        if old is not None and self.__dict__.get("_g_alloc") is not None:
            raise RuntimeError("a data-parallel replica (symmetric gradient buffer) cannot change device")
        st = {"device": device}
        fams = (
            ("user", self.USER_TABLES, self.n_users),
            ("entity", self.ENTITY_TABLES, self.n_entities),
            ("relation", self.RELATION_TABLES, self.n_relations),
        )
        d = self.embedding_size
        # gradient accumulators and row states of all tables live in two flat buffers, so that the dense
        # data-parallel path reduces them with one collective each (hopwise_b200/distributed.py)
        # (a data-parallel exchange may place them in symmetric / multicast memory: distributed.py sets _g_alloc)
        g_numel = sum(rows * len(names) for _, names, rows in fams) * d
        alloc = self.__dict__.get("_g_alloc")
        st["g_flat"] = alloc(g_numel, device) if alloc is not None else torch.zeros(g_numel, device=device)
        st["row_state_flat"] = torch.full((sum(rows for _, _, rows in fams), 2), -1, dtype=torch.int32, device=device)
        # the moments share the gradient buffer's flat layout (an owner-sharded optimiser step walks the three
        # buffers -- and the weights, below -- element for element)
        flat_len = (g_numel + 3) // 4 * 4
        st["m_flat"] = torch.zeros(flat_len, device=device)
        st["v_flat"] = torch.zeros(flat_len, device=device)
        w_alloc = self.__dict__.get("_w_alloc")
        if w_alloc is not None:
            # data-parallel owner-sharded Adam (distributed.py): the weights move into one symmetric buffer with the
            # same layout; every parameter becomes a view of it
            st["w_flat"] = w_alloc(flat_len, device)
            w_off = 0
            with torch.no_grad():
                for _, names, rows in fams:
                    for w in self._tables(names):
                        view = st["w_flat"][w_off : w_off + rows * d].view(rows, d)
                        view.copy_(w)
                        w.data = view
                        w_off += rows * d
            self._ready_key = None
            self._check_ready()
            self.invalidate_target_image()
        g_off = rs_off = 0
        for fam, names, rows in fams:
            g_views, m_views, v_views = [], [], []
            for _ in names:
                g_views.append(st["g_flat"][g_off : g_off + rows * d].view(rows, d))
                m_views.append(st["m_flat"][g_off : g_off + rows * d].view(rows, d))
                v_views.append(st["v_flat"][g_off : g_off + rows * d].view(rows, d))
                g_off += rows * d
            st[fam] = {
                "m": m_views,
                "v": v_views,
                "g": g_views,
                # [rows, 2] int32: {last_step, touch_step}
                "row_state": st["row_state_flat"][rs_off : rs_off + rows],
            }
            st[fam]["g_span"] = (g_off - rows * d * len(names), g_off)
            st[fam]["rs_span"] = (rs_off, rs_off + rows)
            rs_off += rows
        lib = _abi.lib()
        n = lib.kge_adam_table_fill(self.learning_rate, self.betas[0], self.betas[1], None, 0)
        host = (C.c_float * (2 * n))()
        lib.kge_adam_table_fill(self.learning_rate, self.betas[0], self.betas[1], host, n)
        st["adam_table"] = torch.tensor(list(host), dtype=torch.float32).to(device)
        st["adam_table_len"] = n
        st["loss"] = torch.zeros(1, device=device)
        if old is not None:
            st["row_state_flat"].copy_(old["row_state_flat"])
            for fam, _, _ in fams:
                for key in ("m", "v"):
                    for dst, src in zip(st[fam][key], old[fam][key]):
                        dst.copy_(src)
        self._state = st
        self._struct_cache = {}
        return st

    def _model_struct(self, with_state: bool) -> _abi.kge_model_t:
        # the struct only holds pointers and shapes: rebuilt when a table or the optimiser state moves
        with_state = bool(with_state) and self._state is not None
        ckey = (with_state, self._ready_key, id(self._state))
        hit = self._struct_cache.get(with_state)
        if hit is not None and hit[0] == ckey:
            return hit[1]
        m = self._build_model_struct(with_state)
        if self._ready_key is not None:
            self._struct_cache[with_state] = (ckey, m)
        return m

    def _build_model_struct(self, with_state: bool) -> _abi.kge_model_t:
        m = _abi.kge_model_t()
        m.model = _abi.MODEL_KINDS[self.KIND]
        m.d = self.embedding_size
        m.margin = self.margin
        m.ui_relation = self._ui_row(False)
        m.ui_relation_fullsort = self._ui_row(True)
        m.n_items = self.n_items
        st = self._state if with_state else None
        for fam, names, rows in (
            ("user", self.USER_TABLES, self.n_users),
            ("entity", self.ENTITY_TABLES, self.n_entities),
            ("relation", self.RELATION_TABLES, self.n_relations),
        ):
            t = getattr(m, fam)
            t.rows = rows
            t.parts = len(names)
            for p, w in enumerate(self._tables(names)):
                t.w[p] = w.data_ptr()
                if st is not None:
                    t.m[p] = st[fam]["m"][p].data_ptr()
                    t.v[p] = st[fam]["v"][p].data_ptr()
                    t.g[p] = st[fam]["g"][p].data_ptr()
            if st is not None and not self._owner_adam:
                t.row_state = st[fam]["row_state"].data_ptr()   # (owner-sharded dense Adam keeps no row states)
        if st is not None:
            m.adam_table = st["adam_table"].data_ptr()
            m.adam_table_len = st["adam_table_len"]
        return m

    def _adam_struct(self, step: int) -> _abi.kge_adam_t:
        hp = (self.learning_rate, self.betas[0], self.betas[1], self.adam_eps, self.replay_cap)
        a = self.__dict__.get("_adam_cache")
        if a is None or a[0] != hp:   # one struct per hyper-parameter set; only the step changes between calls
            s = _abi.kge_adam_t()
            s.lr, s.beta1, s.beta2, s.eps, s.replay_cap = hp
            s.optimizer = _abi.OPTIMIZERS[self.learner]
            a = (hp, s)
            self.__dict__["_adam_cache"] = a
        a[1].step = step
        return a[1]

    # ------------------------------------------------------------------ training
    @staticmethod
    def _ids(x, device):
        if not isinstance(x, torch.Tensor):
            x = torch.as_tensor(x)
        if x.device != device:
            raise RuntimeError(f"batch ids are on {x.device}, the model is on {device} (call interaction.to(device))")
        if x.dtype is torch.int64 and x.is_contiguous():   # what hopwise's Interaction holds: nothing to convert
            return x
        return x.to(torch.int64).contiguous()

    def _batch_struct(self, interaction, device):
        def get(key):
            try:
                return self._ids(interaction[key], device)
            except KeyError:
                return None

        user, item, neg_item = get(self.USER_ID), get(self.ITEM_ID), get(self.NEG_ITEM_ID)
        head, rel = get(self.HEAD_ENTITY_ID), get(self.RELATION_ID)
        tail, neg_tail = get(self.TAIL_ENTITY_ID), get(self.NEG_TAIL_ENTITY_ID)
        b = _abi.kge_batch_t()
        keep = []
        b.k_rec = b.k_kg = 1
        if user is not None and user.numel():
            if item is None or neg_item is None:
                raise KeyError("recommendation half of the batch needs item and negative-item ids")
            n = user.numel()
            if item.numel() != n or neg_item.numel() % n:
                raise ValueError("user / item / neg_item lengths do not line up")
            b.user, b.item, b.neg_item, b.n_rec = user.data_ptr(), item.data_ptr(), neg_item.data_ptr(), n
            b.k_rec = neg_item.numel() // n
            keep += [user, item, neg_item]
        if head is not None and head.numel():
            if rel is None or tail is None or neg_tail is None:
                raise KeyError("KG half of the batch needs relation, tail and negative-tail ids")
            n = head.numel()
            if rel.numel() != n or tail.numel() != n or neg_tail.numel() % n:
                raise ValueError("head / relation / tail / neg_tail lengths do not line up")
            b.head, b.relation, b.tail, b.neg_tail, b.n_kg = (
                head.data_ptr(), rel.data_ptr(), tail.data_ptr(), neg_tail.data_ptr(), n,
            )
            b.k_kg = neg_tail.numel() // n
            keep += [head, rel, tail, neg_tail]
        return b, keep

    def _launch_forward(self, interaction, with_grad: bool, device=None):
        if device is None:
            device = self._check_ready()
        lib = _abi.lib()
        stream = _abi.stream_ptr()
        lazy = self._state is not None
        if with_grad:
            self._ensure_state(device)
            lazy = True
        if self._pending:  # a loss whose backward never ran: drop its gradient
            self._discard_pending(lib, stream)
        b, keep = self._batch_struct(interaction, device)
        m = self._model_struct(lazy)
        a = self._adam_struct(self._step + 1)
        loss = torch.zeros(1, device=device)
        _abi.check(
            lib.kge_train_forward(C.byref(m), C.byref(b), C.byref(a), 1 if with_grad else 0, loss.data_ptr(), stream),
            "kge_train_forward",
        )
        _plain_set(self, "_keepalive", keep)
        # upper bounds on the distinct rows this batch can touch (sizes the row-sparse exchange)
        _plain_set(self, "_touch_bounds", (
            int(b.n_rec),
            int(b.n_rec) * (1 + int(b.k_rec)) + int(b.n_kg) * (2 + int(b.k_kg)),
            int(b.n_kg) + 1,
        ))
        if with_grad:
            _plain_set(self, "_pending", True)
        return loss.reshape(())

    def _discard_pending(self, lib, stream):
        if self._owner_adam:
            self._state["g_flat"].zero_()
        else:
            m = self._model_struct(True)
            _abi.check(lib.kge_grad_discard(C.byref(m), self._step + 1, stream), "kge_grad_discard")
        _plain_set(self, "_pending", False)

    def _launch_apply(self, grad_out):
        if not self._pending:
            raise RuntimeError("backward called twice for one calculate_loss (the fused step keeps no graph)")
        lib = _abi.lib()
        applied = False
        if self._grad_sync is not None:
            applied = bool(self._grad_sync(self))   # True: the exchange kernel took the optimiser step as well
        if self._owner_adam and not applied:
            raise RuntimeError("owner-sharded Adam is enabled but the exchange did not take the step")
        if applied and grad_out is not None:
            raise RuntimeError("owner-sharded Adam takes loss.backward() directly (no incoming gradient)")
        if not applied:
            # the incoming grad stays on the device: no host sync inside backward (None: the direct
            # loss.backward() of the trainer, whose incoming grad is 1)
            g = grad_out
            if g is not None and (g.dtype != torch.float32 or g.numel() != 1 or g.requires_grad):
                g = g.detach().to(torch.float32).reshape(1).contiguous()
            m = self._model_struct(True)
            a = self._adam_struct(self._step + 1)
            _abi.check(
                lib.kge_adam_apply(C.byref(m), C.byref(a), float(self._grad_scale), _abi.ptr(g), _abi.stream_ptr()),
                "kge_adam_apply",
            )
        _plain_set(self, "_pending_loss", None)
        _plain_set(self, "_step", self._step + 1)
        _plain_set(self, "_pending", False)
        _plain_set(self, "_dirty", not applied)   # (a dense step leaves every row current)
        if applied:
            self.invalidate_target_image()

    def calculate_loss(self, interaction):
        """transe.py:75-98 / distmult.py:68-95 / rotate.py:98-131 / complex.py:95-128."""
        device = self._check_ready()
        if not torch.is_grad_enabled():
            return self._launch_forward(interaction, with_grad=False, device=device)
        if self._anchor is None or self._anchor.device != device:
            self._anchor = torch.zeros(1, device=device, requires_grad=True)
        loss = _FusedStep.apply(self._anchor, self, interaction).as_subclass(_FusedLoss)
        loss._kge_model = self
        _plain_set(self, "_pending_loss", loss)
        return loss

    LOSS_RING = 256

    def train_step(self, interaction):
        """``optimizer.zero_grad(); loss = calculate_loss(batch); loss.backward(); optimizer.step()`` of the
        reference loop (trainer/trainer.py:247-266) as ONE library call: forward and the row-lazy Adam update are
        queued back to back by ``kge_train_step`` with no autograd node in between.  Returns the step's loss, a
        0-dim device tensor with no grad_fn (one slot of a zeroed ring that is replaced, never rewritten, every
        LOSS_RING steps, so a loss a caller keeps stays valid).  With a gradient exchange installed (several GPUs)
        the exchange has to run between the two kernels, and the call takes the two-launch route."""
        if self._grad_sync is not None:
            loss = self.calculate_loss(interaction)
            loss.backward()
            return loss.detach()
        device = self._check_ready()
        self._ensure_state(device)
        lib = _abi.lib()
        stream = _abi.stream_ptr()
        if self._pending:  # a loss whose backward never ran: drop its gradient
            self._discard_pending(lib, stream)
            _plain_set(self, "_pending_loss", None)
        ring = self.__dict__.get("_loss_ring")
        if ring is None or ring[2] == self.LOSS_RING or ring[0].device != device:
            base = torch.zeros(self.LOSS_RING, device=device)
            ring = [base, base.unbind(0), 0, base.data_ptr()]
            self.__dict__["_loss_ring"] = ring
        pos = ring[2]
        ring[2] = pos + 1
        b, keep = self._batch_struct(interaction, device)
        m = self._model_struct(True)
        a = self._adam_struct(self._step + 1)
        _abi.check(
            lib.kge_train_step(C.byref(m), C.byref(b), C.byref(a), float(self._grad_scale), ring[3] + 4 * pos, stream),
            "kge_train_step",
        )
        _plain_set(self, "_keepalive", keep)
        if b.n_rec + b.n_kg:
            _plain_set(self, "_step", self._step + 1)
            _plain_set(self, "_dirty", True)
        return ring[1][pos]

    def flush(self):
        """Bring every row of every table to the current optimiser step (dense pass)."""
        if self._state is None or not self._dirty:
            return
        lib = _abi.lib()
        if self._pending:
            self._discard_pending(lib, _abi.stream_ptr())
        m = self._model_struct(True)
        a = self._adam_struct(self._step)
        _abi.check(lib.kge_adam_flush(C.byref(m), C.byref(a), _abi.stream_ptr()), "kge_adam_flush")
        self._dirty = False

    # ------------------------------------------------------------------ nn.Module hooks
    def train(self, mode: bool = True):
        if not mode:
            self.flush()
        return super().train(mode)

    def state_dict(self, *args, **kwargs):
        self.flush()
        return super().state_dict(*args, **kwargs)

    def load_state_dict(self, state_dict, *args, **kwargs):
        self.flush()  # every row current before the weights are overwritten
        self.__dict__.pop("_table_params", None)
        self.invalidate_target_image()
        return super().load_state_dict(state_dict, *args, **kwargs)

    def _apply(self, fn, *args, **kwargs):
        self.__dict__.pop("_table_params", None)
        # .to(device): optimiser state is rebuilt lazily on the new device (after a flush)
        if self._state is not None:
            self.flush()
        self.invalidate_target_image()
        self._mma_ws = {}
        return super()._apply(fn, *args, **kwargs)

    @property
    def kge_optimizer_state(self):
        """Adam moments for checkpoints (rides in other_parameter(), trainer.py:296-304)."""
        if self._state is None or self._owner_adam:
            return None   # (owner-sharded Adam: every rank holds 1/world of the moments; checkpoints carry weights only)
        self.flush()
        out = {"step": self._step}
        for fam in ("user", "entity", "relation"):
            out[fam] = {
                "m": [t.detach().cpu() for t in self._state[fam]["m"]],
                "v": [t.detach().cpu() for t in self._state[fam]["v"]],
                "row_state": self._state[fam]["row_state"].detach().cpu(),
            }
        return out

    @kge_optimizer_state.setter
    def kge_optimizer_state(self, value):
        if value is None:
            return
        device = self._check_ready()
        st = self._ensure_state(device)
        self._step = int(value["step"])
        for fam in ("user", "entity", "relation"):
            for dst, src in zip(st[fam]["m"], value[fam]["m"]):
                dst.copy_(src)
            for dst, src in zip(st[fam]["v"], value[fam]["v"]):
                dst.copy_(src)
            st[fam]["row_state"].copy_(value[fam]["row_state"])
        self._dirty = False
        self._pending = False

    # ------------------------------------------------------------------ scoring
    def _score_rows(self, heads, rels, tails, head_is_user: bool):
        device = self._check_ready()
        self.flush()
        heads, tails = self._ids(heads, device), self._ids(tails, device)
        rels = None if rels is None else self._ids(rels, device)
        out = torch.empty(heads.numel(), dtype=torch.float32, device=device)
        m = self._model_struct(False)
        _abi.check(
            _abi.lib().kge_predict(
                C.byref(m), heads.data_ptr(), _abi.ptr(rels), tails.data_ptr(), heads.numel(),
                1 if head_is_user else 0, out.data_ptr(), _abi.stream_ptr(),
            ),
            "kge_predict",
        )
        return out

    def _full_sort(self, heads, rels, head_is_user: bool, n_targets: int):
        device = self._check_ready()
        self.flush()
        heads = self._ids(heads, device)
        rels = None if rels is None else self._ids(rels, device)
        out = torch.empty(heads.numel(), n_targets, dtype=torch.float32, device=device)
        m = self._model_struct(False)
        _abi.check(
            _abi.lib().kge_full_sort_scores(
                C.byref(m), heads.data_ptr(), _abi.ptr(rels), heads.numel(), 1 if head_is_user else 0,
                n_targets, out.data_ptr(), _abi.stream_ptr(),
            ),
            "kge_full_sort_scores",
        )
        return out

    def predict(self, interaction):
        return self._score_rows(interaction[self.USER_ID], None, interaction[self.ITEM_ID], True)

    def predict_kg(self, interaction):
        return self._score_rows(
            interaction[self.HEAD_ENTITY_ID], interaction[self.RELATION_ID], interaction[self.TAIL_ENTITY_ID], False
        )

    def full_sort_predict(self, interaction):
        """[n_batch_users, n_items] fp32 the caller owns (trainer.py:731-734 masks it in place)."""
        return self._full_sort(interaction[self.USER_ID], None, True, self.n_items)

    def full_sort_predict_kg(self, interaction):
        return self._full_sort(interaction[self.HEAD_ENTITY_ID], interaction[self.RELATION_ID], False, self.n_entities)

    # ------------------------------------------------------------------ fused full-sort top-k
    def _topk_exact(self, m, users, k, hist_off, hist_items, mask_pad, ids, scores, rels=None, n_targets=None,
                    workspace_budget=TOPK_WORKSPACE_BUDGET):
        lib = _abi.lib()
        n = users.numel()
        n_targets = self.n_items if n_targets is None else n_targets
        head_is_user = 1 if rels is None else 0

        def need(rows):
            b = lib.kge_full_sort_topk_workspace_bytes(C.byref(m), rows, n_targets, k)
            if b < 0:
                raise _abi.KgeError(f"kge_full_sort_topk: unsupported shape (k={k}, d={self.embedding_size})")
            return b

        # k > TOPK_LIST_MAX keeps a buffer of about 2k keys per row and target split in the workspace: the rows go
        # in chunks that keep it under the budget (the result does not depend on the chunking)
        chunk = max(n, 1)
        if k > TOPK_LIST_MAX:
            while chunk > 1 and need(chunk) > workspace_budget:
                chunk = (chunk + 1) // 2
        bounds = [(s, min(n, s + chunk)) for s in range(0, n, chunk)] or [(0, 0)]
        ws = torch.empty(max(max(need(e - s) for s, e in bounds), 8), dtype=torch.uint8, device=users.device)
        for s, e in bounds:
            _abi.check(
                lib.kge_full_sort_topk(
                    C.byref(m), _abi.ptr(users[s:e]), _abi.ptr(None if rels is None else rels[s:e]), e - s,
                    head_is_user, n_targets, _abi.ptr(None if hist_off is None else hist_off[s : e + 1]),
                    _abi.ptr(hist_items), 1 if mask_pad else 0, k, _abi.ptr(ids[s:e]),
                    _abi.ptr(None if scores is None else scores[s:e]), ws.data_ptr(), ws.numel(), _abi.stream_ptr(),
                ),
                "kge_full_sort_topk",
            )

    @staticmethod
    def _mma_shape() -> int:
        """Sweep shape forced through KGE_MMA_CFG = a | f | c | k (tests, experiments); 0 = the library picks."""
        cfg = os.environ.get("KGE_MMA_CFG", "")
        return ord(cfg[0]) if cfg[:1] in ("a", "f", "c", "k") else 0

    def _mma_supported(self, k: int, n_targets=None) -> bool:
        m = self._model_struct(False)
        n_targets = self.n_items if n_targets is None else n_targets
        return _abi.lib().kge_full_sort_topk_mma_workspace_bytes(C.byref(m), 1, n_targets, k, self._mma_shape()) >= 0

    def invalidate_target_image(self):
        """Drop the cached fp16 operand image of the entity table.  Called by everything in this package that
        writes the weights; call it yourself after writing through ``weight.data`` (such writes do not bump the
        tensor version the cache is keyed on)."""
        self._mma_cache = None

    def _mma_image(self, m, device, n_targets=None, shape: int = 0):
        """fp16 operand image of the target rows, cached until the entity table changes."""
        n_targets = self.n_items if n_targets is None else n_targets
        tabs = self._tables(self.ENTITY_TABLES)
        key = (self._step, n_targets, shape, tuple(t.data_ptr() for t in tabs), tuple(t._version for t in tabs))
        if self._mma_cache is not None and self._mma_cache[0] == key:
            return self._mma_cache[1]
        lib = _abi.lib()
        nbytes = lib.kge_mma_image_bytes(C.byref(m), n_targets, shape)
        image = torch.empty(nbytes, dtype=torch.uint8, device=device)
        _abi.check(
            lib.kge_mma_prepare_targets(C.byref(m), n_targets, image.data_ptr(), nbytes, shape, _abi.stream_ptr()),
            "kge_mma_prepare_targets",
        )
        self._mma_cache = (key, image)
        return image

    @property
    def _mma_last_fallback_rows(self) -> int:
        """Rows of the most recent tensor-core call that went through the exact kernel (reads a device counter:
        synchronises; diagnostics and tests only)."""
        return int(self._mma_counters[-1].item()) if self._mma_counters else 0

    def _fold_mma_counters(self):
        old = self._mma_counters[:-1]   # the last one stays readable as _mma_last_fallback_rows
        if old:
            self._mma_total += int(torch.stack(old).sum().item())
            self._mma_counters = self._mma_counters[-1:]

    @property
    def _mma_total_fallback_rows(self) -> int:
        """The same over the model's lifetime."""
        self._fold_mma_counters()
        return self._mma_total + self._mma_last_fallback_rows

    def full_sort_topk_kg(self, head_ids, relation_ids, k: int, hist_off=None, hist_items=None, mask_pad: bool = True,
                          return_scores: bool = True, path: str = "auto", workspace_budget: int = TOPK_WORKSPACE_BUDGET):
        """Link-prediction twin of full_sort_topk: full_sort_predict_kg (transe.py:139-154, distmult.py:135-146,
        rotate.py:192-220, complex.py:192-219) over all entities with a relation per row, the same masking
        (trainer.py:731-734: entity 0 and the known tails in `hist`) and top-k (Collector_KG, collector.py:252-261)."""
        return self.full_sort_topk(head_ids, k, hist_off, hist_items, mask_pad, return_scores, path,
                                   relation_ids=relation_ids, workspace_budget=workspace_budget)

    def full_sort_topk(self, user_ids, k: int, hist_off=None, hist_items=None, mask_pad: bool = True,
                       return_scores: bool = True, path: str = "auto", _debug_scores: bool = False, relation_ids=None,
                       workspace_budget: int = TOPK_WORKSPACE_BUDGET):
        """Fused full_sort_predict + trainer masking + top-k (trainer.py:716-735, collector.py:176-177).

        With ``relation_ids`` the rows are (head entity, relation) queries scored against every entity
        (the link-prediction evaluation); without, users against the items with the user->item relation.

        ``hist_off`` [n+1] / ``hist_items`` (sorted ascending per user) is the CSR of the items to
        mask for each of the ``user_ids``.  Returns (ids [n,k] int64, scores [n,k] fp32 or None),
        ordered by (score desc, id asc).  ``path``: "cuda" = fp32 CUDA-core kernel, "mma" = tcgen05
        filter + exact fp32 re-score (same results), "auto" = "mma" where it is supported and the
        item set is large enough to pay for the operand image.

        Any ``1 <= k <= n_targets`` is taken; the tensor cores serve k <= 32 only.  Above k = 128 the kernel keeps
        a buffer of about 2k keys per row and target split in a workspace, and the rows are processed in chunks
        that keep it under ``workspace_budget`` bytes (the result does not depend on the chunking).
        """
        device = self._check_ready()
        self.flush()
        users = self._ids(user_ids, device)
        n = users.numel()
        rels = None if relation_ids is None else self._ids(relation_ids, device)
        if rels is not None and rels.numel() != n:
            raise ValueError("relation_ids must have one entry per head")
        n_targets = self.n_items if rels is None else self.n_entities
        head_is_user = 1 if rels is None else 0
        if hist_off is not None:
            hist_off, hist_items = self._ids(hist_off, device), self._ids(hist_items, device)
            if hist_off.numel() != n + 1:
                raise ValueError("hist_off must have n_users + 1 entries")
        ids = torch.empty(n, k, dtype=torch.int64, device=device)
        scores = torch.empty(n, k, dtype=torch.float32, device=device) if return_scores else None
        m = self._model_struct(False)
        if path not in ("auto", "mma", "cuda"):
            raise ValueError(path)
        use_mma = path == "mma" or (path == "auto" and n_targets >= 8192 and n >= 64 and self._mma_supported(k, n_targets))
        if not use_mma or n == 0:
            self._topk_exact(m, users, k, hist_off, hist_items, mask_pad, ids, scores, rels, n_targets,
                             workspace_budget)
            return ids, scores
        lib = _abi.lib()
        shape = self._mma_shape()
        # workspace, row flags and the counter are cached per call shape: a fresh ~80 MB allocation per call costs
        # more than the kernels' launch, and nothing in the call needs the host (rows the filter hands back are
        # recomputed by the exact kernel inside the same call, gated by a device counter)
        wkey = (n, n_targets, k, shape, device)
        slot = self._mma_ws.get(wkey)
        if slot is None:
            need = lib.kge_full_sort_topk_mma_workspace_bytes(C.byref(m), n, n_targets, k, shape)
            if need < 0:
                raise _abi.KgeError(f"tensor-core top-k: {lib.kge_last_error().decode()}")
            if len(self._mma_ws) >= 4:
                self._mma_ws.clear()
            slot = (torch.empty(need, dtype=torch.uint8, device=device),
                    torch.empty(n, dtype=torch.int32, device=device))
            self._mma_ws[wkey] = slot
        ws, flags = slot
        counter = torch.empty(1, dtype=torch.int32, device=device)
        image = self._mma_image(m, device, n_targets, shape)
        dbg = None
        if _debug_scores:
            dbg = torch.zeros(n, (n_targets + 127) // 128 * 128, dtype=torch.float32, device=device)
        _abi.check(
            lib.kge_full_sort_topk_mma(
                C.byref(m), users.data_ptr(), _abi.ptr(rels), n, head_is_user, n_targets, image.data_ptr(), _abi.ptr(hist_off),
                _abi.ptr(hist_items), 1 if mask_pad else 0, k, ids.data_ptr(), _abi.ptr(scores), flags.data_ptr(),
                counter.data_ptr(), ws.data_ptr(), ws.numel(), _abi.ptr(dbg), shape, _abi.stream_ptr(),
            ),
            "kge_full_sort_topk_mma",
        )
        self._mma_counters.append(counter)
        if len(self._mma_counters) > 256:   # keeps the list bounded; one sync per 256 calls
            self._fold_mma_counters()
        if _debug_scores:
            return ids, scores, dbg
        return ids, scores

    # ------------------------------------------------------------------ fused full-sort ranks of listed targets
    def full_sort_rank(self, query_ids, pos_off, pos_items, hist_off=None, hist_items=None, mask_pad: bool = True,
                       relation_ids=None):
        """Exact full-catalogue ranks of listed targets, without the score matrix (kge_full_sort_rank_counts).

        The rows and the masking are full_sort_topk's (``relation_ids``: link prediction over all entities).
        ``pos_off`` [n+1] / ``pos_items`` (sorted ascending per row) is the CSR of the targets to rank, e.g. the
        positives.  Returns int64 ``(greater, equal, n_unmasked)``: for every entry of ``pos_items``, how many targets
        of its row's masked scores score strictly above it and exactly equal to it (itself included), and per row
        the number of unmasked targets.  The entry's average rank (collector.py ``_average_rank``) is
        ``greater + (equal + 1) / 2``."""
        device = self._check_ready()
        self.flush()
        users = self._ids(query_ids, device)
        n = users.numel()
        rels = None if relation_ids is None else self._ids(relation_ids, device)
        if rels is not None and rels.numel() != n:
            raise ValueError("relation_ids must have one entry per head")
        n_targets = self.n_items if rels is None else self.n_entities
        if hist_off is not None:
            hist_off, hist_items = self._ids(hist_off, device), self._ids(hist_items, device)
            if hist_off.numel() != n + 1:
                raise ValueError("hist_off must have n_users + 1 entries")
        pos_off, pos_items = self._ids(pos_off, device), self._ids(pos_items, device)
        if pos_off.numel() != n + 1:
            raise ValueError("pos_off must have n_users + 1 entries")
        n_pos = pos_items.numel()
        greater = torch.empty(n_pos, dtype=torch.int64, device=device)
        equal = torch.empty(n_pos, dtype=torch.int64, device=device)
        n_unmasked = torch.empty(n, dtype=torch.int64, device=device)
        m = self._model_struct(False)
        lib = _abi.lib()
        need = lib.kge_full_sort_rank_workspace_bytes(C.byref(m), n, n_targets, n_pos)
        if need < 0:
            raise _abi.KgeError(f"kge_full_sort_rank_counts: unsupported shape (d={self.embedding_size})")
        ws = torch.empty(max(need, 16), dtype=torch.uint8, device=device)
        _abi.check(
            lib.kge_full_sort_rank_counts(
                C.byref(m), users.data_ptr(), _abi.ptr(rels), n, 1 if rels is None else 0, n_targets,
                _abi.ptr(hist_off), _abi.ptr(hist_items), 1 if mask_pad else 0, pos_off.data_ptr(),
                pos_items.data_ptr(), greater.data_ptr(), equal.data_ptr(), n_unmasked.data_ptr(), ws.data_ptr(),
                ws.numel(), _abi.stream_ptr(),
            ),
            "kge_full_sort_rank_counts",
        )
        return greater, equal, n_unmasked

    def full_sort_meanrank(self, query_ids, pos_off, pos_items, hist_off=None, hist_items=None, mask_pad: bool = True,
                           relation_ids=None):
        """float32 [n, 3] rows ``(pos_rank_sum, user_len, pos_len)``: the collector's ``rec.meanrank``
        (collector.py, the ``rec.meanrank`` branch and ``_average_rank``) that GAUC reads, from full_sort_rank.

        Duplicate ids of a row count once, as the reference's ``pos_matrix[u, i] = 1`` does.  The average ranks are
        summed in float64 and rounded once.  ``user_len`` is the reference's ``argmin`` of the sorted row, which is
        the number of unmasked targets only when the row has a masked one: ``mask_pad=True`` (what the trainer
        does) guarantees it, so ``mask_pad=False`` without a history is refused."""
        if not mask_pad and hist_off is None:
            raise ValueError("full_sort_meanrank needs a masked target in every row (mask_pad=True or a history): "
                             "user_len is the argmin of the sorted row")
        greater, equal, n_unmasked = self.full_sort_rank(query_ids, pos_off, pos_items, hist_off, hist_items, mask_pad,
                                                         relation_ids)
        return self._meanrank_rows(greater, equal, n_unmasked, pos_off, pos_items)

    def _meanrank_rows(self, greater, equal, n_unmasked, pos_off, pos_items):
        """rec.meanrank rows from rank counts: a duplicate positive of a row counts once, float64 sums."""
        device = greater.device
        pos_off, pos_items = self._ids(pos_off, device), self._ids(pos_items, device)
        n, n_pos = n_unmasked.numel(), pos_items.numel()
        row = torch.repeat_interleave(torch.arange(n, device=device), pos_off.diff(), output_size=n_pos)
        first = torch.ones(n_pos, dtype=torch.bool, device=device)
        first[1:] = (pos_items[1:] != pos_items[:-1]) | (row[1:] != row[:-1])
        avg_rank = greater.double() + (equal.double() + 1.0) * 0.5
        once = first.double()   # (weights rather than a boolean selection: no host synchronisation)
        rank_sum = torch.zeros(n, dtype=torch.float64, device=device).index_add_(0, row, avg_rank * once)
        pos_len = torch.zeros(n, dtype=torch.float64, device=device).index_add_(0, row, once)
        return torch.stack([rank_sum, n_unmasked.double(), pos_len], dim=1).float()

    # ------------------------------------------------------------------ sampled evaluation over candidate lists
    def _candidate_select(self, user_col, item_col, cand_off, k: int, want_ids=True, want_scores=False,
                          pos_off=None, pos_items=None):
        """predict on the candidate rows, then kge_candidate_select.  Returns (ids, scores, greater, equal,
        n_unmasked), None where not asked for (the rank counts are asked for with the positives CSR)."""
        k = int(k)
        if k < 1:
            raise ValueError(f"k={k} below 1")
        n_cand = len(item_col)
        if len(user_col) != n_cand:
            raise ValueError("user_col and item_col must have one entry per candidate")
        cand_off = torch.as_tensor(cand_off)
        if cand_off.dim() != 1 or cand_off.numel() < 1:
            raise ValueError("cand_off must be a 1-d tensor of n_users + 1 offsets")
        first, last = (int(x) for x in cand_off[[0, -1]].tolist())   # (a host read: a sync when on the device)
        if first != 0 or last != n_cand:
            raise ValueError(f"cand_off must run from 0 to the number of candidates ({n_cand}), got {first}..{last}")
        if k > self.n_items:
            raise ValueError(f"k={k} larger than the number of items ({self.n_items})")
        device = self._check_ready()
        n = cand_off.numel() - 1
        cand_off = self._ids(cand_off.to(device), device)
        users, items = self._ids(user_col, device), self._ids(item_col, device)
        scores = self.predict({self.USER_ID: users, self.ITEM_ID: items})
        ids = torch.empty(n, k, dtype=torch.int64, device=device) if want_ids else None
        top = torch.empty(n, k, dtype=torch.float32, device=device) if want_scores else None
        greater = equal = n_unmasked = None
        if pos_off is not None:
            pos_off, pos_items = self._ids(pos_off, device), self._ids(pos_items, device)
            if pos_off.numel() != n + 1:
                raise ValueError("pos_off must have n_users + 1 entries")
            greater = torch.empty(pos_items.numel(), dtype=torch.int64, device=device)
            equal = torch.empty_like(greater)
            n_unmasked = torch.empty(n, dtype=torch.int64, device=device)
        lib = _abi.lib()
        need = lib.kge_candidate_select_workspace_bytes(n, n_cand)
        ws = torch.empty(max(need, 8), dtype=torch.uint8, device=device)
        _abi.check(
            lib.kge_candidate_select(
                scores.data_ptr(), items.data_ptr(), n_cand, cand_off.data_ptr(), n, self.n_items, _abi.ptr(pos_off),
                _abi.ptr(pos_items), k, _abi.ptr(ids), _abi.ptr(top), _abi.ptr(greater), _abi.ptr(equal),
                _abi.ptr(n_unmasked), ws.data_ptr(), ws.numel(), _abi.stream_ptr(),
            ),
            "kge_candidate_select",
        )
        return ids, top, greater, equal, n_unmasked

    def candidate_topk(self, user_col, item_col, cand_off, k: int, return_scores: bool = True):
        """Sampled evaluation's top-k without the [n_users, n_items] score matrix: ``predict`` on the candidate rows
        (trainer.py ``_neg_sample_batch_eval``), the scatter into -inf rows and ``torch.topk`` (collector.py).

        ``user_col`` / ``item_col`` are the loader's candidate rows (the interaction's user and item columns); row r
        of the result is candidates ``[cand_off[r], cand_off[r+1])``, which may repeat an item (it counts once).
        Returns (ids [n,k] int64, scores [n,k] fp32 or None) by (score desc, id asc) over the row's distinct
        candidates; a row with fewer than k is padded with the smallest non-candidate ids, ascending, score -inf.
        ``cand_off`` must run from 0 to the number of candidates (checked on the host)."""
        ids, scores, *_ = self._candidate_select(user_col, item_col, cand_off, k, True, return_scores)
        return ids, scores

    def candidate_meanrank(self, user_col, item_col, cand_off, pos_off, pos_items):
        """float32 [n, 3] rows ``(pos_rank_sum, user_len, pos_len)`` of the collector's ``rec.meanrank`` over the
        scattered candidate rows (full_sort_meanrank's rows, for the rows candidate_topk sees): every non-candidate
        scores -inf, ``user_len`` is the number of distinct candidates.  ``pos_off`` [n+1] / ``pos_items`` (sorted
        per row) are the positives; a duplicate counts once."""
        _, _, greater, equal, n_unmasked = self._candidate_select(user_col, item_col, cand_off, 1, False, False,
                                                                  pos_off, pos_items)
        return self._meanrank_rows(greater, equal, n_unmasked, pos_off, pos_items)

    def forward(self, *args, **kwargs):  # the reference's forward is the scorer on gathered rows
        raise NotImplementedError("use calculate_loss / predict / full_sort_predict")


def _xavier_normal_initialization(module):
    if isinstance(module, nn.Embedding):  # model/init.py:24-25
        nn.init.xavier_normal_(module.weight.data)


class TransE(FusedKGEModel):
    KIND = "TransE"
    USER_TABLES = ("user_embedding",)
    ENTITY_TABLES = ("entity_embedding",)
    RELATION_TABLES = ("relation_embedding",)


class DistMult(FusedKGEModel):
    KIND = "DistMult"
    USER_TABLES = ("user_embedding",)
    ENTITY_TABLES = ("entity_embedding",)
    RELATION_TABLES = ("relation_embedding",)


class RotatE(FusedKGEModel):
    KIND = "RotatE"
    USER_TABLES = ("user_embedding", "user_embedding_im")
    ENTITY_TABLES = ("entity_embedding", "entity_embedding_im")
    RELATION_TABLES = ("relation_embedding",)
    UI_BY_TOKEN = True
    UI_FULLSORT_BY_TOKEN = True  # rotate.py:136, 163


class ComplEx(FusedKGEModel):
    KIND = "ComplEx"
    USER_TABLES = ("user_re_embedding", "user_im_embedding")
    ENTITY_TABLES = ("entity_re_embedding", "entity_im_embedding")
    RELATION_TABLES = ("relation_re_embedding", "relation_im_embedding")
    HAS_MARGIN = False
    UI_BY_TOKEN = True            # complex.py:103-104, 137-138 (loss / predict)
    UI_FULLSORT_BY_TOKEN = False  # complex.py:168-169 take weight[-1]


class TorusE(FusedKGEModel):
    """toruse.py: TransE's tables and TransE's training objective (TripletMarginLoss on h + r, toruse.py:81-102 -- the
    fused step runs the TransE kernel), scored on the torus: -4 * sum(min(x^2, 1 - x^2)) with
    x = frac(h) + frac(r) - frac(t) (toruse.py:66-76, 131-172).  The scorer is not a contraction, so full-sort
    evaluation takes the CUDA-core kernels."""

    KIND = "TorusE"
    USER_TABLES = ("user_embedding",)
    ENTITY_TABLES = ("entity_embedding",)
    RELATION_TABLES = ("relation_embedding",)


class _ProjectedKGEModel(FusedKGEModel):
    """TransE on rows projected per relation (TransH, TransD).  Scoring composes two library calls: the subclass's
    ``_project(family, ids)`` writes rows projected with the user->item relation, and since the projection of an
    item does not depend on the user, the rest IS TransE on projected tables -- a private TransE view of those
    buffers runs predict, dense full-sort, the fused top-k (tensor-core path included) and the rank counts.  The
    projected items are cached per weight version.  Users are scored against items only: the dense and fused KG
    full-sort entry points refuse, with the subclass's ``KG_REFUSAL`` as the reason."""

    KG_REFUSAL: str = ""

    def _transe_view(self, users, entities):
        """The private TransE model over projected tables: `users` [n, d] rows, `entities` [m, d] rows, the
        relation table shared with this model."""
        view = self.__dict__.get("_view")
        if view is None:
            cfg = {"USER_ID_FIELD": self.USER_ID, "ITEM_ID_FIELD": self.ITEM_ID,
                   "NEG_PREFIX": self.NEG_ITEM_ID[: -len(self.ITEM_ID)],
                   "ENTITY_ID_FIELD": self.ENTITY_ID, "RELATION_ID_FIELD": self.RELATION_ID,
                   "HEAD_ENTITY_ID_FIELD": self.HEAD_ENTITY_ID, "TAIL_ENTITY_ID_FIELD": self.TAIL_ENTITY_ID,
                   "device": self.device, "embedding_size": self.embedding_size, "margin": self.margin}

            class _Shape:
                def num(_, field):
                    return {self.RELATION_ID: self.n_relations}.get(field, 1)

            view = TransE(cfg, _Shape())
            view.eval()
            self.__dict__["_view"] = view   # (not a submodule: its tables are scratch, not parameters of this model)
        with torch.no_grad():
            view.user_embedding.weight.data = users
            view.entity_embedding.weight.data = entities
            view.relation_embedding.weight.data = self.relation_embedding.weight.data
        view.n_users, view.n_items, view.n_entities = users.shape[0], entities.shape[0], entities.shape[0]
        view.__dict__.pop("_table_params", None)
        return view

    def _projected_items(self):
        """Rows [0, n_items) of the entity table projected with the user->item relation, cached per weight version."""
        tabs = self._tables(self.ENTITY_TABLES + self.RELATION_TABLES[1:])
        key = (self._step, tuple(t.data_ptr() for t in tabs), tuple(t._version for t in tabs))
        hit = self.__dict__.get("_items_cache")
        if hit is None or hit[0] != key:
            ids = torch.arange(self.n_items, device=tabs[0].device)
            hit = (key, self._project("entity", ids))
            self.__dict__["_items_cache"] = hit
            view = self.__dict__.get("_view")
            if view is not None:
                view.invalidate_target_image()
        return hit[1]

    def invalidate_target_image(self):
        super().invalidate_target_image()
        self.__dict__.pop("_items_cache", None)

    def _rec_view(self, user_ids):
        view = self._transe_view(self._project("user", user_ids), self._projected_items())
        return view, torch.arange(view.n_users, device=view.user_embedding.weight.device)

    def predict(self, interaction):
        users, items = interaction[self.USER_ID], interaction[self.ITEM_ID]
        view = self._transe_view(self._project("user", users), self._project("entity", items))
        view.invalidate_target_image()
        idx = torch.arange(view.n_users, device=view.user_embedding.weight.device)
        return view.predict({self.USER_ID: idx, self.ITEM_ID: idx})

    def full_sort_predict(self, interaction):
        view, idx = self._rec_view(interaction[self.USER_ID])
        return view.full_sort_predict({self.USER_ID: idx})

    def full_sort_predict_kg(self, interaction):
        raise NotImplementedError(self.KG_REFUSAL)

    def full_sort_topk(self, user_ids, k, hist_off=None, hist_items=None, mask_pad=True, return_scores=True,
                       path="auto", _debug_scores=False, relation_ids=None, workspace_budget=TOPK_WORKSPACE_BUDGET):
        if relation_ids is not None:
            raise NotImplementedError(self.KG_REFUSAL)
        view, idx = self._rec_view(user_ids)
        return view.full_sort_topk(idx, k, hist_off, hist_items, mask_pad, return_scores, path, _debug_scores,
                                   workspace_budget=workspace_budget)

    def full_sort_rank(self, query_ids, pos_off, pos_items, hist_off=None, hist_items=None, mask_pad=True,
                       relation_ids=None):
        if relation_ids is not None:
            raise NotImplementedError(self.KG_REFUSAL)
        view, idx = self._rec_view(query_ids)
        return view.full_sort_rank(idx, pos_off, pos_items, hist_off, hist_items, mask_pad)


class TransH(_ProjectedKGEModel):
    """transh.py: TransE on rows projected per relation.  The second relation table `norm_vec` holds the hyperplane
    vector w; the reference's ``project`` is ``ent - (ent * w.sum()) * w`` (transh.py:73-74), applied to head and both
    tails before TransE's TripletMarginLoss (transh.py:76-107) and norm (transh.py:53-58).  Recommendation triples
    read ``relation_embedding.weight[-1]`` but ``norm_vec(ui_relation)`` (transh.py:63, 90): the kernels take one row
    for both, so a dataset whose [UI-Relation] token is not the last relation id is refused (hopwise's datasets append
    the token last).  The reference scores users against items only; so does this class (``kge_transh_project``
    writes the projected rows)."""

    KIND = "TransH"
    USER_TABLES = ("user_embedding",)
    ENTITY_TABLES = ("entity_embedding",)
    RELATION_TABLES = ("relation_embedding", "norm_vec")
    KG_REFUSAL = "the reference TransH has no KG scoring entry points (transh.py)"

    def __init__(self, config, dataset):
        super().__init__(config, dataset)
        token_row = int(dataset.field2token_id["relation_id"][dataset.ui_relation])
        if token_row != self.n_relations - 1:
            raise NotImplementedError(
                f"TransH: [UI-Relation] is relation {token_row}, not the last row {self.n_relations - 1}; "
                "relation_embedding.weight[-1] and norm_vec(ui_relation) would name different rows (transh.py:63, 90)")

    def predict_kg(self, interaction):
        raise NotImplementedError(self.KG_REFUSAL)

    def _project(self, family, ids):
        device = self._check_ready()
        self.flush()
        emb = (self.user_embedding if family == "user" else self.entity_embedding).weight
        ids = self._ids(ids, device)
        out = torch.empty(ids.numel(), self.embedding_size, dtype=torch.float32, device=device)
        _abi.check(
            _abi.lib().kge_transh_project(emb.data_ptr(), ids.data_ptr(), ids.numel(), self.embedding_size,
                                          self.norm_vec.weight.data_ptr(), None, self.n_relations - 1, out.data_ptr(),
                                          _abi.stream_ptr()),
            "kge_transh_project",
        )
        return out


class TransD(_ProjectedKGEModel):
    """transd.py: every table has an embedding and a transfer vector; ``forward(ent, ent_vec, rel_vec) = rel_vec *
    <ent, ent_vec> + ent`` (transd.py:86-91) projects head and both tails before TransE's TripletMarginLoss
    (transd.py:93-133).  The train step is one fused kernel like the others (KGE_TRANSD); ``kge_transd_project``
    writes the projected rows for scoring.  ``full_sort_predict_kg`` is refused: the reference's version projects the
    head with <h, h> and broadcasts a relation per row over all tails (transd.py:192-217), which no projected table
    expresses."""

    KIND = "TransD"
    USER_TABLES = ("user_embedding", "user_vec_embedding")
    ENTITY_TABLES = ("entity_embedding", "entity_vec_embedding")
    RELATION_TABLES = ("relation_embedding", "relation_vec_embedding")
    CREATION_ORDER = ("user_embedding", "entity_embedding", "relation_embedding", "user_vec_embedding",
                      "entity_vec_embedding", "relation_vec_embedding")   # transd.py:41-47
    KG_REFUSAL = ("TransD scores users against items only: the reference's full_sort_predict_kg projects the head "
                  "with <h, h> and a relation per row over all tails (transd.py:192-217); not built")

    def _project(self, family, ids, rel_ids=None):
        """[len(ids), d] projected rows of `family` ("user" / "entity"); rel_ids None = the user->item relation."""
        device = self._check_ready()
        self.flush()
        emb, vec = self._tables(self.USER_TABLES if family == "user" else self.ENTITY_TABLES)
        rvec = self.relation_vec_embedding.weight
        ids = self._ids(ids, device)
        n = ids.numel()
        rel_ids = None if rel_ids is None else self._ids(rel_ids, device)
        out = torch.empty(n, self.embedding_size, dtype=torch.float32, device=device)
        _abi.check(
            _abi.lib().kge_transd_project(emb.data_ptr(), vec.data_ptr(), _abi.ptr(ids), n, self.embedding_size,
                                          rvec.data_ptr(), _abi.ptr(rel_ids), self.n_relations - 1, out.data_ptr(),
                                          _abi.stream_ptr()),
            "kge_transd_project",
        )
        return out

    def predict_kg(self, interaction):
        heads, rels, tails = (interaction[k] for k in (self.HEAD_ENTITY_ID, self.RELATION_ID, self.TAIL_ENTITY_ID))
        both = torch.cat([self._project("entity", heads, rels), self._project("entity", tails, rels)])
        n = both.shape[0] // 2
        view = self._transe_view(both[:1], both)
        view.invalidate_target_image()
        idx = torch.arange(n, device=both.device)
        return view.predict_kg({self.HEAD_ENTITY_ID: idx, self.RELATION_ID: self._ids(rels, both.device),
                                self.TAIL_ENTITY_ID: idx + n})


MODELS = {"TransE": TransE, "DistMult": DistMult, "RotatE": RotatE, "ComplEx": ComplEx, "TorusE": TorusE,
          "TransH": TransH, "TransD": TransD}
