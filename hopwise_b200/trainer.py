"""FusedKGTrainer: hopwise's own KGTrainer, minus the costs the unchanged trainer would put back.

The fused models (recommender.py) already run under the unmodified ``KGTrainer`` -- ``optimizer.zero_grad();
loss = model.calculate_loss(batch); loss.backward(); optimizer.step()`` works because the embedding parameters
never receive a ``.grad``.  Three things in the reference trainer nevertheless undo what the fused path removes
(paths under /root/reference/hopwise/):

  trainer/trainer.py:82-84     ``AbstractTrainer.__init__`` wraps the model in DistributedDataParallel whenever
                               ``single_spec`` is false, and ``sync_grad_loss`` (:104-112) then touches every parameter
                               (``torch.sum(params) * 0``) every step: a dense pass over every table plus DDP's dense
                               all-reduce -- exactly the traffic the row-sparse exchange (distributed.py) replaces.
  trainer/trainer.py:716-735   ``_full_sort_batch_eval`` materialises ``[users, n_items]`` scores per batch, and
  evaluator/collector.py:176-183  ``Collector.eval_batch_collect`` adds a second ``[users, n_items]`` int matrix and a
                               ``torch.topk``; the loader (general_dataloader.py:231-267) feeds them 2 users at a time
                               at the default ``eval_batch_size``.
  trainer/trainer.py:243-265   the step loop synchronises on ``loss.item()`` every step and copies the batch with a
                               blocking ``interaction.to(device)``.

``FusedKGTrainer(KGTrainer)`` keeps every public method and attribute of the reference class (``fit``, ``evaluate``,
checkpoints, early stopping, logging are inherited unchanged) and overrides only:

  * ``__init__``            no DDP wrap; under ``torch.distributed`` it broadcasts rank 0's weights and installs the
                            row-sparse gradient exchange instead;
  * ``set_reduce_hook`` / ``sync_grad_loss``   no-ops (there are no dense gradients to reduce);
  * ``_train_epoch``        the same loop with the batch copy one step ahead on a side stream and the epoch's loss
                            summed on the device in float64 (the reference adds the same fp32 values in Python
                            doubles: identical result, one host sync per epoch instead of one per step);
  * ``evaluate_data_loop``  fused full-sort top-k over large user blocks straight from the loader's own per-user
                            history / positives (built once per loader), the ``rec.topk`` rows -- and for GAUC the
                            ``rec.meanrank`` rows, from the exact full-catalogue ranks of the positives -- handed to
                            the reference ``Evaluator`` unchanged, so the metric dictionary is the reference's own.
                            Sampled ranking evaluation of the REC task (``eval_args.mode`` uniN / popN,
                            ``NegSampleEvalDataLoader``) iterates the loader once, as the reference does, and
                            selects over each user's candidate list (evaluator.collect_sampled) instead of
                            scattering the scores into [batch_users, n_items] rows.  Anything the fused kernels do
                            not cover (sampled link-prediction loaders, sequential loaders, the labelled value
                            metrics that read ``rec.score`` / ``data.label``) goes through the inherited dense path.
                            Any cutoff is covered: above k = 128 the fused top-k keeps per-row buffers in a
                            workspace instead of sorted lists in shared memory.

``install()`` registers the classes with hopwise's own factories, so ``run_hopwise(model="TransE", ...)`` and the
``hopwise train`` CLI pick them up without edits: ``get_model`` (utils/utils.py:65-98) resolves
``hopwise.model.knowledge_graph_embedding_recommender.<name>.<Name>`` and ``get_trainer`` (:101-129) first tries
``hopwise.trainer.<Name>Trainer``.

hopwise must be importable (this module is the plug-in side of the boundary; it raises ImportError otherwise).
"""

from __future__ import annotations

import importlib
import math

import numpy as np
import torch

try:
    from hopwise.data.dataloader import FullSortLPEvalDataLoader, FullSortRecEvalDataLoader, NegSampleEvalDataLoader
    from hopwise.data.dataloader.abstract_dataloader import NegSampleDataLoader
    from hopwise.data.dataloader.knowledge_dataloader import KGDataLoaderState
    from hopwise.trainer import KGTrainer
    from hopwise.trainer import trainer as _ref_trainer
    from hopwise.utils import EvaluatorType, KnowledgeEvaluationType
except ImportError as exc:  # pragma: no cover
    raise ImportError("hopwise_b200.trainer plugs into hopwise's trainer: hopwise must be importable") from exc

from . import recommender as _rec
from .evaluator import collect_sampled, topk_hits
from .loader import DevicePrefetcher

# hopwise's Config compares `model_class.type` / `.input_type` with ITS enums (configurator.py:219-224).  When
# hopwise_b200.recommender was imported before hopwise was importable it carries look-alike enums of its own:
# rebind the two class attributes to hopwise's members.
from hopwise.utils import InputType as _InputType, ModelType as _ModelType  # noqa: E402

_rec.KnowledgeRecommender.type = _ModelType.KNOWLEDGE
_rec.FusedKGEModel.input_type = _InputType.PAIRWISE

DEFAULT_USER_BLOCK = 148 * 512   # users per fused call: one full wave of the tensor-core sweep


class _NoWrap:
    """Stands in for DistributedDataParallel during ``AbstractTrainer.__init__`` (trainer.py:82-84)."""

    def __init__(self, module, *args, **kwargs):
        self.module = module

    def __call__(self, x):
        return x


class FusedKGTrainer(KGTrainer):
    def __init__(self, config, model):
        if not isinstance(model, _rec.FusedKGEModel):
            raise TypeError(f"FusedKGTrainer drives hopwise_b200 models, got {type(model).__name__}")
        distributed = not config["single_spec"]
        if distributed:
            # the constructor's DDP wrap is unconditional; the fused model has no dense gradient for it to reduce
            orig = _ref_trainer.DistributedDataParallel
            _ref_trainer.DistributedDataParallel = _NoWrap
            try:
                super().__init__(config, model)
            finally:
                _ref_trainer.DistributedDataParallel = orig
            from .distributed import broadcast_weights, enable_row_sparse_data_parallel

            broadcast_weights(model)      # what DDP's constructor does: every replica starts from rank 0's weights
            self.exchange = enable_row_sparse_data_parallel(model, multimem=bool(_cfg(config, "kge_multimem", False)))
        else:
            super().__init__(config, model)
            self.exchange = None
        self.user_block = int(_cfg(config, "kge_eval_user_block", DEFAULT_USER_BLOCK))
        self.fused_eval = bool(_cfg(config, "kge_fused_eval", True))
        self.prefetch = bool(_cfg(config, "kge_prefetch", True))

    # ---- the DDP plumbing of the reference loop (trainer.py:94-112): nothing to do -----------------------------
    def set_reduce_hook(self):
        return None

    def sync_grad_loss(self):
        return 0

    # ---- training -----------------------------------------------------------------------------------------------
    def _train_epoch(self, train_data, epoch_idx, loss_func=None, show_progress=False):
        # KGTrainer._train_epoch (trainer.py:647-666): which half of the data this epoch trains on
        if self.train_rec_step is None or self.train_kg_step is None:
            state = KGDataLoaderState.RSKG
        elif epoch_idx % (self.train_rec_step + self.train_kg_step) < self.train_rec_step:
            state = KGDataLoaderState.RS
        else:
            state = KGDataLoaderState.KG
        if state == KGDataLoaderState.KG or loss_func is not None or show_progress:
            # calculate_kg_loss / a caller's loss / the progress bar: the reference loop, unchanged
            return super()._train_epoch(train_data, epoch_idx, loss_func=loss_func, show_progress=show_progress)
        if not self.config["single_spec"]:
            train_data.knowledge_shuffle(epoch_idx)
        train_data.set_mode(state)
        if not self.config["single_spec"] and train_data.shuffle:
            train_data.sampler.set_epoch(epoch_idx)

        # Trainer._train_epoch (trainer.py:208-268) for one scalar loss, Adam fused into backward
        model = self.model
        model.train()
        device = torch.device(self.device)
        batches = DevicePrefetcher(train_data, device) if (self.prefetch and device.type == "cuda") else None
        losses = []
        for interaction in (batches if batches is not None else train_data):
            if batches is None:
                interaction = interaction.to(device)
            # forward + the fused row-lazy Adam step in one library call (optimizer.step() has nothing to do); the
            # loss stays on the device
            losses.append(model.train_step(interaction))
        # float64 sum of the float32 step losses: the reference's `total_loss + losses.item()`; the epoch's only
        # host synchronisation
        total_loss = float(torch.stack(losses).double().sum().item()) if losses else 0.0
        if math.isnan(total_loss):
            raise ValueError("Training loss is nan")   # trainer.py:337-339 (checked per epoch instead of per step)
        return total_loss

    # ---- evaluation -----------------------------------------------------------------------------------------------
    def _fused_plan(self, eval_data, task):
        """Device-resident evaluation inputs of one loader, in the order this rank's sampler visits the sources:
        ids, CSR of the masked targets (history) and of the positives, both sorted per row.  None when the fused
        kernels do not cover the request."""
        if not self.fused_eval or isinstance(eval_data, NegSampleDataLoader) or getattr(eval_data, "is_sequential", False):
            return None
        if not isinstance(eval_data, (FullSortRecEvalDataLoader, FullSortLPEvalDataLoader)):
            return None
        collector = self.eval_collector if task == KnowledgeEvaluationType.REC else self.eval_collector_kg
        reg = collector.register
        if any(reg.need(key) for key in ("rec.score", "data.label")):
            return None   # the labelled value metrics need the dense score rows
        if torch.device(self.device).type != "cuda":
            return None
        plan = eval_data.__dict__.get("_kge_fused_plan")
        if plan is not None and plan["task"] == task and plan["device"] == str(self.device):
            return plan
        src = eval_data._source_list.numpy()
        idx = np.fromiter(iter(eval_data.sampler), dtype=np.int64)   # positions, in this rank's order (padded under DDP)
        ids = src[idx]

        def csr(per_source):
            parts = [per_source[s].numpy() for s in ids]
            lens = np.fromiter((len(p) for p in parts), dtype=np.int64, count=len(parts))
            vals = np.concatenate(parts) if parts else np.zeros(0, dtype=np.int64)
            rows = np.repeat(np.arange(len(parts)), lens)
            vals = vals[np.lexsort((vals, rows))]               # ascending inside every row
            off = np.zeros(len(parts) + 1, dtype=np.int64)
            np.cumsum(lens, out=off[1:])
            return torch.from_numpy(off).to(self.device), torch.from_numpy(vals).to(self.device)

        plan = {"task": task, "device": str(self.device), "n": len(ids),
                "ids": torch.from_numpy(ids).to(self.device),
                "hist": csr(eval_data._sample2history), "pos": csr(eval_data._sample2positives),
                "n_batches": (len(ids) + eval_data.step - 1) // eval_data.step, "rels": None}
        if task == KnowledgeEvaluationType.LP:
            rel = eval_data._source_df[eval_data.relation_field].numpy()[idx]
            plan["rels"] = torch.from_numpy(rel).to(self.device)
        eval_data.__dict__["_kge_fused_plan"] = plan
        return plan

    def _fused_sampled(self, eval_data, task) -> bool:
        """Whether a sampled (uniN / popN) evaluation goes through the candidate-list selection."""
        if not self.fused_eval or task != KnowledgeEvaluationType.REC:
            return False
        if not isinstance(eval_data, NegSampleEvalDataLoader) or getattr(eval_data, "is_sequential", False):
            return False
        if self.config["eval_type"] != EvaluatorType.RANKING or torch.device(self.device).type != "cuda":
            return False
        reg = self.eval_collector.register
        return not any(reg.need(key) for key in ("rec.score", "data.label"))

    def _sampled_eval_loop(self, eval_data):
        collector, reg, struct = self.eval_collector, self.eval_collector.register, self.eval_collector.data_struct
        # trainer.py _neg_sample_batch_eval + collector.py eval_batch_collect over all batches: one pass of the
        # loader (it draws the negatives from the shared random stream), one selection call per user block
        data, n_batches = collect_sampled(self.model, eval_data, max(collector.topk),
                                          meanrank=bool(reg.need("rec.meanrank")), user_block=max(1, self.user_block))
        for key in ("rec.users", "rec.items", "rec.topk", "rec.meanrank"):
            if reg.need(key):
                struct.update_tensor(key, data[key])
        collector.model_collect(self.model)
        result = self.evaluator.evaluate(collector.get_data_struct())
        if not self.config["single_spec"]:
            result = self._map_reduce(result, 4 * n_batches)   # as the full-sort branch below
        self.wandblogger.log_eval_metrics(result, head="eval")
        return result

    def evaluate_data_loop(self, eval_data, task, tot_target_num, target_tensor, show_progress=True):
        if self._fused_sampled(eval_data, task):
            return self._sampled_eval_loop(eval_data)
        plan = self._fused_plan(eval_data, task)
        if plan is None:
            return super().evaluate_data_loop(eval_data, task, tot_target_num, target_tensor,
                                              show_progress=show_progress)
        rec_task = task == KnowledgeEvaluationType.REC
        collector = self.eval_collector if rec_task else self.eval_collector_kg
        evaluator = self.evaluator if rec_task else self.evaluator_kg
        reg, struct = collector.register, collector.data_struct
        kmax = max(collector.topk)
        (hoff, hval), (poff, pval) = plan["hist"], plan["pos"]
        n, block = plan["n"], max(1, self.user_block)
        for s in range(0, n, block):
            e = min(n, s + block)
            users = plan["ids"][s:e]
            h0, h1 = int(hoff[s].item()), int(hoff[e].item())
            p0, p1 = int(poff[s].item()), int(poff[e].item())
            ho, po = hoff[s : e + 1] - h0, poff[s : e + 1] - p0
            rels = None if plan["rels"] is None else plan["rels"][s:e]
            # trainer.py:731-734 (column 0 and the history -> -inf) + collector.py:176-183, without the score matrix
            ids, _ = self.model.full_sort_topk(users, kmax, ho, hval[h0:h1], mask_pad=True, return_scores=False,
                                               relation_ids=rels)
            if reg.need("rec.users"):
                struct.update_tensor("rec.users", users)
            if reg.need("rec.items"):
                struct.update_tensor("rec.items", ids)
            if reg.need("rec.topk"):
                struct.update_tensor("rec.topk", topk_hits(ids, po, pval[p0:p1]))
            if reg.need("rec.meanrank"):
                # collector.py's rec.meanrank branch without sorting the [users, n_items] score rows
                struct.update_tensor("rec.meanrank", self.model.full_sort_meanrank(
                    users, po, pval[p0:p1], ho, hval[h0:h1], mask_pad=True, relation_ids=rels))
        collector.model_collect(self.model)
        result = evaluator.evaluate(collector.get_data_struct())
        if not self.config["single_spec"]:
            # the reference weights each rank by `len(batched_data)` summed over its batches -- the length of the
            # 4-tuple, i.e. 4 x batches (trainer.py:847-849): reproduced, so the reduced numbers are the reference's
            result = self._map_reduce(result, 4 * plan["n_batches"])
        self.wandblogger.log_eval_metrics(result, head="eval")
        return result


def _cfg(config, key, default):
    try:
        value = config[key]
    except (KeyError, TypeError):
        return default
    return default if value is None else value


# ---- registration with hopwise's factories -----------------------------------------------------------------------
_KGE_PACKAGE = "hopwise.model.knowledge_graph_embedding_recommender"
_installed: dict = {}


def install(models=("TransE", "DistMult", "RotatE", "ComplEx", "TorusE", "TransH", "TransD")):
    """Make hopwise resolve these model names to the fused classes and FusedKGTrainer.

    ``get_model(name)`` imports ``hopwise.model.knowledge_graph_embedding_recommender.<name>`` and takes the
    attribute ``<Name>`` (utils/utils.py:87-98): that attribute is rebound.  ``get_trainer`` looks for
    ``hopwise.trainer.<Name>Trainer`` before falling back to ``KGTrainer`` (utils/utils.py:117-129): that hook is
    set.  ``uninstall()`` restores both."""
    trainer_pkg = importlib.import_module("hopwise.trainer")
    for name in models:
        cls = _rec.MODELS[name]
        module = importlib.import_module(f"{_KGE_PACKAGE}.{name.lower()}")
        if name not in _installed:
            _installed[name] = (module, getattr(module, name))
        setattr(module, name, cls)
        setattr(trainer_pkg, name + "Trainer", FusedKGTrainer)
    return FusedKGTrainer


def uninstall():
    trainer_pkg = importlib.import_module("hopwise.trainer")
    for name, (module, original) in list(_installed.items()):
        setattr(module, name, original)
        if getattr(trainer_pkg, name + "Trainer", None) is FusedKGTrainer:
            delattr(trainer_pkg, name + "Trainer")
        del _installed[name]
