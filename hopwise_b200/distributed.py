"""Data parallelism for the fused KGE path: row-sparse gradient exchange and user-block sharding.

What it replaces (paths under /root/reference/hopwise/):
  trainer/trainer.py:82-112    DistributedDataParallel wrap + set_reduce_hook / sync_grad_loss:
                               a dense all-reduce (mean) of every embedding table each step
  trainer/trainer.py:592-609   _map_reduce: all_gather of per-rank metric means
  data/dataloader/abstract_dataloader.py:59-64   per-rank DistributedSampler shards

One process per GPU (torch.distributed, NCCL over NVLink).  Tables and Adam state are
replicated.  Per step every rank packs the rows its batch touched (ids + gradient rows) into one
flat buffer, a single all-gather moves the buffers, and every rank adds all lists -- its own
included -- into its (zeroed) gradient accumulators in rank order, then applies Adam with the
gradient scaled by 1/world_size (DDP's mean).  The adds see the same values in the same
order on every rank, so the replicas stay bit-identical without ever moving a dense table.
Bytes per rank per step: sum over tables of min(rows, touched) * (8 + parts*d*4), instead of
4 bytes * every parameter.

With ``multimem=True`` the dense route reduces in the NVSwitch instead of through NCCL: the gradient
accumulators are allocated as a symmetric buffer with an NVLS multicast mapping (torch's symmetric-memory
rendezvous is the plumbing: allocation, handle exchange, cross-rank barrier) and
``kge_multimem_all_reduce_f32`` sums the N copies in place (csrc/collective.cu).

A table whose batch can touch at least half of its rows (small tables, or the roofline batches of
bench.py) takes the dense route instead: its gradient accumulator is all-reduced (sum) and every one
of its rows is marked as touched (a row nobody touched then takes the zero-gradient Adam step dense
Adam gives it); the accumulators live in one flat buffer so that one collective covers every dense
table.  NCCL delivers the same sums to every rank, so the
replicas stay bit-identical on this route too.
"""

from __future__ import annotations

import ctypes as C

import torch
import torch.distributed as dist

from . import _abi

FAMILIES = ("user", "entity", "relation")


def shard_bounds(n: int, rank: int, world: int):
    """Contiguous block [lo, hi) of `n` units for `rank`; sizes differ by at most one."""
    base, rem = divmod(n, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)


class FlatLayout:
    """Byte layout of one rank's packed gradient message: per table
    [count int32 (padded to 16 B) | ids int64[cap] | rows fp32[cap, parts*d], 16-byte aligned]."""

    def __init__(self, caps, parts, d):
        self.caps, self.parts, self.d = list(caps), list(parts), int(d)
        self.offsets = []
        off = 0
        for cap, p in zip(self.caps, self.parts):
            cnt = off
            ids = cnt + 16
            rows = (ids + 8 * cap + 15) // 16 * 16   # rows are read and written as float4
            off = rows + 4 * cap * p * self.d
            off = (off + 15) // 16 * 16
            self.offsets.append((cnt, ids, rows))
        self.nbytes = off

    def views(self, buf: torch.Tensor, which: int):
        """(count int32[1], ids int64[cap], rows fp32[cap, parts*d]) views into a uint8 buffer."""
        cnt, ids, rows = self.offsets[which]
        cap, p = self.caps[which], self.parts[which]
        return (
            buf[cnt : cnt + 4].view(torch.int32),
            buf[ids : ids + 8 * cap].view(torch.int64),
            buf[rows : rows + 4 * cap * p * self.d].view(torch.float32).view(cap, p * self.d),
        )


def _cuda_pack(model, which, step, count, ids, rows):
    m = model._model_struct(True)
    _abi.check(
        _abi.lib().kge_grad_pack(C.byref(m), which, step, ids.data_ptr(), rows.data_ptr(), count.data_ptr(),
                                 _abi.stream_ptr()),
        "kge_grad_pack",
    )


def _cuda_add(model, which, step, count, ids, rows):
    m = model._model_struct(True)
    _abi.check(
        _abi.lib().kge_grad_add(C.byref(m), which, step, ids.data_ptr(), rows.data_ptr(), count.data_ptr(),
                                ids.numel(), _abi.stream_ptr()),
        "kge_grad_add",
    )


class RowSparseExchange:
    """Callable installed as ``model._grad_sync``; runs between the forward/gradient kernel and
    the Adam kernel of every step."""

    def __init__(self, model, group=None, pack_fn=_cuda_pack, add_fn=_cuda_add, device=None, multimem=False,
                 owner_adam=False):
        self.group = group
        self.symm = None           # symmetric-memory handle of the gradient buffer (multimem route)
        self.multimem = False
        self.owner_adam = False    # the optimiser step itself runs owner-sharded over the switch (kge_owner_adam_step)
        if multimem or owner_adam:
            self._install_multimem(model, owner_adam)
        self.world = dist.get_world_size(group)
        self.rank = dist.get_rank(group)
        self.pack_fn, self.add_fn = pack_fn, add_fn
        rows = (model.n_users, model.n_entities, model.n_relations)
        parts = (len(model.USER_TABLES), len(model.ENTITY_TABLES), len(model.RELATION_TABLES))
        # a step cannot touch more distinct rows than the table has
        self.layout = FlatLayout(rows, parts, model.embedding_size)
        self._agreed = None        # per-table bounds on touched rows that every rank plans with
        self.device = device
        self.send = self.recv = None
        self.dense = [False, False, False]
        self.bytes_per_step = 0
        self.kernels_per_step = 0   # launches of this library's pack / add kernels in the last step
        self.fused_barriers = True  # multimem route: barriers and touch marks inside the reduction kernel
        self._local_flags, self._epoch = None, 0
        self.timing = False        # record CUDA events around pack / collective / add (bench.py)
        self.timings = []          # [(pack_ms, collective_ms, add_ms)] of the timed steps, read by take_timings()
        self._events = []

    def _install_multimem(self, model, owner_adam=False):
        """Have the model allocate its flat gradient buffer in symmetric memory with a multicast mapping.
        Must run before the first training step (the optimiser state is created lazily there); every rank
        reaches that allocation together, which makes the rendezvous inside it a proper collective.
        With `owner_adam` the weights move into a second such buffer and the model keeps no row-lazy state."""
        import torch.distributed._symmetric_memory as symm_mem

        if model._state is not None:
            raise RuntimeError("multimem exchange must be enabled before the first training step")
        if owner_adam and getattr(model, "learner", "adam") not in ("adam", "adamw"):
            raise NotImplementedError("owner-sharded optimiser step implements Adam and AdamW only")
        group = self.group if self.group is not None else dist.group.WORLD
        ex = self

        def symmetric(numel, device):
            padded = (numel + 3) // 4 * 4
            buf = symm_mem.empty(padded, dtype=torch.float32, device=device)
            buf.zero_()
            hdl = symm_mem.rendezvous(buf, group)
            if not hdl.has_multicast_support or not hdl.multicast_ptr:
                raise RuntimeError("no NVLS multicast mapping for the buffer")
            return buf, hdl, int(hdl.multicast_ptr) + (buf.data_ptr() - int(hdl.buffer_ptrs[hdl.rank]))

        def alloc(numel, device):
            try:
                buf, hdl, mc = symmetric(numel, device)
            except Exception as exc:   # same hardware on every rank: all ranks take this branch together
                if owner_adam:
                    raise RuntimeError(f"owner-sharded Adam needs NVLS multicast memory ({exc})") from exc
                import warnings

                warnings.warn(f"multimem exchange unavailable ({exc}); the dense route uses NCCL's all-reduce")
                ex.multimem = False
                return torch.zeros(numel, device=device)
            ex.symm = hdl
            ex._mc_base = mc
            ex._symm_keep = buf
            return buf[:numel]

        def alloc_weights(numel, device):
            buf, hdl, mc = symmetric(numel, device)
            ex._w_symm, ex._w_mc_base, ex._w_keep = hdl, mc, buf
            return buf

        object.__setattr__(model, "_g_alloc", alloc)
        self.multimem = True
        if owner_adam:
            object.__setattr__(model, "_w_alloc", alloc_weights)
            object.__setattr__(model, "_owner_adam", True)
            self.owner_adam = True

    SIGNAL_SLOT_BASE = 1024   # uint32 slots of the symmetric signal pad this library uses (torch's barrier channels
    #                           live at the front of the 9216-byte pad)

    def _all_reduce_dense(self, g_flat, g0, g1, row_state=None, step=0):
        """Sum the [g0, g1) float range of the flat gradient buffer over the ranks, in place.  Returns True when the
        touch marks of `row_state` (the rows of the reduced tables) were set on the way."""
        if self.multimem and self.symm is not None and g0 % 4 == 0 and (g1 - g0) % 4 == 0:
            if self.fused_barriers:
                # one kernel: barrier (all gradients written) -> in-switch reduce + broadcast -> touch marks ->
                # barrier (all slices final); csrc/collective.cu
                if self._local_flags is None:
                    self._local_flags = torch.zeros(2, dtype=torch.int32, device=g_flat.device)
                self._epoch = self._epoch % 0x7FFFFFFF + 1
                n_mark = 0 if row_state is None else row_state.shape[0]
                _abi.check(
                    _abi.lib().kge_multimem_all_reduce_fused_f32(
                        self._mc_base + 4 * g0, g1 - g0, self.rank, self.world, int(self.symm.signal_pad_ptrs_dev),
                        self.SIGNAL_SLOT_BASE, self._local_flags.data_ptr(), self._epoch,
                        None if row_state is None else row_state.data_ptr(), n_mark, int(step), _abi.stream_ptr()),
                    "kge_multimem_all_reduce_fused_f32",
                )
                self.kernels_per_step += 1
                return row_state is not None
            self.symm.barrier(channel=0)      # every rank's forward kernel has written its gradients
            _abi.check(
                _abi.lib().kge_multimem_all_reduce_f32(self._mc_base + 4 * g0, g1 - g0, self.rank, self.world,
                                                       _abi.stream_ptr()),
                "kge_multimem_all_reduce_f32",
            )
            self.symm.barrier(channel=1)      # every slice has been reduced and broadcast
            self.kernels_per_step += 1
        else:
            dist.all_reduce(g_flat[g0:g1], op=dist.ReduceOp.SUM, group=self.group)
        return False

    def _agree(self, batch_rows):
        """Bounds on the rows a step can touch, identical on every rank.

        The message layout, the all-gather size and the dense / sparse route per table all derive from these
        bounds, so ranks that planned with their LOCAL batch shapes would disagree as soon as the shapes differ (a
        short last batch on one rank, an empty KG half): mismatched all-gather sizes, or an all-reduce on some
        ranks against an all-gather on others -- an NCCL hang.  The first step agrees on the element-wise maximum
        (every rank takes its first step together, so the collective is safe there); later steps only check that
        the local shape still fits.  A job whose batches can grow passes `max_batch_rows` to
        enable_row_sparse_data_parallel instead."""
        if self._agreed is None:
            t = torch.tensor(list(batch_rows), dtype=torch.int64, device=self.device or "cpu")
            dist.all_reduce(t, op=dist.ReduceOp.MAX, group=self.group)
            self._agreed = tuple(int(x) for x in t.tolist())
        if any(b > a for b, a in zip(batch_rows, self._agreed)):
            raise RuntimeError(
                f"a batch can touch {tuple(batch_rows)} rows (user, entity, relation) but the ranks agreed on "
                f"{self._agreed} at the first step; pass max_batch_rows= to enable_row_sparse_data_parallel")
        return self._agreed

    def reset_bounds(self, max_batch_rows=None):
        """Forget the agreed bounds (a new batch size, another model): the next step agrees again -- every rank must
        call this at the same point -- or plans with `max_batch_rows` when given."""
        self._agreed = None if max_batch_rows is None else tuple(int(x) for x in max_batch_rows)

    def _plan(self, model, batch_rows):
        """Tighten the per-table capacity to what a batch can touch (agreed across ranks); pick the route per table."""
        rows = (model.n_users, model.n_entities, model.n_relations)
        parts = self.layout.parts
        if self.device is None:
            self.device = next(model.parameters()).device
        batch_rows = self._agree(batch_rows)
        caps = [max(1, min(r, b)) for r, b in zip(rows, batch_rows)]
        self.dense = [2 * c >= r for c, r in zip(caps, rows)]
        caps = [1 if dn else c for c, dn in zip(caps, self.dense)]   # dense tables send nothing through the lists
        if self.send is None or caps != self.layout.caps:
            self.layout = FlatLayout(caps, parts, model.embedding_size)
            device = self.device or next(model.parameters()).device
            self.send = torch.zeros(self.layout.nbytes, dtype=torch.uint8, device=device)
            self.recv = torch.zeros(self.world * self.layout.nbytes, dtype=torch.uint8, device=device)
        st = model._state
        dense_bytes = sum((st[f]["g_span"][1] - st[f]["g_span"][0]) * 4 for f, dn in zip(FAMILIES, self.dense) if dn)
        self.bytes_per_step = (0 if all(self.dense) else self.layout.nbytes) + dense_bytes

    def _dense_spans(self, model):
        """Maximal runs of adjacent dense tables in the flat buffers: [(g_lo, g_hi, rs_lo, rs_hi)]."""
        st, runs = model._state, []
        for fam, dn in zip(FAMILIES, self.dense):
            if not dn:
                continue
            (g0, g1), (r0, r1) = st[fam]["g_span"], st[fam]["rs_span"]
            if runs and runs[-1][1] == g0 and runs[-1][3] == r0:
                runs[-1] = (runs[-1][0], g1, runs[-1][2], r1)
            else:
                runs.append((g0, g1, r0, r1))
        return runs

    def _mark(self):
        if self.timing:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            self._events.append(e)

    def take_timings(self):
        """[(pack_ms, collective_ms, add_ms)] of the steps since the last call (needs .timing = True; synchronises)."""
        torch.cuda.synchronize()
        out = [(ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2]), ev[2].elapsed_time(ev[3]))
               for ev in (self._events[i : i + 4] for i in range(0, len(self._events) - 3, 4))]
        self._events = []
        return out

    def _owner_step(self, model):
        """Gradient reduction + Adam + weight broadcast in one kernel; every table takes it (dense Adam)."""
        st = model._state
        if self._local_flags is None:
            self._local_flags = torch.zeros(2, dtype=torch.int32, device=st["g_flat"].device)
            self.dense = [True, True, True]
            self.bytes_per_step = 2 * 4 * st["w_flat"].numel() // self.world   # 1/N gradient in, 1/N weights out
        self._epoch = self._epoch % 0x7FFFFFFF + 1
        a = model._adam_struct(model._step + 1)
        _abi.check(
            _abi.lib().kge_owner_adam_step(
                self._mc_base, self._symm_keep.data_ptr(), self._w_mc_base, st["w_flat"].data_ptr(), st["m_flat"].data_ptr(),
                st["v_flat"].data_ptr(), st["w_flat"].numel(), self.rank, self.world, C.byref(a),
                float(model._grad_scale), int(self.symm.signal_pad_ptrs_dev), self.SIGNAL_SLOT_BASE,
                self._local_flags.data_ptr(), self._epoch, _abi.stream_ptr()),
            "kge_owner_adam_step",
        )
        self.kernels_per_step = 1
        return True

    def __call__(self, model):
        if self.owner_adam:
            return self._owner_step(model)
        step = model._step + 1
        self._plan(model, model._touch_bounds)
        sparse = [w for w in range(3) if not self.dense[w]]
        self.kernels_per_step = len(sparse) * (1 + self.world)
        self._mark()
        for which in sparse:
            count, ids, rows = self.layout.views(self.send, which)
            self.pack_fn(model, which, step, count, ids, rows)
        self._mark()
        st = model._state
        for g0, g1, r0, r1 in self._dense_spans(model):
            # Every row of a dense table is marked as touched instead of all-reducing the touch marks: a row
            # nobody touched holds a zero gradient, and a zero-gradient Adam step is exactly what dense Adam (and
            # the lazy replay) does to it -- same weights, one collective less per step.
            if not self._all_reduce_dense(st["g_flat"], g0, g1, st["row_state_flat"][r0:r1], step):
                st["row_state_flat"][r0:r1, 1].fill_(step)
        if not sparse:
            self._mark()
            self._mark()
            return
        dist.all_gather_into_tensor(self.recv, self.send, group=self.group)
        self._mark()
        n = self.layout.nbytes
        for r in range(self.world):  # fixed order on every rank => identical fp32 sums
            chunk = self.recv[r * n : (r + 1) * n]
            for which in sparse:
                count, ids, rows = self.layout.views(chunk, which)
                self.add_fn(model, which, step, count, ids, rows)
        self._mark()


def multicast_available(device, group=None) -> bool:
    """True when every rank can map a symmetric buffer with an NVLS multicast address (collective call)."""
    ok = 1
    try:
        import torch.distributed._symmetric_memory as symm_mem

        buf = symm_mem.empty(1024, dtype=torch.float32, device=device)
        hdl = symm_mem.rendezvous(buf, group if group is not None else dist.group.WORLD)
        ok = int(bool(hdl.has_multicast_support and hdl.multicast_ptr))
    except Exception:
        ok = 0
    flag = torch.tensor([ok], dtype=torch.int32, device=device)
    dist.all_reduce(flag, op=dist.ReduceOp.MIN, group=group)
    return bool(flag.item())


def enable_row_sparse_data_parallel(model, group=None, multimem=False, max_batch_rows=None, owner_adam=False):
    """Turn a FusedKGEModel replica into a data-parallel one (call once, after model.to(device),
    on every rank, with identical initial weights: the reference gets that from DDP's rank-0
    broadcast, here `broadcast_weights` does it).  ``multimem=True``: dense tables are reduced in the
    NVSwitch (NVLS multicast) by this library's own kernel instead of NCCL; needs a multicast-capable
    fabric and must be enabled before the first training step.

    Every rank must plan with the same bounds on the rows a step can touch (message layout, collective sizes and the
    dense / sparse choice derive from them): they are agreed with one MAX all-reduce at the first step, or given as
    ``max_batch_rows`` when later batches can be larger than the first.

    ``owner_adam=True`` (implies multimem; for jobs whose batches touch most rows of every table, like the roofline
    batches): the whole optimiser step moves into the exchange -- each rank reduces 1/world of the gradient in the
    switch, applies dense Adam to it with its shard of the moments and multicasts the new weights
    (``kge_owner_adam_step``): one kernel instead of all-reduce + Adam, 1/world of the optimiser work per rank.  The
    weights then live in a symmetric buffer (the parameters become views of it), there is no row-lazy state, and
    checkpoints carry weights only.  ``owner_adam="auto"`` takes that route when the fabric offers multicast memory
    (probed collectively) and the plain exchange otherwise."""
    if owner_adam == "auto":
        owner_adam = multicast_available(next(model.parameters()).device, group)
    ex = RowSparseExchange(model, group=group, multimem=multimem, owner_adam=owner_adam)
    if max_batch_rows is not None:   # (user rows, entity rows, relation rows) a step can touch, same on all ranks
        ex._agreed = tuple(int(x) for x in max_batch_rows)
    model._grad_sync = ex
    model._grad_scale = 1.0 / ex.world
    return ex


def broadcast_weights(model, src: int = 0, group=None):
    for p in model.parameters():
        dist.broadcast(p.data, src=src, group=group)
    if hasattr(model, "invalidate_target_image"):
        model.invalidate_target_image()   # writes through .data do not bump the version the image cache is keyed on


def reduce_metric_sums(sums: torch.Tensor, n_users: int, group=None):
    """Exact global metric means from per-rank sums (the reference all-gathers rounded per-rank
    means weighted by a batch count, trainer.py:592-609; this is the unrounded global mean)."""
    buf = torch.cat([sums.reshape(-1).to(torch.float64), torch.tensor([float(n_users)], dtype=torch.float64,
                                                                       device=sums.device)])
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return buf[:-1].reshape(sums.shape), int(round(buf[-1].item()))


def reduce_gauc_sums(sums: torch.Tensor, group=None) -> torch.Tensor:
    """Global GAUC sums (evaluator.gauc_sums of this rank's users) with one all-reduce: every rank then holds
    (sum of auc_u * pos_len, sum of pos_len) over all users, and GAUC = sums[0] / sums[1] exactly as on one GPU."""
    buf = sums.reshape(-1).to(torch.float64).clone()
    dist.all_reduce(buf, op=dist.ReduceOp.SUM, group=group)
    return buf
