#!/usr/bin/env python
"""Benchmark of the KGE hot path: KG triples/s of the fused train step (headline) plus users/s of
the fused full-sort top-k, on synthetic KGs of BASELINE.json's shapes.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

One JSON line on stdout (rank 0).  `value` = positive (rec + KG) triples per second over all
ranks with the id tensors resident in HBM; `e2e` = the same step driven the way hopwise's trainer
drives it, from pinned HOST id buffers: H2D of the 7 id arrays -> calculate_loss -> backward ->
loss.item() (D2H) every step.  `roofline` follows SURVEY.md 8(d): algorithmic bytes per positive
triple = 24*d*T*(2+K) + 8*(3+K), over the measured HBM peak.  `--impl reference` times the
reference's own algorithm on the host cores (the torch-CPU oracle port: the same torch operators
the reference's Python calls, dense autograd + dense torch.optim.Adam).

`--dump-outputs DIR` writes what the headline train step hands its caller after the last timed step -- the loss and
the updated tables -- as DIR/<name>.npy (float32), so that two builds can be compared output for output on the same
seeded inputs.
"""

from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

# the benchmark leaves the tree it runs from as it found it (that tree may be read-only): no bytecode caches
sys.dont_write_bytecode = True

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

# ---- workloads (SURVEY.md 8(d)) ---------------------------------------------------------------
WORKLOADS = {
    # BASELINE.json configs[1]: TransE L2, synthetic ML-1M-small-shaped KG, d=100, 1 negative
    "cfg2_transe_ml1m": dict(model="TransE", U=6041, I=3001, E=30001, R=22, d=100, k=1,
                             n_rec=262144, n_kg=262144, triples=1_000_000, inters=1_000_000),
    # the reference's default batch on the same KG (latency-bound: ~30 MB per step)
    "cfg2_transe_ml1m_b2048": dict(model="TransE", U=6041, I=3001, E=30001, R=22, d=100, k=1,
                                   n_rec=2048, n_kg=2048, triples=1_000_000, inters=1_000_000),
    # BASELINE.json configs[4] shape on one GPU: tables far larger than L2 (no-duplicate regime)
    "cfg5_transe_alibaba": dict(model="TransE", U=115001, I=30001, E=1000001, R=54, d=128, k=1,
                                n_rec=262144, n_kg=262144, triples=50_000_000, inters=5_000_000),
    # the same shape at the reference's batch: the row-sparse exchange regime (4k rows of a 1M-row table per step)
    "cfg5_transe_alibaba_b2048": dict(model="TransE", U=115001, I=30001, E=1000001, R=54, d=128, k=1,
                                      n_rec=2048, n_kg=2048, triples=50_000_000, inters=5_000_000),
    # BASELINE.json configs[2]: RotatE d=256, 64 negatives per triple
    "cfg3_rotate_yelp": dict(model="RotatE", U=45920, I=45539, E=90001, R=44, d=256, k=64,
                             n_rec=2048, n_kg=2048, triples=1_800_000, inters=1_200_000),
}
FULLSORT = {
    # BASELINE.json configs[3]: DistMult / ComplEx full-sort, 1M users x 200k items, top-20
    "cfg4_distmult": dict(model="DistMult", U=1_000_001, I=200_001, E=200_001, R=3, d=64, k=20, hist=50),
    "cfg4_complex": dict(model="ComplEx", U=1_000_001, I=200_001, E=200_001, R=3, d=64, k=20, hist=50),
}
PARTS = {"TransE": 1, "DistMult": 1, "RotatE": 2, "ComplEx": 2}


def bytes_per_triple(model, d, k):
    return 24 * d * PARTS[model] * (2 + k) + 8 * (3 + k)


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=float(p["hbm_gbs"]), bf16_tflops=float(p["bf16_tflops"]), source="measured")
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, source="fallback")


def profiled_traffic(workload):
    """DRAM bytes (read + write) of the two launches of one step, from the committed `ncu --set full` capture of
    this workload (profiles/r1_traffic.json, written by scripts/traffic_from_profiles.py); None when not captured."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(path):
        t = json.load(open(path)).get(workload)
        if t:
            return t["per_step_bytes"], t["source"]
    return None, None


def synth_batches(w, n_batches, seed):
    """Positive triples drawn from a fixed synthetic KG + uniform negatives (ids only)."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n_batches):
        out.append({
            "user_id": rng.integers(1, w["U"], w["n_rec"]),
            "item_id": rng.integers(1, w["I"], w["n_rec"]),
            "neg_item_id": rng.integers(1, w["I"], w["n_rec"] * w["k"]),
            "head_id": rng.integers(1, w["E"], w["n_kg"]),
            "relation_id": rng.integers(1, w["R"] - 1, w["n_kg"]),
            "tail_id": rng.integers(1, w["E"], w["n_kg"]),
            "neg_tail_id": rng.integers(1, w["E"], w["n_kg"] * w["k"]),
        })
    return out


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the timed region runs."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i",
                 str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *exc):
        if self.proc is not None:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap")
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                mx = max(mx, float(r[1]))
                for n, v in zip(names, r[2:6]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except (ValueError, IndexError):
                continue
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx or None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_model(w, device, seed=2024):
    from kge_helpers import make_product_model

    return make_product_model(w["model"], w["U"], w["I"], w["E"], w["R"], w["d"], device=device, seed=seed)


def dist_info():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def max_over_ranks(x, device, world):
    if world == 1:
        return x
    import torch.distributed as dist

    t = torch.tensor([x], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist

        dist.barrier()
    torch.cuda.synchronize()


class no_gc:
    """Timed regions run with the cyclic collector off (collected right before): a generation-2 pass between two kernel
    launches of a block is tens of milliseconds of idle GPU inside that block's events."""

    def __enter__(self):
        import gc

        gc.collect()
        self._was = gc.isenabled()
        gc.disable()

    def __exit__(self, *exc):
        import gc

        if self._was:
            gc.enable()
        return False


# ---- timed legs -------------------------------------------------------------------------------
def time_train_device(model, dev_batches, steps, warmup, flush_buf, world):
    """K steps with ids resident in HBM; per-step CUDA events, L2 flushed (untimed) in between."""
    nb = len(dev_batches)
    warmup = max(warmup, nb)   # every batch buffer is touched once before the timed region
    for i in range(warmup):
        model.calculate_loss(dev_batches[i % nb]).backward()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    with no_gc():
        barrier(world)
        for i in range(steps):
            if flush_buf is not None:
                flush_buf.zero_()
            b = dev_batches[(warmup + i) % nb]
            ev[i][0].record()
            loss = model.calculate_loss(b)
            ev[i][1].record()
            loss.backward()
            ev[i][2].record()
        barrier(world)
    fwd = np.array([e[0].elapsed_time(e[1]) for e in ev])
    upd = np.array([e[1].elapsed_time(e[2]) for e in ev])
    return fwd, upd, float(loss.item())   # per-step milliseconds (forward / backward = exchange + Adam)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, state, loss):
    """The loss of the last timed step and the tables it left (`state`: the model's state_dict(), which first brings
    every lazily updated row to the current step, as it does for any caller), as float32 .npy files of at most
    DUMP_BYTES in all.  Smaller tables are written whole; what does not fit shares the rest of the budget equally, as
    a sorted sample of rows drawn with a fixed seed, so every run and every build writes the same rows."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), np.array([loss], dtype=np.float32))
    tables = sorted(state.items(), key=lambda kv: kv[1].numel())
    budget = DUMP_BYTES - 4096   # (the loss file and the .npy headers)
    for i, (name, t) in enumerate(tables):
        row_bytes = 4 * t[0].numel()
        keep = min(t.shape[0], budget // (len(tables) - i) // row_bytes)
        budget -= keep * row_bytes
        if keep < t.shape[0]:
            rows = np.sort(np.random.default_rng(0).choice(t.shape[0], keep, replace=False))
            t = t[torch.from_numpy(rows).to(t.device)]
        np.save(os.path.join(out_dir, f"{name}.npy"), t.float().cpu().numpy())


def time_train_e2e(model, host_batches, steps, warmup, world, device, reference_order=False):
    """The training loop from pinned host ids through the public API: H2D of the step's 7 id vectors, the step, a
    device->host read of every step's loss.  The copies run one batch ahead on a side stream
    (hopwise_b200.loader.DevicePrefetcher); every step's copy and every loss read are inside the timed region.

    Two orders.  `reference_order`: loss = calculate_loss(); loss.item(); loss.backward() -- the reference trainer's
    body (trainer.py:257-263), whose mid-step sync leaves the GPU idle while the host turns around.  Default: the
    step is issued as one call (model.train_step) and the loss of step i is read while step i+1 runs -- every step's
    loss still crosses to the host inside the timed region, one step late (FusedKGTrainer itself reads the losses
    once per epoch)."""
    from hopwise_b200.loader import DevicePrefetcher, pack_batch

    # the loader's side: one pinned buffer per batch, ids as int32 (row indices; the copy stream widens them on the
    # device) -- half the bytes of the int64 vectors over PCIe, which is what bounds this loop
    host_batches = [pack_batch(b, narrow=True) for b in host_batches]
    nb = len(host_batches)
    stream = torch.cuda.current_stream()

    pending = []

    def one(db):
        if reference_order:
            loss = model.calculate_loss(db)
            val = loss.item()   # trainer.py:259 -- the per-step device->host sync of the reference loop
            loss.backward()
            return val
        # the step's loss goes to pinned host memory with an asynchronous copy right behind the step; the host reads
        # it after the copy's event, once the NEXT step has been issued (loss.item() would wait for the whole stream,
        # the step just issued included)
        loss = model.train_step(db)
        slot = len(pending) % 2 if not pending else (pending[-1][0] + 1) % 2
        host_loss[slot].copy_(loss.detach().reshape(1), non_blocking=True)
        ev = read_events[slot]
        ev.record()
        pending.append((slot, ev))
        if len(pending) > 1:
            s0, e0_ = pending.pop(0)
            e0_.synchronize()
            return float(host_loss[s0])   # the previous step's loss
        return None

    host_loss = [torch.zeros(1).pin_memory() for _ in range(2)]
    read_events = [torch.cuda.Event() for _ in range(2)]

    def drain():
        while pending:
            s0, e0_ = pending.pop(0)
            e0_.synchronize()
            float(host_loss[s0])

    warmup = max(warmup, nb)   # every pinned batch has been through one H2D copy before the timed region (the
    #                            first copy out of a pinned buffer costs ~1 ms extra)
    loader = DevicePrefetcher([host_batches[i % nb] for i in range(warmup)], device)
    for db in loader:
        one(db)
    drain()
    loader.batches = [host_batches[(warmup + i) % nb] for i in range(steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with no_gc():
        barrier(world)
        stamps = [time.perf_counter()]
        e0.record(stream)
        for db in loader:
            one(db)
            stamps.append(time.perf_counter())   # (each step ends with a host sync on a loss)
        drain()                                  # the last step's loss, still inside the timed region
        e1.record(stream)
        barrier(world)
    per_step = np.diff(np.array(stamps)) * 1e3
    return e0.elapsed_time(e1), float(np.median(per_step)), float(per_step.max())


def time_fullsort(fs, device, n_users_step, steps, warmup, world, rank, path="auto"):
    """users/s of fused full-sort + mask + top-k on a block of users per step."""
    from kge_helpers import make_product_model

    m = make_product_model(fs["model"], fs["U"], fs["I"], fs["E"], fs["R"], fs["d"], device=device)
    rng = np.random.default_rng(2024 + rank)
    blocks = []
    for _ in range(min(4, steps + warmup)):
        users = torch.from_numpy(rng.integers(1, fs["U"], n_users_step)).to(device)
        hist = np.sort(rng.integers(1, fs["I"], (n_users_step, fs["hist"])), axis=1)
        off = torch.arange(0, fs["hist"] * n_users_step + 1, fs["hist"], dtype=torch.long, device=device)
        blocks.append((users, off, torch.from_numpy(hist.reshape(-1)).to(device)))
    for i in range(max(warmup, len(blocks))):   # every block once before the timed region (first-touch effects)
        u, o, h = blocks[i % len(blocks)]
        m.full_sort_topk(u, fs["k"], o, h, return_scores=False, path=path)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    with no_gc():
        barrier(world)
        ev[0].record()
        for i in range(steps):
            u, o, h = blocks[i % len(blocks)]
            ids, _ = m.full_sort_topk(u, fs["k"], o, h, return_scores=False, path=path)
            ev[i + 1].record()
        barrier(world)
    ms = ev[0].elapsed_time(ev[-1])
    in_order = [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]
    per_rep = sorted(in_order)
    fallback = m._mma_total_fallback_rows if path != "cuda" else 0   # over warm-up and timed blocks
    del m
    torch.cuda.empty_cache()   # (outside the timed region)
    return ms, fallback, per_rep[len(per_rep) // 2], in_order


def full_eval_leg(fs, device, world, rank):
    """cfg4 end to end: every one of the 1,000,000 users once.  Users are sharded in contiguous blocks over the ranks
    (hopwise_b200.distributed.shard_bounds); each rank runs fused full-sort top-20 + hit flags + metric sums over its
    shard (hopwise_b200.evaluator.evaluate_full_sort in blocks of one sweep wave) and the per-rank sums are reduced
    (reduce_metric_sums) -- all inside the timed region; the result dictionary is the Evaluator's."""
    from hopwise_b200.distributed import reduce_metric_sums, shard_bounds
    from hopwise_b200.evaluator import metrics_from_sums, topk_hits, topk_metric_sums
    from kge_helpers import make_product_model

    m = make_product_model(fs["model"], fs["U"], fs["I"], fs["E"], fs["R"], fs["d"], device=device)
    n_total = fs["U"] - 1
    lo, hi = shard_bounds(n_total, rank, world)
    n = hi - lo
    rng = np.random.default_rng(77 + rank)
    users = torch.arange(1 + lo, 1 + hi, dtype=torch.long, device=device)
    hist = torch.from_numpy(np.sort(rng.integers(1, fs["I"], (n, fs["hist"])), axis=1).reshape(-1)).to(device)
    hoff = torch.arange(0, fs["hist"] * n + 1, fs["hist"], dtype=torch.long, device=device)
    npos = 3
    pos = torch.from_numpy(np.sort(rng.integers(1, fs["I"], (n, npos)), axis=1).reshape(-1)).to(device)
    poff = torch.arange(0, npos * n + 1, npos, dtype=torch.long, device=device)
    block = 148 * 512

    def run():
        sums = torch.zeros(5, fs["k"], dtype=torch.float64, device=device)
        for s0 in range(0, n, block):
            e0 = min(n, s0 + block)
            ids, _ = m.full_sort_topk(users[s0:e0], fs["k"], hoff[s0 : e0 + 1] - s0 * fs["hist"],
                                      hist[s0 * fs["hist"] : e0 * fs["hist"]], return_scores=False)
            rec = topk_hits(ids, poff[s0 : e0 + 1] - s0 * npos, pos[s0 * npos : e0 * npos])
            sums += topk_metric_sums(rec)
        if world > 1:
            sums, total = reduce_metric_sums(sums, n)
        else:
            total = n
        return metrics_from_sums(sums, total, [fs["k"]], decimals=None)

    run()   # warm-up: operand image, workspaces, first touches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    with no_gc():
        barrier(world)
        e0.record()
        result = run()   # ends with the D2H read of the metric sums
        e1.record()
        barrier(world)
    ms = max_over_ranks(e0.elapsed_time(e1), device, world)
    fb = m._mma_total_fallback_rows
    del m
    torch.cuda.empty_cache()
    return {"users": n_total, "users_per_rank": n, "ms": ms, "users_per_s": n_total / (ms * 1e-3),
            "metrics": {k: float(v) for k, v in result.items()}, "rows_recomputed_exactly": fb,
            "what": "1M users x 200,001 items, top-20 + hits + Recall/MRR/NDCG/Hit/Precision, shards reduced over ranks"}


def host_threads():
    """All the host cores this process may use (torch.distributed.run exports OMP_NUM_THREADS=1 to its workers:
    the reference arm must not inherit that)."""
    try:
        return max(1, len(os.sched_getaffinity(0)))
    except AttributeError:
        return max(1, os.cpu_count() or 1)


def cpu_reference_steps(w, steps, warmup, budget_s=None, threads=None):
    """The reference's train step on the host cores.  With oracle/_ref present (the unmodified hopwise package,
    oracle/build_ref.py) this is hopwise's own model class -- its calculate_loss, dense autograd and the
    torch.optim.Adam its trainer builds (trainer.py:190) -- on an Interaction batch: kind "reference".  Without
    it, the torch-CPU restatement of oracle/kge_torch.py: kind "port".
    Returns (triples/s, steps timed, threads, seconds, kind, per-step seconds)."""
    from kge_helpers import tile_batch, to_cpu_batch

    torch.set_num_threads(threads or host_threads())
    batches = [to_cpu_batch(tile_batch(b, w["k"], w["k"])) for b in synth_batches(w, 2, 99)]
    kind = "port"
    try:
        from oracle import ref as oref

        if not oref.ref_available():
            raise RuntimeError("oracle/_ref not built")
        oref.import_ref()
        sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
        import importlib

        from _ref_harness import REF_CONFIG, FakeDataset
        from hopwise.data.interaction import Interaction

        mod = importlib.import_module(f"hopwise.model.knowledge_graph_embedding_recommender.{w['model'].lower()}")
        torch.manual_seed(2024)
        model = getattr(mod, w["model"])(dict(REF_CONFIG, embedding_size=w["d"], margin=1.0),
                                         FakeDataset(w["U"], w["I"], w["E"], w["R"]))
        opt = torch.optim.Adam(model.parameters(), lr=1e-3, weight_decay=0.0)   # trainer.py:165-190 defaults
        batches = [Interaction(b) for b in batches]

        def one(b):                      # trainer.py:252-265
            opt.zero_grad()
            loss = model.calculate_loss(b)
            loss.backward()
            opt.step()
            return loss

        kind = "reference"
    except Exception as exc:   # the port is the documented fallback, and the line says which one ran
        print(f"[bench] reference arm falls back to the oracle port: {exc!r}", file=sys.stderr)
        from kge_helpers import make_oracle_model
        from oracle.kge_torch import make_optimizer, train_step

        ora = make_oracle_model(w["model"], w["U"], w["I"], w["E"], w["R"], w["d"])
        opt = make_optimizer(ora)

        def one(b):
            return train_step(ora, opt, b)

    for i in range(warmup):
        one(batches[i % 2])
    per = []
    t0 = time.perf_counter()
    for i in range(steps):
        t1 = time.perf_counter()
        one(batches[i % 2])
        per.append(time.perf_counter() - t1)
        if budget_s is not None and time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    done = len(per)
    return done * (w["n_rec"] + w["n_kg"]) / dt, done, torch.get_num_threads(), dt, kind, per


def config1_pipeline(arm):
    """BASELINE config 1 -- TransE on the bundled ml-100k, d = 64, batch 2048, 1 negative -- through hopwise's OWN
    pipeline (Config -> create_dataset -> data_preparation -> get_model / get_trainer -> trainer), run from
    oracle/_ref.  arm "reference": hopwise's TransE + KGTrainer on the host cores.  arm "ours": the same
    factories after hopwise_b200.trainer.install(), i.e. hopwise_b200.TransE + FusedKGTrainer on the GPU; config,
    dataset, loaders and the (CPU, numpy) samplers are the reference's in both arms.  Timed: one training epoch
    (39 steps, 158,708 positive triples incl. the loader) and one full-sort evaluation of the test split."""
    try:
        from oracle import ref as oref

        if not oref.ref_available():
            return {"unavailable": "oracle/_ref is not built (oracle/build_ref.py needs /root/reference)"}
        oref.import_ref()
        import tempfile

        from hopwise.config import Config
        from hopwise.data import create_dataset, data_preparation
        from hopwise.utils import get_model, get_trainer, init_seed

        ours = arm == "ours"
        if ours:
            import hopwise_b200.trainer as fused

            fused.install()
        cwd = os.getcwd()
        visible = os.environ.get("CUDA_VISIBLE_DEVICES")     # hopwise's Config exports gpu_id into it
        os.chdir(tempfile.mkdtemp(prefix="hopwise_bench_"))   # hopwise writes log/ and log_tensorboard/ into the cwd
        try:
            torch.set_num_threads(host_threads())
            config = Config(model="TransE", dataset="ml-100k",
                            config_dict={"embedding_size": 64, "train_batch_size": 2048, "epochs": 1, "use_gpu": ours,
                                         # hopwise picks the device from gpu_id ("" = CPU, configurator.py:540-554)
                                         "gpu_id": "0" if ours else "",
                                         "show_progress": False, "eval_step": 1, "seed": 2024})
            init_seed(config["seed"], config["reproducibility"])
            dataset = create_dataset(config)
            train_data, valid_data, test_data = data_preparation(config, dataset)
            init_seed(config["seed"], config["reproducibility"])
            model = get_model(config["model"])(config, train_data.dataset).to(config["device"])
            trainer = get_trainer(config["MODEL_TYPE"], config["model"])(config, model)
            sync = torch.cuda.synchronize if ours else (lambda: None)
            triples = 0
            if ours:   # warm-up epoch: CUDA context, optimiser state, pinned staging (the reference needs none)
                trainer._train_epoch(train_data, 0)
            n_rec = len(train_data._dataset.inter_feat) if hasattr(train_data, "_dataset") else 78836
            steps = len(train_data)
            triples = n_rec + steps * 2048
            sync()
            t0 = time.perf_counter()
            loss = trainer._train_epoch(train_data, 1 if ours else 0)
            sync()
            t_train = time.perf_counter() - t0
            if ours:
                trainer.evaluate(test_data, load_best_model=False)   # builds the device plan of the loader
            sync()
            t0 = time.perf_counter()
            result = trainer.evaluate(test_data, load_best_model=False)
            sync()
            t_eval = time.perf_counter() - t0
            n_eval = len(test_data.uid_list)
            return {"arm": arm, "model": type(model).__module__ + "." + type(model).__name__,
                    "trainer": type(trainer).__name__, "device": str(config["device"]),
                    "train_epoch_s": t_train, "steps": steps, "triples_per_s": triples / t_train,
                    "epoch_loss": float(loss), "eval_s": t_eval, "eval_users": n_eval,
                    "eval_users_per_s": n_eval / t_eval, "metrics": {k: float(v) for k, v in result.items()},
                    "cores": torch.get_num_threads(),
                    "what": "one epoch (hopwise's loader + CPU samplers included) and one test-split evaluation"}
        finally:
            os.chdir(cwd)
            if visible is None:
                os.environ.pop("CUDA_VISIBLE_DEVICES", None)
            else:
                os.environ["CUDA_VISIBLE_DEVICES"] = visible
            if ours:
                fused.uninstall()
    except Exception as exc:   # report, never hide
        return {"error": repr(exc)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cfg2_transe_ml1m", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extras", action="store_true", help="headline only (used under ncu)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the loss and the tables of the last timed train step as DIR/<name>.npy (float32, at "
                         "most 64 MB: larger tables as a fixed, seeded sample of rows)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes what the CUDA train step computed: it needs --impl ours")
    args.warmup = max(args.warmup, 3)
    rank, world, local = dist_info()
    # stdout carries the one JSON line and nothing else: libraries that print to fd 1 (NCCL's version banner,
    # hopwise's loggers) are pointed at stderr for the run
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.write(json_fd, (json.dumps(line) + "\n").encode())
    w = WORKLOADS[args.workload]
    triples_step = w["n_rec"] + w["n_kg"]
    config = {"workload": f"{args.workload}: {w['model']} d={w['d']} U={w['U']} I={w['I']} E={w['E']} R={w['R']} "
                          f"K={w['k']} batch={w['n_rec']}rec+{w['n_kg']}kg positives/step/GPU, uniform synthetic KG, Adam lr=1e-3",
              "parallelism": f"dp{world}" if world > 1 else "single",
              "l2": "L2 flushed (256 MiB memset) between timed steps"}

    if args.impl == "reference":
        if rank != 0:
            return
        # bounded sample: one step is the full batch when it fits a few seconds, else a slice
        # W warm-up steps and K timed steps as asked (a step of the full batch is ~0.4 s on 16 cores); the budget
        # only guards a box with very few cores
        tps, done, threads, dt, kind, per = cpu_reference_steps(w, args.steps, args.warmup, budget_s=240)
        line = {"metric": "KG triples/sec (train step)", "value": tps, "unit": "triples/s", "n_gpus": args.gpus,
                "steps": done, "warmup": args.warmup, "ms_per_step": 1e3 * dt / done,
                "median_ms_per_step": 1e3 * float(np.median(per)),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "impl": "reference", "config": config,
                "cpu_baseline": {"value": tps, "unit": "triples/s", "cores": threads, "kind": kind,
                                 "sample": f"{done} steps of the full {triples_step}-triple batch "
                                           + ("(hopwise's own model class from oracle/_ref, dense autograd + torch.optim.Adam)"
                                              if kind == "reference" else "(torch-CPU oracle port, dense Adam)")},
                "e2e": {"value": tps, "unit": "triples/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0}
        if not args.no_extras:
            line["extras"] = {"cfg1_ml100k_pipeline": config1_pipeline("reference")}
        emit(line)
        return

    assert torch.cuda.is_available(), "bench.py --impl ours needs a CUDA device"
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        import torch.distributed as dist

        # measured on 8 B200 (scripts/allreduce_probe.py): the 14.7 MB gradient all-reduce of this workload takes
        # 78 us with the ring algorithm, 95 us with NCCL's default choice (NVLS); a user's own setting wins
        os.environ.setdefault("NCCL_ALGO", "Ring")
        dist.init_process_group("nccl", device_id=device)
    from hopwise_b200 import _abi

    _abi.lib()
    model = make_model(w, device)
    exchange = None
    if world > 1:
        from hopwise_b200.distributed import broadcast_weights, enable_row_sparse_data_parallel

        broadcast_weights(model)
        # dense route: this library's in-switch (NVLS multimem) all-reduce on more than 4 GPUs -- measured, ms/step
        # in-switch vs NCCL: 8 B200 0.527 vs 0.564, 4 B200 0.487 vs 0.479, 2 B200 0.483 vs 0.462 (the two barriers
        # around the kernel cost more than NCCL's exchange until the ring gets long).  KGE_MULTIMEM=0 / 1 forces it.
        mm = os.environ.get("KGE_MULTIMEM")
        # The optimiser step itself runs owner-sharded over the switch when the fabric has multicast memory (one
        # kernel: reduce 1/N of the gradient, dense Adam on it, multicast the weights) -- it fits this workload,
        # whose batch touches every row.  Measured, ms/step at 8 / 2 B200: owner 0.417 / 0.406, in-switch
        # all-reduce + Adam 0.463 / 0.441, NCCL all-reduce + Adam 0.489 / 0.440 (profiles/r2_bench_n8_*.json).
        # KGE_OWNER_ADAM=0 / 1 and KGE_MULTIMEM=0 / 1 force a route.
        oa = os.environ.get("KGE_OWNER_ADAM")
        owner = "auto" if oa is None and mm is None else oa == "1"
        exchange = enable_row_sparse_data_parallel(model, multimem=(world > 4) if mm is None else mm != "0",
                                                   owner_adam=owner)
        if os.environ.get("KGE_MULTIMEM_FUSED") == "0":   # A/B: host-launched barriers around the plain kernel
            exchange.fused_barriers = False

    n_batches = 4
    host = synth_batches(w, n_batches, seed=2024 + rank)
    host_t = [{k: torch.from_numpy(v).pin_memory() for k, v in b.items()} for b in host]
    dev_t = [{k: v.to(device) for k, v in b.items()} for b in host_t]
    flush_buf = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=device)
    h2d = sum(v.numel() * 4 for v in host_t[0].values())   # staged as int32 (time_train_e2e)
    peaks = measured_peaks()

    with ClockSampler(local) as clocks:
        fwd, upd, last_loss = time_train_device(model, dev_t, args.steps, args.warmup, flush_buf, world)
    clk = clocks.summary()
    if args.dump_outputs:
        state = model.state_dict()   # on every rank: the lazy-row flush is the same work on all of them
        if rank == 0:
            dump_outputs(args.dump_outputs, state, last_loss)
        del state
    per_step = fwd + upd
    step_ms = max_over_ranks(float(per_step.mean()), device, world)          # EXACTLY K timed steps, max over ranks
    step_med_ms = max_over_ranks(float(np.median(per_step)), device, world)
    fwd_ms_avg = max_over_ranks(float(fwd.mean()), device, world)
    upd_ms_avg = max_over_ranks(float(upd.mean()), device, world)
    value = world * triples_step / (step_ms * 1e-3)

    rank_split = None
    if world > 1:
        # what the synchronous step costs beyond the slowest rank's forward: per step, the slowest forward over the
        # ranks and the shortest backward (the rank that arrives last waits for nobody: its backward is the exchange
        # + optimiser cost proper; the others' include waiting for it)
        import torch.distributed as dist

        mine = torch.tensor(np.stack([fwd, upd]), dtype=torch.float64, device=device)
        allr = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        allr = torch.stack(allr).cpu().numpy()          # [world, 2, steps]
        rank_split = {"fwd_ms_mean_over_ranks": float(allr[:, 0].mean()),
                      "fwd_ms_slowest_rank_per_step": float(allr[:, 0].max(axis=0).mean()),
                      "backward_ms_last_arriver_per_step": float(allr[:, 1].min(axis=0).mean()),
                      "backward_ms_mean_over_ranks": float(allr[:, 1].mean())}

    e2e_ms, e2e_median_ms, e2e_max_ms = time_train_e2e(model, host_t, args.steps, args.warmup, world, device)
    e2e_ms = max_over_ranks(e2e_ms / args.steps, device, world)
    e2e_value = world * triples_step / (e2e_ms * 1e-3)
    ref_order_ms, _, _ = time_train_e2e(model, host_t, args.steps, args.warmup, world, device, reference_order=True)
    ref_order_ms = max_over_ranks(ref_order_ms / args.steps, device, world)

    bpt = bytes_per_triple(w["model"], w["d"], w["k"])
    achieved = triples_step * bpt / (step_ms * 1e-3) / 1e9
    traffic, traffic_src = profiled_traffic(args.workload)
    dram_frac = None if traffic is None else traffic / (step_ms * 1e-3) / 1e9 / peaks["hbm_gbs"]
    # What bounds the step depends on whether the tables fit the 126 MB L2.  cfg2 (36k rows, every row referenced
    # ~40x per step) is L2-resident: DRAM moves a few % of the algorithmic bytes and the kernel is bound by
    # instruction issue and L2 atomics, so the algorithmic fraction (> 1 there) is NOT a statement about HBM; the
    # line says so (`bound`), carries the measured DRAM fraction beside it, and reports the HBM-regime workload
    # (cfg5: 1M-row tables, no reuse) as `roofline_hbm`.
    l2_resident = (w["U"] + w["E"]) * w["d"] * PARTS[w["model"]] * 16 < 100e6   # w, m, v, g of user + entity tables
    roof = {"bound": "issue/L2 (tables L2-resident; see dram_frac)" if l2_resident else "hbm",
            "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s",
            "frac": achieved / peaks["hbm_gbs"], "algorithmic_frac": achieved / peaks["hbm_gbs"],
            "dram_frac": dram_frac, "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes": triples_step * bpt, "peak_source": peaks["source"],
            "kernels": "train_fwd_kernel + adam_apply_kernel (the two launches of one step)",
            "fwd_ms": fwd_ms_avg, "adam_ms": upd_ms_avg, "bytes_per_triple": bpt}

    line = {"metric": "KG triples/sec (train step)", "value": value, "unit": "triples/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": step_ms, "median_ms_per_step": step_med_ms,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "e2e": {"value": e2e_value, "unit": "triples/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": 4,
                    "ms_per_step": e2e_ms, "median_ms_per_step": e2e_median_ms, "max_ms_per_step": e2e_max_ms,
                    "what": "pinned int32 ids -> H2D (copy stream, one batch ahead) -> model.train_step -> async D2H of the "
                            "loss into pinned memory, read by the host one step later (after its event) while the "
                            "next step runs; all inside the timed region",
                    "reference_loop_order_ms_per_step": ref_order_ms,
                    "reference_loop_order": "calculate_loss -> loss.item() -> backward (trainer.py:257-263): the "
                                            "mid-step sync idles the GPU while the host turns around"},
            # this library's kernels in the timed region: forward + Adam per step, plus the pack / add kernels of
            # the row-sparse exchange when a table takes that route (NCCL's own kernels are not counted)
            "gpu_launches": args.steps * ((1 if exchange is not None and exchange.owner_adam else 2)
                                          + (exchange.kernels_per_step if exchange is not None else 0)),
            "roofline": roof, "clocks": clk, "final_loss": last_loss}
    if exchange is not None:
        line["rank_split"] = rank_split
        line["exchange_bytes_per_rank_per_step"] = exchange.bytes_per_step
        line["exchange"] = ("owner-sharded Adam over the switch: multimem.ld_reduce of 1/N of the gradient, dense Adam, "
                            "multimem.st of the weights, barriers inside the kernel (csrc/collective.cu)"
                            if exchange.owner_adam else
                            ("nvls multimem all-reduce (csrc/collective.cu)"
                             + (", barriers and touch marks inside the kernel" if exchange.fused_barriers else "")
                             ) if exchange.multimem else "nccl all-reduce")
        line["exchange_routes_dense"] = list(exchange.dense)

    def train_leg(name, steps, world_, data_parallel=False):
        """One more training workload on this rank's GPU (and, with data_parallel, its exchange across ranks)."""
        wx = WORKLOADS[name]
        mx = make_model(wx, device)
        ex = None
        if data_parallel:
            from hopwise_b200.distributed import broadcast_weights, enable_row_sparse_data_parallel

            broadcast_weights(mx)
            ex = enable_row_sparse_data_parallel(mx, multimem=False)
            ex.timing = True
        hb = synth_batches(wx, 4, seed=7 + rank)
        db = [{k: torch.from_numpy(v).to(device) for k, v in b.items()} for b in hb]
        f, u, _ = time_train_device(mx, db, steps, args.warmup, flush_buf, world_)
        if ex is not None:
            ex.take_timings()   # (drop the warm-up's events: time_train_device warms up first ... they are mixed in)
        per = f + u
        ms = max_over_ranks(float(per.mean()), device, world_)
        med = max_over_ranks(float(np.median(per)), device, world_)
        t = wx["n_rec"] + wx["n_kg"]
        bx = bytes_per_triple(wx["model"], wx["d"], wx["k"])
        out = {"triples_per_s": world_ * t / (ms * 1e-3), "ms_per_step": ms, "median_ms_per_step": med,
               "fwd_ms": float(f.mean()), "adam_ms": float(u.mean()), "bytes_per_triple": bx,
               "hbm_frac": t * bx / (ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
               "hbm_frac_from_median": t * bx / (med * 1e-3) / 1e9 / peaks["hbm_gbs"]}
        if t <= 8192 and ex is None:
            # the reference's default batch is launch/latency bound: also time the trainer's one-call step
            # (model.train_step: forward + Adam queued by one library call) back to back, as an epoch runs it
            n_loop = 400
            for i in range(20):
                mx.train_step(db[i % 4])
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            e0.record()
            for i in range(n_loop):
                mx.train_step(db[i % 4])
            e1.record()
            host_s = time.perf_counter() - t0
            torch.cuda.synchronize()
            out["train_step_call"] = {
                "what": f"{n_loop} back-to-back model.train_step calls (no L2 flush, no per-step sync)",
                "device_ms_per_step": e0.elapsed_time(e1) / n_loop, "host_issue_ms_per_step": 1e3 * host_s / n_loop,
                "triples_per_s": t / (e0.elapsed_time(e1) / n_loop * 1e-3)}
        if ex is not None:
            # split of the exchange (inside `adam_ms`, which covers backward = exchange + Adam): a few more steps
            for i in range(8):
                mx.calculate_loss(db[i % 4]).backward()
            tm = np.array(ex.take_timings())
            out.update({"exchange": "row-sparse: pack -> one NCCL all-gather -> add" if not all(ex.dense) else
                                    "dense all-reduce", "routes_dense": list(ex.dense),
                        "exchange_bytes_per_rank_per_step": ex.bytes_per_step,
                        "pack_ms": float(np.median(tm[:, 0])), "collective_ms": float(np.median(tm[:, 1])),
                        "add_ms": float(np.median(tm[:, 2])), "kernels_per_step": 2 + ex.kernels_per_step})
        del mx, db
        torch.cuda.empty_cache()
        return out

    if not args.no_extras:
        extras = {}
        # more training workloads: the reference's default batch on the same KG (launch / latency bound), the HBM
        # regime (cfg5: 1M entities), 64 negatives (cfg3); on several GPUs the same with the exchange running
        legs = ("cfg2_transe_ml1m_b2048", "cfg5_transe_alibaba", "cfg5_transe_alibaba_b2048", "cfg3_rotate_yelp")
        if args.workload == "cfg2_transe_ml1m":
            for name in legs:
                try:
                    extras[name] = train_leg(name, args.steps, world, data_parallel=world > 1)
                except Exception as exc:  # report, never hide
                    extras[name] = {"error": repr(exc)}
            c5 = extras.get("cfg5_transe_alibaba", {})
            if "hbm_frac" in c5:   # first-class: the HBM-regime roofline statement of the same kernels
                line["roofline_hbm"] = {
                    "workload": "cfg5_transe_alibaba (TransE d=128, E=1,000,001: tables 8x the L2, no row reuse)",
                    "bound": "hbm", "achieved": c5["hbm_frac"] * peaks["hbm_gbs"], "peak": peaks["hbm_gbs"],
                    "unit": "GB/s", "frac": c5["hbm_frac"], "frac_from_median": c5["hbm_frac_from_median"],
                    "ms_per_step": c5["ms_per_step"], "bytes_per_triple": c5["bytes_per_triple"]}
        # the whole reference step at its default batch, loader included: batch order from the CPU torch
        # generators, gathers + both MT19937 samplers + fused step on the device (hopwise_b200.loader.DeviceKGLoader)
        if args.workload == "cfg2_transe_ml1m" and world == 1:
            try:
                from hopwise_b200.loader import DeviceKGLoader
                from hopwise_b200.sampler import KGSampler, MTStream, RecSampler

                wx = WORKLOADS["cfg2_transe_ml1m_b2048"]
                rng = np.random.default_rng(2024)
                iu, ii = rng.integers(1, wx["U"], wx["inters"]), rng.integers(1, wx["I"], wx["inters"])
                kh, kr, kt = (rng.integers(1, wx["E"], wx["triples"]), rng.integers(1, wx["R"] - 1, wx["triples"]),
                              rng.integers(1, wx["E"], wx["triples"]))
                mt = MTStream(seed=2024, device=device)
                loader = DeviceKGLoader(iu, ii, kh, kr, kt, RecSampler(iu, ii, wx["U"], wx["I"], stream=mt, device=device),
                                        KGSampler(heads=kh, tails=kt, entity_num=wx["E"], stream=mt, device=device),
                                        batch_size=wx["n_rec"], seed=2024, device=device)
                mx = make_model(wx, device)
                n_steps = max(args.steps, 20) * 5
                it = iter(loader)
                for _ in range(10):
                    b = next(it)
                    mx.train_step(b)
                torch.cuda.synchronize()
                stamps = [time.perf_counter()]
                for _ in range(n_steps):
                    b = next(it)
                    mx.train_step(b).item()     # the reference loop reads the loss every step (trainer.py:257-263)
                    stamps.append(time.perf_counter())
                torch.cuda.synchronize()
                per = np.diff(np.array(stamps))
                # the same with every loss read one step late through pinned memory (an async D2H copy + event right
                # behind the step, read once the next step has been issued): loss.item() waits for the whole stream,
                # the next batch's loader kernels included
                host_loss = [torch.zeros(1).pin_memory() for _ in range(2)]
                evs = [torch.cuda.Event() for _ in range(2)]
                losses = []
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for i in range(n_steps):
                    loss = mx.train_step(next(it))
                    host_loss[i % 2].copy_(loss.reshape(1), non_blocking=True)
                    evs[i % 2].record()
                    if i:
                        evs[(i - 1) % 2].synchronize()
                        losses.append(float(host_loss[(i - 1) % 2]))
                evs[(n_steps - 1) % 2].synchronize()
                losses.append(float(host_loss[(n_steps - 1) % 2]))
                late_s = (time.perf_counter() - t0) / n_steps
                extras["cfg2_b2048_device_loader"] = {
                    "what": "loader (order + gathers + KG and rec negative sampling) + fused step + loss.item(), wall clock",
                    "ms_per_step": float(per.mean()) * 1e3, "median_ms_per_step": float(np.median(per)) * 1e3,
                    "triples_per_s": (wx["n_rec"] + wx["n_kg"]) / float(per.mean()),
                    "ms_per_step_loss_read_one_step_late": late_s * 1e3, "loss_sum": float(np.sum(losses))}
                del mx, loader
                torch.cuda.empty_cache()
            except Exception as exc:
                extras["cfg2_b2048_device_loader"] = {"error": repr(exc)}
        # BASELINE config 1 through hopwise's own pipeline (oracle/_ref) with the fused models + FusedKGTrainer
        if args.workload == "cfg2_transe_ml1m" and world == 1:
            extras["cfg1_ml100k_pipeline"] = config1_pipeline("ours")
        # second headline metric: users/s of full-sort top-k (user blocks sharded across ranks)
        for name, fs in FULLSORT.items():
            try:
                n_users_step = 148 * 512   # two CTAs of 256 users per SM: one full wave of the tcgen05 sweep
                reps = max(6, args.steps // 2)
                flops = 2.0 * fs["I"] * fs["d"] * PARTS[fs["model"]]
                entry = {"metric": "users/sec (full-sort top-20)", "users_per_block_per_gpu": n_users_step}
                for path in ("mma", "cuda"):
                    if path == "cuda":
                        reps = 3   # ~0.1 s per block
                    ms, fb, med, in_order = time_fullsort(fs, device, n_users_step, reps, 3, world, rank, path=path)
                    ms = max_over_ranks(ms / reps, device, world)
                    med = max_over_ranks(med, device, world)
                    # headline = the MEAN block (nothing in the call waits for the host any more: the exact fallback
                    # is gated on the device, the workspace is cached); the median is beside it
                    ups = world * n_users_step / (ms * 1e-3)
                    entry[path] = {"users_per_s": ups, "mean_ms_per_block": ms, "median_ms_per_block": med,
                                   "users_per_s_from_median": world * n_users_step / (med * 1e-3),
                                   "algorithmic_tflops": ups * flops / 1e12,
                                   "tensor_frac_of_bf16_peak": ups / world * flops / 1e12 / peaks["bf16_tflops"],
                                   "rows_recomputed_exactly": fb, "per_block_ms": [round(x, 3) for x in in_order]}
                entry["paths"] = {"mma": "tcgen05 fp16 filter (proven bound) + exact fp32 re-score (same ids/scores)",
                                  "cuda": "fp32 CUDA-core tile kernel"}
                extras[name] = entry
            except Exception as exc:
                extras[name] = {"error": repr(exc)}
        # the whole cfg4 evaluation: 1,000,000 users sharded in contiguous blocks over the ranks, top-20, hits,
        # Recall / MRR / NDCG / Hit / Precision sums and their reduction over the ranks inside the timed region
        try:
            extras["cfg4_distmult_full_eval"] = full_eval_leg(FULLSORT["cfg4_distmult"], device, world, rank)
        except Exception as exc:
            extras["cfg4_distmult_full_eval"] = {"error": repr(exc)}
        line["extras"] = extras

    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        tps, done, threads, dt, kind, _ = cpu_reference_steps(w, 1000, 1, budget_s=15)
        line["cpu_baseline"] = {"value": tps, "unit": "triples/s", "cores": threads, "kind": kind,
                                "sample": f"{done} steps of the full {triples_step}-triple batch in {dt:.1f}s ("
                                          + ("hopwise's own model class from oracle/_ref" if kind == "reference"
                                             else "torch-CPU oracle port") + ", dense autograd + dense Adam)"}
    if rank == 0:
        emit(line)
    if world > 1:
        import torch.distributed as dist

        dist.destroy_process_group()


if __name__ == "__main__":
    main()
