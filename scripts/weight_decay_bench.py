"""Step time of the fused train step with and without weight decay; prints one JSON line (and writes it with --out).

TransE, one negative, on the bench.py workloads' synthetic graphs (uniform ids, seed 2024):
  cfg2 -- 6,041 users, 30,001 entities, d = 100: the tables fit the 126 MB L2; batches 2,048 + 2,048 and 262,144 + 262,144;
  cfg5 -- 115,001 users, 1,000,001 entities, d = 128: the tables are ~8x the L2; batch 2,048 + 2,048.
Per (workload, batch) `model.train_step` (one kge_train_step call) is timed with CUDA events for Adam (weight decay 0),
AdamW(lr 1e-3, weight_decay 0.01) and SGD(lr 0.1, weight_decay 0.01), each from the same initial weights and batches.
At cfg5 one `flush()` after the timed AdamW steps is timed too: under weight decay it moves every row of every table
(1.1 M rows), where Adam's moves only the rows that lag.  Last, the same AdamW steps through oracle/kge_torch's model
with autograd and dense torch.optim.AdamW on the same GPU (its losses of the first two steps are compared with the
fused ones).  The card's name, power limit and top SM clock are read in the same run.

    python scripts/weight_decay_bench.py [--steps 50] [--warmup 10] [--out FILE]
"""

import argparse
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from rank_bench import gpu_info, timed  # noqa: E402

GRAPHS = {"cfg2": dict(U=6041, I=3001, E=30001, R=22, d=100), "cfg5": dict(U=115001, I=30001, E=1000001, R=54, d=128)}
CASES = (("cfg2", 2048), ("cfg2", 262_144), ("cfg5", 2048))
LEARNERS = {"adam": dict(learner="adam", lr=1e-3), "adamw": dict(learner="adamw", lr=1e-3, weight_decay=0.01),
            "sgd": dict(learner="sgd", lr=0.1, weight_decay=0.01)}


def batches(rng, g, n, count, dev):
    out = []
    for _ in range(count):
        b = {"user_id": rng.integers(1, g["U"], n), "item_id": rng.integers(1, g["I"], n),
             "neg_item_id": rng.integers(1, g["I"], n), "head_id": rng.integers(1, g["E"], n),
             "relation_id": rng.integers(0, g["R"] - 1, n), "tail_id": rng.integers(1, g["E"], n),
             "neg_tail_id": rng.integers(1, g["E"], n)}
        out.append({k: torch.from_numpy(v).to(dev) for k, v in b.items()})
    return out


def cycle(items):
    state = {"i": 0}

    def nxt():
        x = items[state["i"] % len(items)]
        state["i"] += 1
        return x
    return nxt


def summary(ms):
    ms = np.asarray(ms)
    return {"ms_per_step_median": float(np.median(ms)), "ms_per_step_mean": float(ms.mean()),
            "ms_per_step_min": float(ms.min()), "steps": len(ms)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("weight_decay_bench.py measures on the GPU: no CUDA device")
    from kge_helpers import make_product_model
    from oracle.kge_torch import OracleKGE, Shapes, make_optimizer
    from oracle.kge_torch import train_step as torch_train_step

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    out = {"metric": "weight_decay_train_step", "gpu": gpu_info(), "model": "TransE", "negatives": 1,
           "graphs": GRAPHS, "learners": LEARNERS, "steps": args.steps, "warmup": args.warmup, "cases": {}}
    for gname, n in CASES:
        g = GRAPHS[gname]
        rng = np.random.default_rng(2024)
        bs = batches(rng, g, n, 8, dev)
        res = {}
        init = None
        for lname, cfg in LEARNERS.items():
            with torch.device(dev):
                m = make_product_model("TransE", g["U"], g["I"], g["E"], g["R"], g["d"], device=dev, **cfg)
            if init is None:
                init = {k: v.clone() for k, v in m.state_dict().items()}
            if lname == "adamw":   # (from the initial weights, as the torch comparator's below)
                res["adamw_first_losses"] = [float(m.train_step(bs[0])), float(m.train_step(bs[1]))]
            res[lname] = summary(timed(lambda nxt=cycle(bs): m.train_step(nxt()), args.steps, args.warmup))
            if lname == "adamw":
                if gname == "cfg5":
                    ms = timed(m.flush, 1, 0)   # one flush of every row (1.1 M rows, d = 128)
                    res["adamw_flush_ms"] = ms[0]
            del m
            torch.cuda.empty_cache()
        res["adamw_over_adam_median"] = res["adamw"]["ms_per_step_median"] / res["adam"]["ms_per_step_median"]
        res["sgd_over_adam_median"] = res["sgd"]["ms_per_step_median"] / res["adam"]["ms_per_step_median"]
        with torch.device(dev):
            ora = OracleKGE("TransE", Shapes(g["U"], g["I"], g["E"], g["R"], g["d"]))
        ora.load_state_dict(init)
        opt = make_optimizer(ora, lr=1e-3, weight_decay=0.01, learner="adamw")

        def torch_step(nxt=cycle(bs)):
            opt.zero_grad()
            ora.calculate_loss(nxt()).backward()
            opt.step()
        res["torch_autograd_dense_adamw"] = summary(timed(torch_step, args.steps, args.warmup))
        ora.load_state_dict(init)
        opt = make_optimizer(ora, lr=1e-3, weight_decay=0.01, learner="adamw")
        res["torch_first_losses"] = [torch_train_step(ora, opt, bs[0]), torch_train_step(ora, opt, bs[1])]
        res["speedup_over_torch_median"] = (res["torch_autograd_dense_adamw"]["ms_per_step_median"]
                                            / res["adamw"]["ms_per_step_median"])
        del ora, opt, init
        torch.cuda.empty_cache()
        out["cases"][f"{gname}_b{n}"] = res
        print(json.dumps({f"{gname}_b{n}": {k: v["ms_per_step_median"] if isinstance(v, dict) else v
                                            for k, v in res.items()}}), file=sys.stderr, flush=True)
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
