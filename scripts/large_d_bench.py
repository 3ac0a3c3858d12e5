"""Training step and link-prediction top-10 at embedding_size 1,000; prints one JSON line (and writes it with --out).

TransE, RotatE and ComplEx at d = 1,000 (RotatE / ComplEx: two tables per entity), one negative per positive, on two
synthetic graphs (uniform ids, seed 2024):
  fb15k237 -- 14,541 entities, 237 relations (+ the user->item relation), 10,000 users, 10,000 items: the shape of
              FB15k-237.  The entity weights are 58 MB per table, so they stay in the 126 MB L2 for TransE (one table)
              and fill it for RotatE / ComplEx (two); weights + Adam moments + gradient accumulators (16 B per
              element) do not fit;
  e1m      -- 1,000,001 entities, 100,000 users and items: every table far beyond the L2, the step is bound by HBM.
Per (graph, model, batch) the fused step (`model.train_step`: one kge_train_step call) is timed with CUDA events,
and so is the comparator on the same GPU: oracle/kge_torch's model with autograd and dense torch.optim.Adam
(zero_grad, loss, backward, step), started from the same weights.  Both see the same batches; the losses of the
first two steps (the second one after one update) are compared.  Batches: the reference's 2,048 + 2,048 and a
roofline batch of 65,536 + 65,536.  `bytes_per_triple = 24·d·T·(2+K) + 8·(3+K)` (SURVEY §(d)) over the step time
gives the algorithmic bandwidth, reported as a fraction of 6,552 GB/s (the measured HBM bandwidth SURVEY §(d) uses;
on fb15k237 the rows repeat and come from L2, so the fraction there is not a DRAM figure).
Last, full-sort link-prediction top-10 (`full_sort_topk_kg`, CUDA cores, every entity a target, the pad entity and
10 known tails per query masked) on fb15k237 for 20,000 (head, relation) queries: queries/s.
The card's name, power limit and top SM clock are read in the same run.

    python scripts/large_d_bench.py [--steps 10] [--warmup 3] [--out FILE]
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

D = 1000
HBM_GBS = 6552.0
GRAPHS = {"fb15k237": dict(U=10_000, I=10_000, E=14_541, R=238), "e1m": dict(U=100_000, I=100_000, E=1_000_001, R=238)}
MODELS = ("TransE", "RotatE", "ComplEx")
PARTS = {"TransE": 1, "RotatE": 2, "ComplEx": 2}
BATCHES = {"b2048": 2048, "roofline": 65_536}
N_LP, K_LP, HIST_LP = 20_000, 10, 10


def bytes_per_triple(model, d, k):
    return 24 * d * PARTS[model] * (2 + k) + 8 * (3 + k)


def batches(rng, g, n, count, dev):
    out = []
    for _ in range(count):
        b = {"user_id": rng.integers(1, g["U"], n), "item_id": rng.integers(1, g["I"], n),
             "neg_item_id": rng.integers(1, g["I"], n), "head_id": rng.integers(1, g["E"], n),
             "relation_id": rng.integers(0, g["R"] - 1, n), "tail_id": rng.integers(1, g["E"], n),
             "neg_tail_id": rng.integers(1, g["E"], n)}
        out.append({k: torch.from_numpy(v).to(dev) for k, v in b.items()})
    return out


def stats(ms, positives, bpt):
    ms = np.asarray(ms)
    med = float(np.median(ms))
    gbs = positives * bpt / (med / 1e3) / 1e9
    return {"ms_per_step_median": med, "ms_per_step_mean": float(ms.mean()), "ms_per_step_min": float(ms.min()),
            "positives_per_s": positives / (med / 1e3), "algorithmic_gb_per_s": gbs,
            "fraction_of_6552_gbs": gbs / HBM_GBS, "steps": len(ms)}


def cycle(items):
    state = {"i": 0}

    def nxt():
        x = items[state["i"] % len(items)]
        state["i"] += 1
        return x
    return nxt


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("large_d_bench.py measures on the GPU: no CUDA device")
    from kge_helpers import make_product_model
    from oracle.kge_torch import OracleKGE, Shapes, make_optimizer
    from oracle.kge_torch import train_step as torch_train_step

    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    out = {"metric": "large_d_train_step_and_lp_topk", "gpu": gpu_info(), "d": D, "negatives": 1,
           "graphs": GRAPHS, "batches": {k: f"{v} + {v}" for k, v in BATCHES.items()}, "hbm_gbs": HBM_GBS,
           "steps": args.steps, "warmup": args.warmup, "train": {}, "lp_topk": {}}
    for gname, g in GRAPHS.items():
        for name in MODELS:
            res = {}
            for bname, n in BATCHES.items():
                rng = np.random.default_rng(2024)
                bs = batches(rng, g, n, 4, dev)
                bpt = bytes_per_triple(name, D, 1)
                with torch.device(dev):   # (the tables are initialised on the device)
                    m = make_product_model(name, g["U"], g["I"], g["E"], g["R"], D, device=dev)
                init = {k: v.clone() for k, v in m.state_dict().items()}
                fused_losses = [float(m.train_step(bs[0])), float(m.train_step(bs[1]))]
                fused = timed(lambda nxt=cycle(bs): m.train_step(nxt()), args.steps, args.warmup)
                del m
                torch.cuda.empty_cache()
                with torch.device(dev):
                    ora = OracleKGE(name, Shapes(g["U"], g["I"], g["E"], g["R"], D))
                ora.load_state_dict(init)
                del init
                opt = make_optimizer(ora)
                torch_losses = [torch_train_step(ora, opt, bs[0]), torch_train_step(ora, opt, bs[1])]

                def torch_step(nxt=cycle(bs)):
                    opt.zero_grad()
                    ora.calculate_loss(nxt()).backward()
                    opt.step()
                comp = timed(torch_step, args.steps, args.warmup)
                del ora, opt
                torch.cuda.empty_cache()
                f, c = stats(fused, 2 * n, bpt), stats(comp, 2 * n, bpt)
                res[bname] = {"fused_train_step": f, "torch_autograd_dense_adam": c,
                              "speedup_median": c["ms_per_step_median"] / f["ms_per_step_median"],
                              "bytes_per_triple": bpt,
                              "losses": {"fused": fused_losses, "torch": torch_losses,
                                         "max_rel_diff": max(abs(a - b) / abs(b) for a, b in
                                                             zip(fused_losses, torch_losses))}}
            out["train"].setdefault(gname, {})[name] = res
            print(json.dumps({gname: {name: {b: (r["fused_train_step"]["ms_per_step_median"],
                                                 r["torch_autograd_dense_adam"]["ms_per_step_median"],
                                                 r["losses"]["max_rel_diff"]) for b, r in res.items()}}}),
                  file=sys.stderr, flush=True)
    g = GRAPHS["fb15k237"]
    for name in MODELS:
        rng = np.random.default_rng(2024)
        with torch.device(dev):
            m = make_product_model(name, g["U"], g["I"], g["E"], g["R"], D, device=dev)
        heads = torch.from_numpy(rng.integers(1, g["E"], N_LP)).to(dev)
        rels = torch.from_numpy(rng.integers(0, g["R"] - 1, N_LP)).to(dev)
        hist = np.sort(rng.integers(1, g["E"], (N_LP, HIST_LP)), axis=1)
        ho = torch.arange(0, HIST_LP * N_LP + 1, HIST_LP, dtype=torch.long, device=dev)
        hi = torch.from_numpy(hist.reshape(-1)).to(dev)
        ms = timed(lambda: m.full_sort_topk_kg(heads, rels, K_LP, ho, hi, path="cuda"), args.steps, args.warmup)
        med = float(np.median(ms))
        out["lp_topk"][name] = {"queries": N_LP, "targets": g["E"], "k": K_LP, "ms_per_call_median": med,
                                "ms_per_call_mean": float(np.mean(ms)), "queries_per_s": N_LP / (med / 1e3),
                                "flop_per_s": 2.0 * N_LP * g["E"] * PARTS[name] * D / (med / 1e3)}
        del m
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
