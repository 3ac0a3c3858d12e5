"""Fused full-sort top-k above k = 128 at the BASELINE config 4 shape; prints one JSON line (and writes it to --out).

DistMult and ComplEx, d = 64, 200,001 items, 50 history items per user, seed 2024.  Legs:
  (a) model.full_sort_topk(path="cuda") on a block of 75,776 users at k = 128 (the sorted-list epilogue) and at
      k = 200, 500, 1000 (the large-k epilogue: per-row buffers in the workspace, a merge kernel);
  (b) the dense route the trainer took for k > 128 before the large-k epilogue, on 2,048 users: full_sort_predict,
      the trainer's masking, then torch.topk, at the same k.
Each leg is reported in users/s (mean and median over the timed calls, after warm-up).  The entity table (51 MB for
DistMult, 102 MB for ComplEx) fits the 126 MB L2 and is not flushed between calls: every leg reads it warm.
The script checks that (a) and (b) return the same ids on the users they share, up to the order of exactly tied
scores (torch.topk orders ties as it likes; the fused path by ascending id), and the same scores.  The card's name,
power limit and top SM clock are read in the same run (an nvidia-smi query).

    python scripts/topk_large_bench.py [--steps 5] [--warmup 1] [--out FILE]
"""

import argparse
import json
import os
import subprocess
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

N_BLOCK, N_DENSE, I, HIST, D = 75_776, 2_048, 200_001, 50, 64
KS = (128, 200, 500, 1000)


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def dense_topk(m, users, hist_rows, hist_cols, k):
    """trainer.py's _full_sort_batch_eval masking + the collector's torch.topk, on dense rows."""
    scores = m.full_sort_predict({"user_id": users})
    scores[:, 0] = -torch.inf
    scores[hist_rows, hist_cols] = -torch.inf
    return torch.topk(scores, k, dim=-1)


def timed(fn, steps, warmup):
    for _ in range(warmup):
        fn()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    torch.cuda.synchronize()
    ev[0].record()
    for i in range(steps):
        fn()
        ev[i + 1].record()
    torch.cuda.synchronize()
    return [ev[i].elapsed_time(ev[i + 1]) for i in range(steps)]


def rate(ms, n_users):
    ms = np.asarray(ms)
    return {"users_per_s_mean": float(n_users / (ms.mean() / 1e3)), "users_per_s_median": float(n_users / (np.median(ms) / 1e3)),
            "ms_per_call_mean": float(ms.mean()), "ms_per_call_median": float(np.median(ms)), "calls": len(ms)}


def compare(ids_f, sc_f, dense):
    """Fused (ids, scores) against torch.topk's (values, indices) on the same rows.  The scores must be equal position
    by position.  torch.topk orders tied scores as it likes and may cut a tie at the k-th score differently: its ids
    are put in the canonical order (score desc, id asc) and compared at every position scoring above the k-th score."""
    vals, idx = dense
    o = torch.argsort(idx, dim=1, stable=True)
    v1, i1 = torch.gather(vals, 1, o), torch.gather(idx, 1, o)
    canon = torch.gather(i1, 1, torch.argsort(-v1, dim=1, stable=True))
    above = vals > vals[:, -1:]
    scores_equal = bool(torch.equal(sc_f, vals))
    ids_equal = bool(torch.equal(ids_f[above], canon[above]))
    return {"scores_equal": scores_equal, "ids_equal_above_kth_score": ids_equal,
            "positions_compared": int(above.sum()), "raw_id_positions_differing": int((ids_f != idx).sum()),
            "ok": scores_equal and ids_equal}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("topk_large_bench.py measures on the GPU: no CUDA device")
    from kge_helpers import make_product_model

    dev = torch.device("cuda")
    out = {"script": "scripts/topk_large_bench.py", "gpu": gpu_info(), "torch": torch.__version__,
           "shape": {"items": I, "d": D, "history_per_user": HIST, "block_users": N_BLOCK, "dense_users": N_DENSE,
                     "k": list(KS), "seed": 2024},
           "l2": "entity table L2-resident across calls (not flushed)", "steps": args.steps, "warmup": args.warmup,
           "results": {}}
    for name in ("DistMult", "ComplEx"):
        m = make_product_model(name, N_BLOCK + 1, I, I, 3, D, device=dev, seed=2024)
        rng = np.random.default_rng(2024)
        users = torch.arange(1, N_BLOCK + 1, device=dev)
        hist = np.sort(rng.integers(1, I, (N_BLOCK, HIST)), axis=1)
        ho = torch.arange(0, HIST * N_BLOCK + 1, HIST, dtype=torch.long, device=dev)
        hi = torch.from_numpy(hist.reshape(-1)).to(dev)
        nd = N_DENSE
        hist_rows = torch.arange(nd, device=dev).repeat_interleave(HIST)
        hist_cols = hi[: nd * HIST]
        res = {}
        for k in KS:
            fused = rate(timed(lambda: m.full_sort_topk(users, k, ho, hi, return_scores=False, path="cuda"),
                               args.steps, args.warmup), N_BLOCK)
            dense = rate(timed(lambda: dense_topk(m, users[:nd], hist_rows, hist_cols, k), args.steps, 1), nd)
            ids_f, sc_f = m.full_sort_topk(users[:nd], k, ho[: nd + 1], hi, path="cuda")
            res[f"k{k}"] = {"a_full_sort_topk_cuda": fused, "b_dense_predict_mask_topk": dict(dense, note=f"measured on {nd} users"),
                            "a_speedup_over_b_per_user": fused["users_per_s_median"] / dense["users_per_s_median"],
                            "check_common_users": dict(compare(ids_f, sc_f, dense_topk(m, users[:nd], hist_rows,
                                                                                     hist_cols, k)), users=nd)}
        base = res["k128"]["a_full_sort_topk_cuda"]["ms_per_call_median"]
        for k in KS[1:]:
            res[f"k{k}"]["a_time_over_k128"] = res[f"k{k}"]["a_full_sort_topk_cuda"]["ms_per_call_median"] / base
        out["results"][name] = res
        del m
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
