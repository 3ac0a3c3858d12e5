"""GAUC's rank counts at the BASELINE config 4 shape; prints one JSON line.

DistMult and ComplEx, d = 64, 200,001 items, 50 history items per user, 1-5 positives per user, seed 2024.  Legs:
  (a) model.full_sort_meanrank on a block of 75,776 users (one wave of the tensor-core top-k sweep);
  (b) model.full_sort_topk(k=20, path="cuda") on the same block: the same CUDA-core sweep with the top-k epilogue;
  (c) the dense route (a) replaces, on 2,048 users: full_sort_predict, the trainer's masking, then the collector's
      sort and average rank (torch on the GPU), as hopwise's trainer and collector run it.
Each leg is reported in users/s (mean and median over the timed calls, after warm-up).  The entity table (51 MB for
DistMult, 102 MB for ComplEx) fits the 126 MB L2 and is not flushed between calls: every leg reads it warm.
Two placements of the positives: uniformly random under the xavier initialisation (the rank epilogue's worst case:
positives rank anywhere, so most targets score above a row's lowest positive), and drawn from each user's own top 50.
The script checks that (a) and (c) give the same rec.meanrank rows and GAUC on the users they share.  The card's name,
power limit and top SM clock are read in the same run (an nvidia-smi query).

    python scripts/rank_bench.py [--steps 10] [--warmup 2]
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

N_BLOCK, N_DENSE, I, HIST, D, K = 75_776, 2_048, 200_001, 50, 64, 20


def gpu_info():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True, check=True).stdout.strip().splitlines()[0]
    name, power, clock = (x.strip() for x in out.split(","))
    return {"name": name, "power_limit": power, "clocks_max_sm": clock}


def average_rank(scores):
    """The collector's _average_rank on rows sorted descending: ties share the mean of their positions."""
    length, width = scores.shape
    true_col = torch.full((length, 1), True, dtype=torch.bool, device=scores.device)
    obs = torch.cat([true_col, scores[:, 1:] != scores[:, :-1]], dim=1)
    bias = torch.arange(0, length, device=scores.device).repeat(width).reshape(width, -1).transpose(1, 0).reshape(-1)
    dense = obs.view(-1).cumsum(0) + bias
    count = torch.where(torch.cat([obs, true_col], dim=1))[1]
    return 0.5 * (count[dense] + count[dense - 1] + 1).view(length, -1)


def dense_meanrank(m, users, hist_rows, hist_cols, pos_rows, pos_cols):
    """trainer.py's _full_sort_batch_eval masking + the collector's rec.meanrank branch, on dense rows."""
    scores = m.full_sort_predict({"user_id": users})
    scores[:, 0] = -torch.inf
    scores[hist_rows, hist_cols] = -torch.inf
    srt, idx = torch.sort(scores, dim=-1, descending=True)
    pos_matrix = torch.zeros_like(scores, dtype=torch.int)
    pos_matrix[pos_rows, pos_cols] = 1
    pos_index = torch.gather(pos_matrix, dim=1, index=idx)
    avg_rank = average_rank(srt)
    pos_rank_sum = torch.where(pos_index == 1, avg_rank, torch.zeros_like(avg_rank)).sum(dim=-1, keepdim=True)
    user_len = srt.argmin(dim=1, keepdim=True)
    pos_len = pos_matrix.sum(dim=1, keepdim=True)
    return torch.cat([pos_rank_sum, user_len.to(pos_rank_sum.dtype), pos_len.to(pos_rank_sum.dtype)], dim=1).float()


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


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("rank_bench.py measures on the GPU: no CUDA device")
    from kge_helpers import make_product_model

    from hopwise_b200.evaluator import gauc_from_sums, gauc_sums

    dev = torch.device("cuda")
    out = {"script": "scripts/rank_bench.py", "gpu": gpu_info(), "torch": torch.__version__,
           "shape": {"items": I, "d": D, "history_per_user": HIST, "positives_per_user": "1-5", "block_users": N_BLOCK,
                     "dense_users": N_DENSE, "topk_k": K, "seed": 2024},
           "l2": "entity table L2-resident across calls (not flushed)", "steps": args.steps, "warmup": args.warmup,
           "results": {}}
    for name in ("DistMult", "ComplEx"):
        m = make_product_model(name, N_BLOCK + 1, I, I, 3, D, device=dev, seed=2024)
        rng = np.random.default_rng(2024)
        users = torch.arange(1, N_BLOCK + 1, device=dev)
        hist = np.sort(rng.integers(1, I, (N_BLOCK, HIST)), axis=1)
        ho = torch.arange(0, HIST * N_BLOCK + 1, HIST, dtype=torch.long, device=dev)
        hi = torch.from_numpy(hist.reshape(-1)).to(dev)
        n_pos = rng.integers(1, 6, N_BLOCK)
        po = torch.from_numpy(np.concatenate([[0], np.cumsum(n_pos)])).to(dev)
        top50, _ = m.full_sort_topk(users, 50, ho, hi, return_scores=False, path="cuda")
        top50 = top50.cpu().numpy()
        res = {}
        for placement in ("uniform", "own_top50"):
            if placement == "uniform":
                rows = [np.sort(rng.choice(np.arange(1, I), k, replace=False)) for k in n_pos]
            else:
                rows = [np.sort(rng.choice(top50[u], k, replace=False)) for u, k in enumerate(n_pos)]
            pi = torch.from_numpy(np.concatenate(rows)).to(dev)
            leg_a = timed(lambda: m.full_sort_meanrank(users, po, pi, ho, hi), args.steps, args.warmup)
            leg_b = timed(lambda: m.full_sort_topk(users, K, ho, hi, return_scores=False, path="cuda"),
                          args.steps, args.warmup)
            nd = N_DENSE
            hist_rows = torch.arange(nd, device=dev).repeat_interleave(HIST)
            hist_cols = hi[: nd * HIST]
            pos_rows = torch.arange(nd, device=dev).repeat_interleave(torch.from_numpy(n_pos[:nd]).to(dev))
            pos_cols = pi[: int(po[nd].item())]
            leg_c = timed(lambda: dense_meanrank(m, users[:nd], hist_rows, hist_cols, pos_rows, pos_cols),
                          max(2, args.steps // 2), 1)
            # (a) and (c) on the users they share
            fused = m.full_sort_meanrank(users, po, pi, ho, hi)[:nd]
            dense = dense_meanrank(m, users[:nd], hist_rows, hist_cols, pos_rows, pos_cols)
            g_fused = gauc_from_sums(gauc_sums(fused), None)
            g_dense = gauc_from_sums(gauc_sums(dense), None)
            ra, rb, rc = rate(leg_a, N_BLOCK), rate(leg_b, N_BLOCK), rate(leg_c, nd)
            res[placement] = {
                "a_full_sort_meanrank": ra, "b_full_sort_topk_cuda": rb,
                "c_dense_sort_average_rank": dict(rc, note=f"measured on {nd} users"),
                "a_over_b_time": ra["ms_per_call_median"] / rb["ms_per_call_median"],
                "a_speedup_over_c_per_user": ra["users_per_s_median"] / rc["users_per_s_median"],
                "check_common_users": {"users": nd, "meanrank_rows_equal": bool(torch.equal(fused, dense)),
                                       "max_abs_row_diff": float((fused - dense).abs().max()),
                                       "gauc_fused": g_fused, "gauc_dense": g_dense,
                                       "gauc_abs_diff": abs(g_fused - g_dense)},
            }
        out["results"][name] = res
        del m
        torch.cuda.empty_cache()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
