"""Sampled evaluation (eval_args.mode uni100) over candidate lists against the dense route; prints one JSON line.

DistMult and ComplEx, d = 64, 200,001 items, 1-5 positives per user, 100 uniform negatives per positive (the
candidate rows hopwise's NegSampleEvalDataLoader emits: a user's positives, then its negatives), seed 2024.  Legs:
  (a) fused: kge_predict on the candidate rows, then kge_candidate_select (top-20 ids and the rank counts GAUC
      reads), one call over a block of 20,000 users; reported whole and split into its two kernels;
  (b) dense, top-k only: per loader batch of 40 users (eval_batch_size 4096 at ~3 x 101 rows per user) predict,
      torch.full(-inf) over [40, 200,001], the scatter, torch.topk, the int pos_matrix and the gather -- what
      trainer.py's _neg_sample_batch_eval and the collector's rec.topk branch run;
  (c) dense with GAUC: (b) plus the collector's rec.meanrank branch (a full sort of every row and _average_rank).
Each leg is reported in users/s (mean and median over the timed calls, after warm-up).  The entity table (51 MB for
DistMult, 102 MB for ComplEx) fits the 126 MB L2 and is not flushed between calls.  The candidate columns are on the
device before the timed window (the loader's host collation is not part of any leg).  The script checks that (a) and
(c) give the same rec.topk and rec.meanrank rows on the users they share.  The card's name, power limit and top SM
clock are read in the same run (an nvidia-smi query).

    python scripts/sampled_eval_bench.py [--steps 10] [--warmup 2] [--out FILE]
"""

import argparse
import ctypes as C
import json
import os
import sys

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "scripts")]

import numpy as np  # noqa: E402
import torch  # noqa: E402

from rank_bench import average_rank, gpu_info, rate, timed  # noqa: E402

N_FUSED, N_DENSE, BATCH_USERS, I, D, K, NEG = 20_000, 1_000, 40, 200_001, 64, 20, 100


def candidates(rng, n):
    """Per user 1-5 positives then NEG uniform negatives per positive (ids in [1, I)), as the loader lays them out."""
    n_pos = rng.integers(1, 6, n)
    pos = [rng.choice(np.arange(1, I), p, replace=False) for p in n_pos]
    rows = [np.concatenate([p, rng.integers(1, I, len(p) * NEG)]) for p in pos]
    lens = np.array([len(r) for r in rows])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.int64)
    return np.concatenate(rows), off, pos


def dense_batch(m, uc, ic, row, pu, pi, n, gauc):
    """trainer.py _neg_sample_batch_eval + collector.py rec.topk (and rec.meanrank) for one loader batch."""
    scores = m.predict({"user_id": uc, "item_id": ic})
    dense = torch.full((n, I), -torch.inf, device=uc.device)
    dense[row, ic] = scores
    _, topk_idx = torch.topk(dense, K, dim=-1)
    pos_matrix = torch.zeros_like(dense, dtype=torch.int)
    pos_matrix[pu, pi] = 1
    pos_len = pos_matrix.sum(dim=1, keepdim=True)
    rec = torch.cat([torch.gather(pos_matrix, dim=1, index=topk_idx), pos_len], dim=1)
    if not gauc:
        return rec, None
    srt, idx = torch.sort(dense, dim=-1, descending=True)
    pos_index = torch.gather(pos_matrix, dim=1, index=idx)
    avg = average_rank(srt)
    rank_sum = torch.where(pos_index == 1, avg, torch.zeros_like(avg)).sum(dim=-1, keepdim=True)
    user_len = srt.argmin(dim=1, keepdim=True)
    return rec, torch.cat([rank_sum, user_len.to(rank_sum.dtype), pos_len.to(rank_sum.dtype)], dim=1).float()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("sampled_eval_bench.py measures on the GPU: no CUDA device")
    from kge_helpers import make_product_model

    from hopwise_b200 import _abi
    from hopwise_b200.evaluator import gauc_from_sums, gauc_sums, topk_hits

    dev = torch.device("cuda")
    out = {"script": "scripts/sampled_eval_bench.py", "gpu": gpu_info(), "torch": torch.__version__,
           "shape": {"items": I, "d": D, "positives_per_user": "1-5", "negatives_per_positive": NEG,
                     "fused_block_users": N_FUSED, "dense_users": N_DENSE, "dense_batch_users": BATCH_USERS,
                     "topk_k": K, "seed": 2024},
           "l2": "entity table L2-resident across calls (not flushed)", "steps": args.steps, "warmup": args.warmup,
           "results": {}}
    lib = _abi.lib()
    for name in ("DistMult", "ComplEx"):
        m = make_product_model(name, N_FUSED + 1, I, I, 3, D, device=dev, seed=2024)
        rng = np.random.default_rng(2024)
        items, off, pos = candidates(rng, N_FUSED)
        lens = np.diff(off)
        ic = torch.from_numpy(items).to(dev)
        uc = torch.from_numpy(np.repeat(np.arange(1, N_FUSED + 1), lens)).to(dev)
        off_d = torch.from_numpy(off).to(dev)
        po_h = np.concatenate([[0], np.cumsum([len(p) for p in pos])]).astype(np.int64)
        po = torch.from_numpy(po_h).to(dev)
        pi = torch.from_numpy(np.concatenate([np.sort(p) for p in pos])).to(dev)
        n_cand = int(off[-1])

        def fused():
            ids, _, g, e, nu = m._candidate_select(uc, ic, off_d, K, True, False, po, pi)
            return topk_hits(ids, po, pi), m._meanrank_rows(g, e, nu, po, pi)

        leg_a = timed(fused, args.steps, args.warmup)
        leg_predict = timed(lambda: m.predict({"user_id": uc, "item_id": ic}), args.steps, args.warmup)
        scores = m.predict({"user_id": uc, "item_id": ic})
        ids = torch.empty(N_FUSED, K, dtype=torch.int64, device=dev)
        g = torch.empty(pi.numel(), dtype=torch.int64, device=dev)
        e, nu = torch.empty_like(g), torch.empty(N_FUSED, dtype=torch.int64, device=dev)
        ws = torch.empty(lib.kge_candidate_select_workspace_bytes(N_FUSED, n_cand), dtype=torch.uint8, device=dev)

        def select():
            _abi.check(lib.kge_candidate_select(scores.data_ptr(), ic.data_ptr(), n_cand, off_d.data_ptr(), N_FUSED,
                                                I, po.data_ptr(), pi.data_ptr(), K, ids.data_ptr(), None,
                                                g.data_ptr(), e.data_ptr(), nu.data_ptr(), ws.data_ptr(), ws.numel(),
                                                _abi.stream_ptr()), "kge_candidate_select")

        leg_select = timed(select, args.steps, args.warmup)
        # the dense route on the first N_DENSE users, in loader batches
        batches = []
        for s in range(0, N_DENSE, BATCH_USERS):
            e_ = min(N_DENSE, s + BATCH_USERS)
            c0, c1 = int(off[s]), int(off[e_])
            row = torch.from_numpy(np.repeat(np.arange(e_ - s), lens[s:e_])).to(dev)
            pu = torch.from_numpy(np.repeat(np.arange(e_ - s), [len(p) for p in pos[s:e_]])).to(dev)
            pb = torch.from_numpy(np.concatenate(pos[s:e_])).to(dev)
            batches.append((uc[c0:c1], ic[c0:c1], row, pu, pb, e_ - s))

        def dense(gauc):
            return [dense_batch(m, *b, gauc) for b in batches]

        reps = max(2, args.steps // 2)
        leg_b = timed(lambda: dense(False), reps, 1)
        leg_c = timed(lambda: dense(True), reps, 1)
        rec_f, mr_f = fused()
        got = dense(True)
        rec_d, mr_d = torch.cat([x[0] for x in got]), torch.cat([x[1] for x in got])
        ra, rc = rate(leg_a, N_FUSED), rate(leg_c, N_DENSE)
        rp, rs = rate(leg_predict, N_FUSED), rate(leg_select, N_FUSED)
        out["results"][name] = {
            "candidates": n_cand, "max_row": int(lens.max()),
            "a_fused_predict_select": ra,
            "a_split": {"kge_predict": rp, "kge_candidate_select": rs,
                        "select_share_of_median": rs["ms_per_call_median"] / (rp["ms_per_call_median"]
                                                                              + rs["ms_per_call_median"])},
            "b_dense_topk": dict(rate(leg_b, N_DENSE), note=f"measured on {N_DENSE} users in batches of {BATCH_USERS}"),
            "c_dense_topk_gauc": dict(rc, note=f"measured on {N_DENSE} users in batches of {BATCH_USERS}"),
            "a_speedup_over_c_per_user": ra["users_per_s_median"] / rc["users_per_s_median"],
            "check_common_users": {"users": N_DENSE, "rec_topk_equal": bool(torch.equal(rec_f[:N_DENSE], rec_d)),
                                   "meanrank_rows_equal": bool(torch.equal(mr_f[:N_DENSE], mr_d)),
                                   "gauc_fused": gauc_from_sums(gauc_sums(mr_f[:N_DENSE]), None),
                                   "gauc_dense": gauc_from_sums(gauc_sums(mr_d), None)},
        }
        del m, batches
        torch.cuda.empty_cache()
    line = json.dumps(out)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
