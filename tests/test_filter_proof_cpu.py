"""The argument behind the tensor-core full-sort filter (csrc/mma_topk.cu, DESIGN.md 3.4), checked in numpy.

The CUDA path reports exact fp32 scores; the fp16 tensor-core sweep only decides which targets get re-scored.
This file restates that decision rule on the CPU -- operands scaled by powers of two and rounded to fp16, chunk /
group maxima, the running threshold thr = tau - 2 eps with tau = k-th largest chunk maximum among chunks without
masked targets, list compaction when a 128-entry list fills -- and checks on random, heavy-tailed, near-tie and
ADVERSARIALLY ROUNDED data that
  (1) |a^ - S a| <= eps_i = row_eps(...) for every pair (the bound of csrc/mma_topk.cu, restated below), and
  (2) every member of the exact top-k (unmasked targets, score desc / id asc) sits in a group the rule keeps,
      or the row is flagged for the exact path.
Round 1 used bf16 operands with eps = 1.02 * 2^-8 |q| max|t|, which is too small by 2x when the two roundings
of a product line up (test_half_ulp_adversary holds the counter-example: it violates the old bound and must
satisfy the new one).  It does not run the CUDA code (the -m gpu tests compare that with the fp32 kernel bit for
bit); it guards the rule itself against a change that would make the filter lossy.
"""

import numpy as np
import pytest
import torch

CH, GRP, CAND, ROOM = 32, 4, 128, 16


def _f16(x):
    return np.ascontiguousarray(x, dtype=np.float32).astype(np.float16).astype(np.float32)


def _bf16(x):
    return torch.from_numpy(np.ascontiguousarray(x, dtype=np.float32)).to(torch.bfloat16).to(torch.float32).numpy()


def _exp_for(maxabs):
    """e with maxabs * 2^e in [2^7, 2^8) (csrc/mma_topk.cu img_scale / the sweep's per-row scale)."""
    return 0 if maxabs <= 0 else int(np.clip(7 - int(np.floor(np.log2(maxabs))), -60, 60))


def row_eps(nqs, tms, kp, c, chain, last):
    """csrc/mma_topk.cu row_eps(), term by term.  chain: the magnitude of the exact fp32 chain's terms; last: RotatE's
    S |margin| (|q| + tmax), for the rounding of margin - sqrtf(acc) (both 0 for the fp16 sweep's own error)."""
    e = (2.0 ** -10 + 2.0 ** -20) * nqs * tms
    e += 2.0 ** -14 * np.sqrt(kp) * (nqs + tms) * 1.001
    e += kp * 2.0 ** -28
    e += kp * 2.0 ** -22 * (nqs * tms * 1.001 + 256.0 * c)
    e += 3.0 * 2.0 ** -14 * c
    e += (kp + 2) * 2.0 ** -24 * chain
    e += 2.0 ** -23 * last
    return e * 1.01


def sweep_operands(Q, T, dist, margin=0.0, sweep_only=False):
    """What the image kernel and the sweep's setup build: scaled fp16 operands, per-row scale S_i and eps_i.
    Returns (ahat [rows, n] fp32 in scaled units, S [rows], eps [rows] scaled).  margin: RotatE's (0 for the other
    models); sweep_only: eps without the rescore's terms (chain and last), i.e. the bound of |a^ - S a| alone.  A row the fp16 scaling cannot hold
    (a non-finite |q|^2, or an L2 row whose c_i = 2^e_c is no normal fp16 number) gets eps = inf and a nan ahat row:
    the kernel flags it for the exact path."""
    d = T.shape[1]
    kd = d + (3 if dist else 0)
    kp = (kd + 15) // 16 * 16
    tn2 = (T.astype(np.float32) ** 2).sum(1, dtype=np.float32)
    tmax = np.float32(np.sqrt(tn2.max())) * np.float32(1.0001)
    e_t = _exp_for(np.abs(T).max())
    e_w = _exp_for(0.5 * tn2.max())
    Th = _f16(np.ldexp(T.astype(np.float32), e_t))
    if dist:
        W = np.ldexp(np.float32(-0.5) * tn2, e_w).astype(np.float32)
        with np.errstate(over="ignore", invalid="ignore"):   # (|t|^2 / 2 > 2^68: e_w is clamped, W overflows fp16)
            hi = _f16(W)
            mid = _f16(W - hi)
            lo = _f16(W - hi - mid)
    ahat, S, eps = [], [], []
    for q in Q:
        with np.errstate(over="ignore", invalid="ignore"):
            bad = not np.isfinite((q.astype(np.float32) ** 2).sum(dtype=np.float32))
            e_i = _exp_for(np.abs(q).max()) if not bad else 0
        e_c = 0
        if dist:
            e_c = e_i + e_t - e_w
            if e_c > 15:
                e_i -= e_c - 15
                e_c = 15
            bad = bad or e_c < -14 or e_i < -60
        S.append(2.0 ** (e_i + e_t))
        if bad:
            ahat.append(np.full(len(T), np.nan, dtype=np.float32))
            eps.append(np.inf)
            continue
        qh = _f16(np.ldexp(q.astype(np.float32), e_i))
        row = (qh[None, :].astype(np.float64) @ Th.astype(np.float64).T)[0]
        if dist:
            c = np.float64(2.0 ** e_c)
            with np.errstate(invalid="ignore"):
                row = row + c * (hi.astype(np.float64) + mid + lo)
        ahat.append(row.astype(np.float32))          # (fp32 accumulation: the bound has a term for it)
        nq = np.sqrt((q.astype(np.float64) ** 2).sum()) * 1.0001
        nqs, tms = nq * 2.0 ** e_i, float(tmax) * 2.0 ** e_t
        qt_i = nqs + float(tmax) * 2.0 ** e_i
        chain = 0.5 * qt_i * (nq * 2.0 ** e_t + tms) if dist else nqs * tms
        last = abs(margin) * qt_i * 2.0 ** e_t
        if sweep_only:
            chain = last = 0.0
        eps.append(row_eps(nqs, tms, kp, 2.0 ** e_c if dist else 0.0, chain, last))
    return np.stack(ahat), np.array(S), np.array(eps)


def _filter_row(ahat, eps, k, masked, trig=CAND - 5, lists=None, stats=None):
    """One row of the sweep and of the rescore's selection: returns (set of kept (chunk, group) pairs, flagged).

    `lists` = the row's candidate lists, one per (target split, column slice): each a sequence of tiles, each tile the
    ids of the chunks the list sees in it (a list is checked for compaction at the end of every tile).  Default: one
    list of every chunk, four chunks per tile.  `stats`, when given, receives what the rescore kernel sees: E (entries
    of all lists), groups (groups it scores), tau and thr (its final threshold, scaled units)."""
    n = len(ahat)
    n_chunks = (n + CH - 1) // CH
    if lists is None:
        lists = [[tuple(range(c, min(c + 4, n_chunks))) for c in range(0, n_chunks, 4)]]
    top = max(c for lst in lists for tile in lst for c in tile) + 1
    pad = np.full(max(top, n_chunks) * CH, 0.0, dtype=np.float32)   # the image pads the last tile with zero rows
    pad[:n] = ahat
    unsafe = np.zeros(len(pad) // CH, dtype=bool)
    for j in np.nonzero(masked)[0]:
        unsafe[j // CH] = True
    if n % CH:
        unsafe[n // CH:] = True
    unsafe[n_chunks:] = True
    entries, thr0 = [], -np.inf      # entry = (chunk max, chunk id, group mask, unsafe)

    def compact(entries):
        safe = sorted((e[0] for e in entries if not e[3]), reverse=True)
        tau = safe[k - 1] if len(safe) >= k else -np.inf
        new_thr = np.float32(tau) - np.float32(2.0) * np.float32(eps)
        return [e for e in entries if e[0] >= new_thr], new_thr

    for lst in lists:
        mine, thr = [], -np.inf
        for tile in lst:
            for c in tile:
                gm = pad[c * CH:(c + 1) * CH].reshape(CH // GRP, GRP).max(axis=1)
                tm = gm.max()
                if tm >= thr:
                    mine.append((tm, c, gm >= thr, bool(unsafe[c])))
            if len(mine) > trig:
                mine, thr = compact(mine)
                if len(mine) > CAND - ROOM:
                    return set(), True
        entries += mine
        thr0 = max(thr0, thr)
    # re-score side: final tau over everything that clears every list's threshold, then the groups of the survivors
    safe = sorted((e[0] for e in entries if not e[3] and e[0] >= thr0), reverse=True)
    tau = safe[k - 1] if len(safe) >= k else -np.inf
    final_thr = max(thr0, np.float32(tau) - np.float32(2.0) * np.float32(eps))
    kept = {(e[1], g) for e in entries if e[0] >= final_thr for g in np.nonzero(e[2])[0]}
    if stats is not None:
        stats.update(E=len(entries), groups=len(kept), tau=tau, thr=final_thr)
    return kept, False


# enough targets for several compactions per row (a list fills after 123 appended chunks of 32 targets)
CASES = [("normal", 64, 20000), ("heavy_tail", 64, 20000), ("near_ties", 32, 12000), ("dist", 100, 16000),
         ("tiny", 16, 700)]


@pytest.mark.parametrize("kind,d,n", CASES)
def test_filter_keeps_the_exact_topk(kind, d, n):
    rng = np.random.default_rng(sum(map(ord, kind)))   # (hash() is salted per process)
    rows, k = 12, 20
    T = rng.standard_normal((n, d)).astype(np.float32) * np.float32(0.1)
    Q = rng.standard_normal((rows, d)).astype(np.float32) * np.float32(0.1)
    if kind == "heavy_tail":
        T[rng.integers(0, n, 30)] *= 3.0     # (x25 makes eps swallow the score spread: every row is flagged)
        T[rng.integers(0, n, 10)] *= -4.0
    if kind == "near_ties":          # 64 targets within a few bf16 ulps of each other at the top, spread over chunks
        base = rng.standard_normal(d).astype(np.float32)
        idx = rng.choice(n, 64, replace=False)
        T[idx] = base + rng.standard_normal((64, d)).astype(np.float32) * np.float32(1e-4)
        Q[:] = base * np.float32(0.5) + Q * np.float32(0.01)
    dist = kind == "dist"
    a = Q.astype(np.float64) @ T.astype(np.float64).T
    if dist:                          # -|q - t|^2 = 2 (q.t - |t|^2 / 2) - |q|^2: the sweep ranks q.t - |t|^2 / 2
        a = a - 0.5 * (T.astype(np.float64) ** 2).sum(1)[None, :]
    ahat, S, eps_all = sweep_operands(Q, T, dist)
    for i in range(rows):
        eps = eps_all[i]
        assert np.abs(ahat[i].astype(np.float64) - S[i] * a[i]).max() <= eps, "error bound violated"
        masked = np.zeros(n, dtype=bool)
        masked[0] = True                                     # the [PAD] target
        masked[rng.integers(1, n, int(rng.integers(0, 60)))] = True   # history
        kept, flagged = _filter_row(ahat[i], eps, k, masked)
        if flagged:
            continue                                         # the row goes to the exact fp32 kernel
        valid = np.nonzero(~masked)[0]
        order = valid[np.lexsort((valid, -a[i, valid]))][:k]  # exact top-k: score desc, id asc
        for j in order:
            assert (j // CH, (j % CH) // GRP) in kept, f"row {i}: exact top-k member {j} was filtered out"


def test_half_ulp_adversary():
    """Every element sits half an ulp above a representable value, so both roundings of every product go the same
    way.  bf16: q = t = (1 + 2^-8) * ones(64) rounds to ones, |a^ - a| = 0.50 > round 1's eps = 0.257 (the bug);
    fp16 with the bound of row_eps: the same construction at fp16's half ulp stays inside eps."""
    d = 64
    q = np.full(d, 1.0 + 2.0 ** -8, dtype=np.float32)
    a = float(q.astype(np.float64) @ q.astype(np.float64))
    ahat_bf16 = float(_bf16(q).astype(np.float64) @ _bf16(q).astype(np.float64))
    old_eps = 1.02 * 2.0 ** -8 * np.sqrt(a) * np.sqrt(a) * 1.0001
    assert abs(ahat_bf16 - a) > old_eps                      # round 1's bound does not hold
    assert abs(ahat_bf16 - a) <= (2.0 ** -7 + 2.0 ** -16) * a   # the valid bf16 bound is twice as wide
    for half_ulp, sign in ((2.0 ** -11, 1.0), (2.0 ** -11, -1.0)):
        # fp16 has 11 significant bits: 1 + 2^-11 is a tie that rounds to even (1.0); 1 - 2^-12 ties to 1.0 as well
        x = np.float32(1.0 + half_ulp) if sign > 0 else np.float32(1.0 - half_ulp / 2)
        Q = np.full((1, d), x, dtype=np.float32)
        T = np.full((40, d), x, dtype=np.float32)
        T[1::2] *= np.float32(0.5)                           # different norms, same rounding direction
        exact = Q.astype(np.float64) @ T.astype(np.float64).T
        ahat, S, eps = sweep_operands(Q, T, dist=False)
        err = np.abs(ahat[0].astype(np.float64) - S[0] * exact[0]).max()
        assert err <= eps[0]
        assert err >= 0.45 * eps[0], "the adversary should come close to the bound (the bound is tight)"
    # the L2 form: a = q.t - |t|^2 / 2 with the hi/mid/lo split of the norm term
    rng = np.random.default_rng(5)
    T = (np.float32(1.0 + 2.0 ** -11) * np.sign(rng.standard_normal((64, d)))).astype(np.float32)
    Q = T[:4].copy()
    exact = Q.astype(np.float64) @ T.astype(np.float64).T - 0.5 * (T.astype(np.float64) ** 2).sum(1)[None, :]
    ahat, S, eps = sweep_operands(Q, T, dist=True)
    for i in range(4):
        assert np.abs(ahat[i].astype(np.float64) - S[i] * exact[i]).max() <= eps[i]


def test_tiny_and_huge_magnitudes_stay_inside_the_bound():
    """Power-of-two scaling keeps the operands in fp16's normal range whatever the tables' magnitude; rows with
    elements far below the row maximum fall into the subnormal range, which the bound's absolute term covers."""
    rng = np.random.default_rng(9)
    for scale_q, scale_t in ((1e-6, 1e-6), (1e3, 1e-4), (1e-5, 50.0)):
        T = (rng.standard_normal((500, 48)) * scale_t).astype(np.float32)
        Q = (rng.standard_normal((6, 48)) * scale_q).astype(np.float32)
        Q[:, ::3] *= np.float32(1e-6)                        # subnormal after scaling
        T[:, 1::4] *= np.float32(1e-7)
        for dist in (False, True):
            if dist and scale_q / scale_t > 1e5:
                continue                                      # c_i leaves fp16's range: the kernel flags such rows
            exact = Q.astype(np.float64) @ T.astype(np.float64).T
            if dist:
                exact = exact - 0.5 * (T.astype(np.float64) ** 2).sum(1)[None, :]
            ahat, S, eps = sweep_operands(Q, T, dist)
            for i in range(len(Q)):
                assert np.abs(ahat[i].astype(np.float64) - S[i] * exact[i]).max() <= eps[i]


def test_rows_with_fewer_than_k_valid_targets_never_get_a_threshold():
    """With fewer than k chunks free of masked targets tau stays -inf: nothing is ever dropped."""
    rng = np.random.default_rng(3)
    n, k = 640, 20
    ahat = rng.standard_normal(n).astype(np.float32)
    masked = np.ones(n, dtype=bool)
    masked[rng.integers(1, n, 12)] = False                  # 12 valid targets only
    kept, flagged = _filter_row(ahat, 1e-3, k, masked)
    assert flagged or all((j // CH, (j % CH) // GRP) in kept for j in np.nonzero(~masked)[0])
