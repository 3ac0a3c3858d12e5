"""Adversarial tables for the tensor-core full-sort filter (csrc/mma_topk.cu) and the regime each one reaches.

Every case is a set of query rows Q (what the sweep's query_value yields: the product model gets identity relation
rows, so Q is the head table itself) and target rows T, one float32 row per target with the parts of ComplEx / RotatE
side by side.  `simulate` runs the numpy restatement of tests/test_filter_proof_cpu.py (scaled fp16 operands, row_eps,
the per-list sweep with its compactions, the rescore's selection) over the row's lists as plan_mma lays them out, and
says per row whether the kernel flags it and why:
  "bad"       the fp16 scaling cannot hold the row (non-finite |q|^2, or c_i = 2^e_c outside fp16's normal range)
  "overflow"  a candidate list could not be compacted (cand_cnt = -1)
  "few"       fewer than k exactly scored targets clear the rescore's pre-filter (n_pass < k)
and, for the rows it does not flag, what the rescore kernel sees (entries, groups, passing keys) and whether the fp16
order is wrong at the k-th place (the filter, not the approximation, decided the answer).
tests/test_mma_filter_cases_cpu.py asserts that each case reaches the regime it is built for; tests/test_gpu_mma_filter.py
runs the same cases on the device and checks the flagged-row count against `simulate`.
"""

import functools
from dataclasses import dataclass, field

import numpy as np

from test_filter_proof_cpu import CAND, CH, GRP, _filter_row, sweep_operands

N_SMS = 148          # B200
MAX_SPLITS = 4
RS_GIDS = 256
RS_KEYS = 64
MODELS = ("DistMult", "ComplEx", "TransE", "RotatE")
PARTS = {"DistMult": 1, "ComplEx": 2, "TransE": 1, "RotatE": 2}
DIST = {"DistMult": False, "ComplEx": False, "TransE": True, "RotatE": True}


def plan(model, d, n, n_targets, cfg="", n_sms=N_SMS):
    """csrc/mma_topk.cu plan_mma: sweep shape, tile width, column slices and target splits."""
    parts, dist = PARTS[model], DIST[model]
    kp = (parts * d + (3 if dist else 0) + 15) // 16 * 16
    assert kp <= 640
    two, one = 112 * 1024, 200 * 1024
    fixed2 = 128 * 2 * kp * 2 + 32 * 8 + 2 * 128 * 2 * 4 + 64
    c = cfg
    if c == "a" and fixed2 + 2 * 128 * kp * 2 > two:
        c = ""
    if c == "f" and fixed2 + 2 * 128 * kp * 2 > one:
        c = ""
    if c == "c" and fixed2 + 2 * 64 * kp * 2 > one:
        c = ""
    if not c:
        if fixed2 + 3 * 128 * kp * 2 <= two:
            c = "a"
        elif fixed2 + 2 * 128 * kp * 2 <= one:
            c = "f"
        else:
            c = "c" if fixed2 + 2 * 64 * kp * 2 <= one else "k"
    nh = 1 if c == "k" else 2
    tn = 64 if c == "c" else 128
    ncol = 2 if c in "fk" else 1
    n_tiles = (n_targets + tn - 1) // tn
    mm = 128 * nh
    row_blocks = max((n + mm - 1) // mm, 1)
    s = max(min(n_sms * (2 if c == "a" else 1) // row_blocks, MAX_SPLITS, n_tiles // 16), 1)
    tps = (n_tiles + s - 1) // s
    splits = (n_tiles + tps - 1) // tps
    nent = max(splits * ncol * CAND, RS_GIDS)
    return dict(cfg=c, kp=kp, tn=tn, ncol=ncol, nh=nh, n_tiles=n_tiles, splits=splits, tps=tps, nent=nent)


def lists_for(pl):
    """The chunk ids each (target split, column slice) list sees, tile by tile, in sweep order."""
    per_tile = pl["tn"] // CH
    nch = per_tile // pl["ncol"]
    out = []
    for s in range(pl["splits"]):
        tiles = range(s * pl["tps"], min(pl["n_tiles"], (s + 1) * pl["tps"]))
        for cs in range(pl["ncol"]):
            out.append([tuple(t * per_tile + cs * nch + x for x in range(nch)) for t in tiles])
    return out


@dataclass
class Case:
    id: str
    model: str
    k: int
    Q: np.ndarray                  # [n, P] float32
    T: np.ndarray                  # [n_targets, P] float32
    regime: str                    # "filter" | "overflow" | "survivors" | "few" | "bad" | "mixed"
    hist: list = None              # per row: sorted int64 array of masked targets, or None
    mask_pad: bool = True
    kg: bool = False               # rows are (head entity, relation) queries through full_sort_topk_kg
    heads: np.ndarray = None       # kg: entity id of each row (Q = T[heads])
    expect: dict = field(default_factory=dict)   # regime-specific expectations, see test_mma_filter_cases_cpu.py

    @property
    def d(self):
        return self.T.shape[1] // PARTS[self.model]

    @property
    def dist(self):
        return DIST[self.model]

    def masked(self, r):
        m = np.zeros(len(self.T), dtype=bool)
        if self.mask_pad:
            m[0] = True
        if self.hist is not None and len(self.hist[r]):
            m[self.hist[r]] = True
        return m

    def exact(self, Q=None):
        """float64 ranking score (q.t, or q.t - |t|^2 / 2 for the L2 models: the same order as -|q - t|)."""
        Q = self.Q if Q is None else Q
        with np.errstate(invalid="ignore", over="ignore"):
            a = Q.astype(np.float64) @ self.T.astype(np.float64).T
        if self.dist:
            a -= 0.5 * (self.T.astype(np.float64) ** 2).sum(1)[None, :]
        return a


MARGIN = {"RotatE": 1.0}   # the product's default margin; the other scorers report acc or -sqrtf(acc) unshifted


def _fma32(acc, x):
    """fmaf(., ., acc) with the exact product x (float64): the float64 sum rounded to odd, then to float32, is the
    correctly rounded float32 result (float64 carries more than 24 + 2 bits, so the two roundings cannot compound)."""
    a = acc.astype(np.float64)
    s = a + x
    bb = s - a
    err = (a - (s - bb)) + (x - bb)                              # two-sum: s + err == a + x exactly
    odd = (s.view(np.int64) & 1) == 1
    s = np.where((err != 0) & ~odd, np.nextafter(s, np.where(err > 0, np.inf, -np.inf)), s)
    return s.astype(np.float32)


def chain_scores(case, q):
    """The rescore's exact scores of one query row against every target: the CUDA-core kernel's fp32 chain (columns in
    order, one fused multiply-add per column; score = acc, or margin - sqrtf(acc) for the L2 models), emulated exactly
    (fp32 differences and sqrt are correctly rounded in numpy; products of two fp32 are exact in float64)."""
    q32 = q.astype(np.float32)
    acc = np.zeros(len(case.T), dtype=np.float32)
    with np.errstate(over="ignore", invalid="ignore"):
        for c in range(case.T.shape[1]):
            t = case.T[:, c]
            if case.dist:
                x = (q32[c] - t).astype(np.float32).astype(np.float64) ** 2
            else:
                x = t.astype(np.float64) * np.float64(q32[c])
            acc = _fma32(acc, x)
        if case.dist:
            return np.float32(MARGIN.get(case.model, 0.0)) - np.sqrt(acc)
    return acc


def simulate(case, cfg="", n_sms=N_SMS):
    """Per row: {"flag": None | "bad" | "overflow" | "few", "E", "groups", "n_pass", "wrong_order", "kept_all"};
    kept_all: every member of the top-k the kernels report (fp32 chain scores, ties by id) is among the scored targets."""
    n, nt = case.Q.shape[0], case.T.shape[0]
    pl = plan(case.model, case.d, n, nt, cfg, n_sms)
    lists = lists_for(pl)
    uniq, inv = np.unique(case.Q, axis=0, return_inverse=True) if case.hist is None else (case.Q, np.arange(n))
    inv = np.asarray(inv).reshape(-1)
    ahat, S, eps = sweep_operands(uniq, case.T, case.dist, MARGIN.get(case.model, 0.0))
    a_all = case.exact(uniq)
    out_u = []
    for u in range(len(uniq)):
        r = int(np.nonzero(inv == u)[0][0])
        out_u.append(_simulate_row(case, ahat[u], S[u], eps[u], a_all[u], chain_scores(case, uniq[u]), case.masked(r),
                                   lists))
    return [out_u[inv[r]] for r in range(n)], pl


def _simulate_row(case, ahat, S, eps, a, score, masked, lists):
    k = case.k
    res = dict(flag=None, E=0, groups=0, n_pass=0, wrong_order=False, kept_all=True)
    if not np.isfinite(eps):
        res["flag"] = "bad"
        return res
    st = {}
    kept, flagged = _filter_row(ahat, eps, k, masked, lists=lists, stats=st)
    if flagged:
        res["flag"] = "overflow"
        return res
    res.update(E=st["E"], groups=st["groups"])
    nt = len(a)
    scored = np.zeros(nt, dtype=bool)
    for c, g in kept:
        lo = c * CH + g * GRP
        scored[lo:min(lo + GRP, nt)] = True
    scored &= ~masked
    sa = S * a
    if np.isfinite(st["tau"]):
        passing = scored & (sa >= st["tau"] - 1.25 * eps)
    else:
        passing = scored
    res["n_pass"] = int(passing.sum())
    if res["n_pass"] < k:
        res["flag"] = "few"
        return res
    valid = np.nonzero(~masked)[0]
    # members as the kernels rank them (fp32 chain scores, ties by id): those must all have been scored
    res["kept_all"] = bool(scored[valid[np.lexsort((valid, -score[valid]))][:k]].all())
    order = valid[np.lexsort((valid, -a[valid]))]
    members, rest = order[:k], order[k:]
    if len(rest):
        res["wrong_order"] = bool(ahat[members].min() < ahat[rest].max())
    return res


# ---- builders -------------------------------------------------------------------------------------------------------
def _rng(name):
    return np.random.default_rng(sum(map(ord, name)))


def _spread(n_targets, m, rng, per_chunk=1):
    """m target ids spread over the whole range (so over chunks, tiles, target splits and column slices), `per_chunk`
    of them in distinct groups of one chunk."""
    n_chunks = n_targets // CH
    chunks = np.unique(np.linspace(1, n_chunks - 1, (m + per_chunk - 1) // per_chunk).astype(np.int64))
    ids = []
    for c in chunks:
        groups = rng.choice(CH // GRP, per_chunk, replace=False)
        ids += [c * CH + g * GRP + int(rng.integers(0, GRP)) for g in groups]
    return np.array(sorted(ids)[:m], dtype=np.int64)


def _parts_width(model, d):
    return PARTS[model] * d


def _base(model, d, n, n_targets, rng):
    """A direction b every row's query follows (q = b / 2 + noise; q = b + noise for the L2 models, whose score
    q.t - |t|^2 / 2 peaks at t = q) and random targets well below the targets placed near b."""
    P = _parts_width(model, d)
    q_scale = 1.0 if DIST[model] else 0.5
    b = (rng.standard_normal(P) * 0.3).astype(np.float32)
    T = (rng.standard_normal((n_targets, P)) * 0.1).astype(np.float32)
    Q = (b * np.float32(q_scale) + rng.standard_normal((n, P)).astype(np.float32) * np.float32(0.02)).astype(np.float32)
    return b, Q, T


def near_tie(model, k, m, n_targets=20000, n=130, d=None):
    """m targets within ~1e-4 relative of each other at the top of every row, spread over the catalogue."""
    d = d or (64 if PARTS[model] == 1 else 32)
    rng = _rng(f"tie{model}{k}{m}")
    b, Q, T = _base(model, d, n, n_targets, rng)
    idx = _spread(n_targets, m, rng)
    T[idx] = b * (1 + rng.standard_normal((m, len(b))).astype(np.float32) * np.float32(1e-4))
    return Case(f"near_tie-{model}-k{k}-m{m}", model, k, Q, T, "filter")


def norm_tie(model, k, m=None, n_targets=12000, n=160, d=None):
    """L2 models: a cluster with equal q.t for every row whose order only |t|^2 (the hi / mid / lo columns) decides."""
    d = d or (64 if PARTS[model] == 1 else 32)
    m = m or 3 * k
    rng = _rng(f"norm{model}{k}")
    b, _, T = _base(model, d, n, n_targets, rng)
    Q = (b[None, :] * np.linspace(0.4, 0.6, n, dtype=np.float32)[:, None]).astype(np.float32)
    idx = _spread(n_targets, m, rng)
    delta = rng.standard_normal((m, len(b)))
    delta -= np.outer(delta @ b.astype(np.float64), b) / float(b.astype(np.float64) @ b)   # orthogonal to b, so to q
    delta *= (0.01 * np.linalg.norm(b) * np.sqrt(rng.uniform(0.5, 1.0, m)) / np.linalg.norm(delta, axis=1))[:, None]
    T[idx] = (b + delta).astype(np.float32)
    return Case(f"norm_tie-{model}-k{k}", model, k, Q, T, "filter")


def duplicates(model, k, n_targets=20000, n=128):
    """2k exact copies of one row across target splits: the k-th place is a tie, broken by id ascending."""
    d = 64 if PARTS[model] == 1 else 32
    rng = _rng(f"dup{model}{k}")
    b, Q, T = _base(model, d, n, n_targets, rng)
    T[_spread(n_targets, 2 * k + 1, rng)] = b
    return Case(f"duplicates-{model}-k{k}", model, k, Q, T, "filter", expect=dict(tie_at_k=True))


def overflow(model, k, n_zero, n_other=40, n_targets=40000):
    """Rows whose approximate scores are all equal (a zero query; for the L2 models over targets of equal norm): every
    list fills with chunks within eps of the top and cannot be compacted.  Above 1,024 such rows in one call the
    fallback takes its second region."""
    d = 64 if PARTS[model] == 1 else 32
    rng = _rng(f"ovf{model}{k}")
    P = _parts_width(model, d)
    if DIST[model]:
        T = (np.where(rng.random((n_targets, P)) < 0.5, -1.0, 1.0) * 0.125).astype(np.float32)
    else:
        T = (rng.standard_normal((n_targets, P)) * 0.1).astype(np.float32)
    Q = np.zeros((n_zero + n_other, P), dtype=np.float32)
    Q[n_zero:] = rng.standard_normal((n_other, P)) * 0.1
    return Case(f"overflow-{model}-k{k}-rows{n_zero}", model, k, Q, T, "overflow",
                expect=dict(flagged=n_zero))


def survivors(model, k, n_targets=20000, n=64, per_chunk=3, m_chunks=400):
    """A cluster of 400 chunks, three targets each in distinct groups, all within eps of the top: the rescore gets
    more than 256 entries, more groups than one fill holds and more than 64 passing keys, without a list overflow."""
    d = 64 if PARTS[model] == 1 else 32
    rng = _rng(f"surv{model}{k}")
    b, Q, T = _base(model, d, n, n_targets, rng)
    idx = _spread(n_targets, m_chunks * per_chunk, rng, per_chunk)
    T[idx] = b * (1 + rng.standard_normal((len(idx), len(b))).astype(np.float32) * np.float32(1e-5))
    return Case(f"survivors-{model}-k{k}", model, k, Q, T, "survivors")


def masking(model, k, n_targets=8192, n=128):
    """History in each row's best chunks (those chunks may not feed tau), target 0 the best of every row under the pad
    mask, one history longer than 256 items, and rows left with exactly k and with k - 1 unmasked targets."""
    d = 64 if PARTS[model] == 1 else 32
    rng = _rng(f"mask{model}{k}")
    b, Q, T = _base(model, d, n, n_targets, rng)
    idx = _spread(n_targets, 4 * k, rng)
    T[idx] = b * (1 + rng.standard_normal((len(idx), len(b))).astype(np.float32) * np.float32(1e-4))
    T[0] = b if DIST[model] else b * np.float32(1.5)   # (the L2 score peaks at t = q, close to b)
    case = Case(f"masking-{model}-k{k}", model, k, Q, T, "mixed")
    a = case.exact()
    hist = []
    for r in range(n):
        best = np.argsort(-a[r, 1:], kind="stable")[: k + 3] + 1
        hist.append(np.sort(best[::2]))                # every other of the best: their chunks are unsafe
    pool = np.setdiff1d(np.arange(1, n_targets), idx)
    hist[1] = np.union1d(hist[1], rng.choice(pool, 300, replace=False))      # longer than RS_HIST
    keep = rng.choice(np.arange(1, n_targets), k + 1, replace=False)
    hist[2] = np.setdiff1d(np.arange(1, n_targets), keep[:k])                # exactly k unmasked
    hist[3] = np.setdiff1d(np.arange(1, n_targets), keep[: k - 1])           # k - 1 unmasked
    case.hist = [h.astype(np.int64) for h in hist]
    case.expect = dict(few_rows=[3], long_hist_row=1, exactly_k_row=2)
    return case


def geometry(model, k, n_targets, n):
    """Catalogue sizes around the 8,192 threshold (partial last chunk) with the best target in the last chunk, and
    row counts that give one row block with four splits, or partial row halves and blocks."""
    d = 64 if PARTS[model] == 1 else 32
    rng = _rng(f"geo{model}{n_targets}{n}")
    P = _parts_width(model, d)
    b = (rng.standard_normal(P) * 0.3).astype(np.float32)
    Q = (b + rng.standard_normal((n, P)).astype(np.float32) * np.float32(0.1)).astype(np.float32)
    T = (rng.standard_normal((n_targets, P)) * 0.1).astype(np.float32)
    T[n_targets - 1] = b * np.float32(0.5)
    T[n_targets - 2] = b * np.float32(0.45)
    return Case(f"geometry-{model}-n{n_targets}-rows{n}", model, k, Q, T, "filter", expect=dict(last_in_topk=True))


def magnitudes(model, k, kind, n_targets=9000, n=96):
    """Tables scaled by 1e-12 / 1e-8 / 1e12 (RotatE at 1e-8: every margin - sqrtf(acc) rounds to the margin, so the
    reported scores tie and only the bound's rounding term for them keeps the filter from dropping the members), per-row query scales from 2^-60 to 2^60 (the E_CLAMP clamp, the e_c > 15
    lowering, e_c < -14 rows), elements that are fp16-subnormal after scaling, and a non-finite query."""
    d = 64 if PARTS[model] == 1 else 32
    rng = _rng(f"mag{model}{k}{kind}")
    b, Q, T = _base(model, d, n, n_targets, rng)
    T[_spread(n_targets, 3 * k, rng)] = b * (1 + rng.standard_normal((3 * k, len(b))).astype(np.float32) * np.float32(1e-4))
    regime = "filter"
    if kind in ("tiny", "tiny8", "huge"):
        s = np.float32({"tiny": 1e-12, "tiny8": 1e-8, "huge": 1e12}[kind])
        Q, T = Q * s, T * s
    elif kind == "rowscale":
        e = np.arange(n) % 21 * 6 - 60                  # 2^-60 .. 2^60
        Q = np.ldexp(Q, e[:, None]).astype(np.float32)
        regime = "mixed"
    elif kind == "subnormal":
        Q[:, ::3] *= np.float32(1e-6)
        T[:, 1::4] *= np.float32(1e-7)
    elif kind == "nonfinite":
        Q[5, 3] = np.inf                                 # |q|^2 = inf
        Q[6, 0] = np.float32(3e20)                       # finite query whose |q|^2 overflows fp32
        regime = "mixed"
    expect = {}
    if kind == "huge" and DIST[model]:
        # max |t|^2 / 2 > 2^68: the clamped e_w overflows the fp16 norm columns (no bound to check), and every row is
        # re-done by the exact kernel
        regime, expect = "few", dict(no_bound=True)
    return Case(f"magnitudes-{model}-{kind}-k{k}", model, k, Q.astype(np.float32), T.astype(np.float32), regime,
                expect=expect)


def long_k(model, k, n_targets=9000, n=128):
    """K = 640 (DistMult d = 640, TransE d = 637): products of alternating sign that cancel over the whole depth."""
    d = 640 if model == "DistMult" else 637
    rng = _rng(f"longk{model}{k}")
    sign = np.where(np.arange(d) % 2 == 0, 1.0, -1.0)
    Q = (sign * (1 + 0.05 * rng.standard_normal((n, d)))).astype(np.float32) * np.float32(0.1)
    T = (1 + 0.3 * rng.standard_normal((n_targets, d))).astype(np.float32) * np.float32(0.1)
    T[_spread(n_targets, 3 * k, rng)] = np.float32(0.1) * (1 + sign * np.float32(0.1)).astype(np.float32)
    return Case(f"long_k-{model}-d{d}-k{k}", model, k, Q, T, "filter")


def kg_near_tie(k=10, n_entities=12000, n=192):
    """Link prediction through full_sort_topk_kg: heads inside a near-tie cluster of entities."""
    model, d = "DistMult", 64
    rng = _rng("kg")
    b, _, T = _base(model, d, 1, n_entities, rng)
    idx = _spread(n_entities, 4 * k, rng)
    T[idx] = b * (1 + rng.standard_normal((len(idx), d)).astype(np.float32) * np.float32(1e-4))
    heads = idx[np.arange(n) % len(idx)]
    return Case(f"kg-near_tie-k{k}", model, k, T[heads].copy(), T, "filter", kg=True, heads=heads)


@functools.lru_cache(maxsize=None)
def all_cases():
    out = []
    for model, k, ms in (("DistMult", 1, (2, 3)), ("DistMult", 32, (33, 128)), ("ComplEx", 10, (11, 40)),
                         ("ComplEx", 32, (128,)), ("TransE", 10, (11, 40)), ("TransE", 32, (33,)),
                         ("RotatE", 1, (2,)), ("RotatE", 32, (33, 128))):
        out += [near_tie(model, k, m) for m in ms]
    out += [norm_tie("TransE", 10), norm_tie("RotatE", 32)]
    out += [duplicates(m, k) for m, k in (("DistMult", 10), ("ComplEx", 1), ("TransE", 32), ("RotatE", 10))]
    out += [overflow("DistMult", 10, 2560), overflow("ComplEx", 32, 200), overflow("TransE", 1, 200),
            overflow("RotatE", 10, 200)]
    out += [survivors("DistMult", 10), survivors("TransE", 32, per_chunk=2, m_chunks=400)]
    out += [masking("DistMult", 10), masking("TransE", 32), masking("RotatE", 1), masking("ComplEx", 10)]
    out += [geometry(m, 10, nt, n) for m, nt, n in (("DistMult", 8192, 1), ("TransE", 8193, 3), ("ComplEx", 8223, 129),
                                                     ("RotatE", 8225, 257), ("DistMult", 8319, 513))]
    out += [magnitudes("DistMult", 10, "tiny"), magnitudes("RotatE", 10, "tiny8"), magnitudes("TransE", 10, "huge"), magnitudes("DistMult", 32, "rowscale"),
            magnitudes("TransE", 10, "rowscale"), magnitudes("ComplEx", 10, "subnormal"),
            magnitudes("RotatE", 32, "subnormal"), magnitudes("DistMult", 10, "nonfinite")]
    out += [long_k("DistMult", 10), long_k("TransE", 32)]
    out += [kg_near_tie()]
    return {c.id: c for c in out}
