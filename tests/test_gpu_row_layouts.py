"""Every row layout of the train, optimiser and scoring kernels against float64 closed forms.

The row kernels are compiled once per row layout (VEC, G, NCH), which kge_pick_rowcfg (csrc/common.cuh) picks from d
alone, and the forward pass has a two-triples-per-warp shape (4, 16, 2) besides.  The layouts differ exactly where a
kernel goes wrong: partial and wholly empty last chunks, the padding of the TransE-family residuals, group sums over
8, 16 or 32 lanes, register pressure.  D_LADDER reaches every layout at its edges and with partial and empty chunks;
test_ladder_reaches_every_instantiation (no GPU needed) checks that, and prints which test reaches which kernel
instantiation.

Gradients are compared element by element against oracle.kge_numpy's closed forms with a bound scaled by the sum of
the absolute contributions to that element, so a lost or doubled column fails even in a table of small values.  The
optimiser kernels are fed the kernel's own gradient (read back), which isolates the update arithmetic from the
gradient's rounding."""

import numpy as np
import pytest
import torch

from conftest import MODELS
from kge_helpers import closed_form_forward, make_product_model, tile_batch, to_device_batch
from oracle import fullsort as ofs
from oracle.kge_numpy import EPS_PAIRWISE, adam_dense_step, loss_weights, score

gpu = pytest.mark.gpu

D_LADDER = (1, 4, 31, 32, 33, 36, 62, 64, 65, 68, 127, 128, 130, 132, 161, 255, 256, 260, 384, 512)
LAYOUTS = ((4, 8, 1), (4, 16, 1), (4, 32, 1), (4, 32, 2), (4, 32, 4), (1, 32, 1), (1, 32, 2), (1, 32, 4), (1, 32, 8))
TWO_PER_WARP = (4, 16, 2)
TRAIN_KINDS = ("TransE", "DistMult", "RotatE", "ComplEx", "TransH", "TransD")   # (TorusE trains as TransE)
SCORE_KINDS = ("TransE", "DistMult", "RotatE", "TorusE", "ComplEx")            # (TransH / TransD score as TransE)
HINGE = ("TransE", "TorusE", "TransH", "TransD", "DistMult")
FAMILIES = ("user", "entity", "relation")
B200_SMS = 148
# ladder points that run K negatives in the compact layout (k_rec = 2, k_kg = 3): one or more per layout
K_NEG_D = (31, 32, 36, 62, 65, 128, 161, 256, 384)
# one d per layout for the tests that do not need the whole ladder (partial or empty last chunks where there are any)
LAYOUT_D = (4, 36, 68, 132, 384, 31, 33, 65, 161)
# kge_adam_t carries the hyper-parameters as float, so the kernels run Adam with beta1 = fp32(0.9) and beta2 =
# fp32(0.999) = 0.99900001...: 1 - beta2 is then 1.3e-5 (relative) below 0.001, in v and in its bias correction alike.
# The float64 references take the same values.
ADAM = {"lr": float(np.float32(1e-3)), "b1": float(np.float32(0.9)), "b2": float(np.float32(0.999))}
RMSPROP_ALPHA = float(np.float32(0.99))


# ---- Python mirror of the dispatch ----------------------------------------------------------------------------------
def pick_rowcfg(d):
    """kge_pick_rowcfg (csrc/common.cuh:43-60): the (VEC, G, NCH) of a row of d floats, None when d is refused."""
    if d <= 0:
        return None
    if d % 4 == 0:
        nv = d // 4
        if nv <= 8:
            return (4, 8, 1)
        if nv <= 16:
            return (4, 16, 1)
        n = (nv + 31) // 32
        return (4, 32, 1 if n <= 1 else (2 if n <= 2 else 4)) if n <= 4 else None
    n = (d + 31) // 32
    return (1, 32, 1 if n <= 1 else (2 if n <= 2 else (4 if n <= 4 else 8))) if n <= 8 else None


# sm_100 shared memory: opt-in limit per CTA, per SM, and what the runtime reserves per CTA
SMEM_OPTIN, SMEM_PER_SM, SMEM_RESERVED = 232448, 233472, 1024


def fwd_instantiation(name, d, n_rec, n_kg, ue_rows, R, with_grad=True, n_sm=B200_SMS):
    """(kind, layout, WARP_RACC) of the train_fwd_kernel that kge_train_forward (csrc/train.cu:1083-1151) launches.
    `ue_rows`: user + entity rows.  The WARP_RACC residency query is mirrored by the shared-memory bound: the kernel
    wants two resident CTAs (FwdBounds::MIN_CTAS of the two-per-warp shape), registers allow exactly that."""
    kind = "TransE" if name == "TorusE" else name
    cfg = pick_rowcfg(d)
    two = (cfg == (4, 32, 1) and ue_rows * d * 16.0 < 96e6 and n_rec + n_kg >= n_sm * 256
           and kind in ("TransE", "DistMult"))
    racc = False
    if two and with_grad:
        ws = 8 * R * d * 4 + R * 4   # warp_racc_smem_bytes: one relation part
        racc = ws <= SMEM_OPTIN and 2 * (ws + SMEM_RESERVED + 32) <= SMEM_PER_SM   # (+ the static s_loss)
    return kind, (TWO_PER_WARP if two else cfg), racc


def scan_window(rows, n_sm):
    """scan_window (csrc/train.cu:1001-1006): rows per warp window of the row-state scans."""
    win = 32
    while win > 4 and (rows + win - 1) // win < n_sm * 32:
        win >>= 1
    return win


def ladder_sizes(d, n_sm):
    """(n_rec, n_kg): both halves run at least two passes of the grid-stride loop (grid_for(..., 8) caps the grid at
    8 CTAs of 256 threads per SM); for TransE / DistMult at (4, 32, 1) that stays below the two-per-warp threshold."""
    per_pass = n_sm * 8 * (256 // pick_rowcfg(d)[1])
    return per_pass + 37, per_pass + 101


def ladder_k(d):
    return (2, 3) if d in K_NEG_D else (1, 1)


# two-per-warp cases: (tag, d, R, (k_rec, k_kg), with_grad); sizes relative to the threshold T = n_SM * 256
TWO_CASES = [
    ("edge", 68, 22, (1, 1), True),        # n_total == T: takes the shape, WARP_RACC
    ("below", 68, 22, (1, 1), True),       # n_total == T - 1: (4, 32, 1)
    ("edge", 100, 400, (3, 3), True),      # relation copies too large for shared memory: per-triple atomics
    ("rec_only", 128, 22, (1, 1), True),
    ("kg_only", 128, 22, (3, 3), True),    # (odd n_kg)
    ("odd_kg", 100, 22, (1, 3), True),
    ("edge", 100, 22, (1, 1), False),      # no gradient: the shape without WARP_RACC
]


def two_sizes(tag, T):
    return {"edge": (T // 2, T - T // 2), "below": (T // 2, T - T // 2 - 1), "rec_only": (T, 0),
            "kg_only": (0, T + 1), "odd_kg": (T // 2 - 2, T // 2 + 3)}[tag]


# table shapes of the forward tests: small, so that rows collect many contributions
U, I, E, R = 500, 300, 1500, 12
N_ISO = 8   # entity rows [E - N_ISO, E): only ever the positive and the negative of one pair


def _fwd_id(name, d):
    return f"{name}-d{d}"


def _two_id(name, case):
    tag, d, r, k, grad = case
    return f"{name}-{tag}-d{d}-R{r}-k{k[0]}x{k[1]}" + ("" if grad else "-nograd")


def test_ladder_reaches_every_instantiation():
    """The ladder hits every layout, with a partial and an empty last chunk on every multi-chunk G = 32 layout, and
    every kernel instantiation is reached by a case of this file (the map is printed; run with -s to see it)."""
    assert {pick_rowcfg(d) for d in D_LADDER} == set(LAYOUTS)
    assert {pick_rowcfg(d) for d in LAYOUT_D} == set(LAYOUTS) and len(LAYOUT_D) == len(LAYOUTS)
    assert {pick_rowcfg(d) for d in K_NEG_D} == set(LAYOUTS)
    for d in (257, 513, 516, 0):
        assert pick_rowcfg(d) is None
    for vec, g, nch in LAYOUTS:
        if g != 32 or nch == 1:
            continue
        ds = [d for d in D_LADDER if pick_rowcfg(d) == (vec, g, nch)]
        units = [d // vec for d in ds]   # float4s or floats per row; lane l holds units l + 32 j
        # partial last chunk: fewer than 32 units in the last used chunk; empty (NCH >= 4, which rounds the used
        # chunks up): a chunk no lane uses
        assert any(u % 32 for u in units), (vec, nch)
        assert nch == 2 or any((u + 31) // 32 < nch for u in units), (vec, nch)
    reach = {}
    for name in MODELS:
        for d in D_LADDER:
            inst = ("train_fwd", *fwd_instantiation(name, d, *ladder_sizes(d, B200_SMS), U + E, R))
            assert inst[2] == pick_rowcfg(d), (name, d)   # (the ladder's batches keep one triple per warp)
            reach.setdefault(inst, []).append(f"test_forward_and_adam_at_every_layout[{_fwd_id(name, d)}]")
            for kern in ("adam_apply", "predict"):
                kind = "TransE" if name in ("TransH", "TransD") and kern == "predict" else name
                reach.setdefault((kern, kind if kern == "predict" else "", pick_rowcfg(d)), []).append(
                    f"test_{'forward_and_adam' if kern == 'adam_apply' else 'scores'}_at_every_layout[{_fwd_id(name, d)}]")
            if name in ("TransH", "TransD"):
                reach.setdefault((f"{name.lower()}_project", "", pick_rowcfg(d)), []).append(
                    f"test_scores_at_every_layout[{_fwd_id(name, d)}]")
    T = B200_SMS * 256
    for name in ("TransE", "DistMult"):
        for case in TWO_CASES:
            tag, d, r, k, grad = case
            inst = ("train_fwd", *fwd_instantiation(name, d, *two_sizes(tag, T), U + E, r, grad))
            reach.setdefault(inst, []).append(f"test_two_triples_per_warp[{_two_id(name, case)}]")
    for d in LAYOUT_D:
        for kern, test in (("adam_flush", "test_lazy_adam_replay_and_flush"), ("grad_take", "test_row_sparse_exchange"),
                           ("grad_add", "test_row_sparse_exchange")):
            reach.setdefault((kern, "", pick_rowcfg(d)), []).append(f"{test}[d{d}]")
    want = {("train_fwd", k, lay, False) for k in TRAIN_KINDS for lay in LAYOUTS}
    want |= {("train_fwd", k, TWO_PER_WARP, racc) for k in ("TransE", "DistMult") for racc in (False, True)}
    want |= {(kern, "", lay) for kern in ("adam_apply", "adam_flush", "grad_take", "grad_add", "transh_project",
                                          "transd_project") for lay in LAYOUTS}
    want |= {("predict", k, lay) for k in SCORE_KINDS for lay in LAYOUTS}
    assert len(want) == 58 + 6 * 9 + 45
    missing = want - set(reach)
    assert not missing, sorted(missing)
    assert set(reach) <= want, sorted(set(reach) - want)
    for inst in sorted(want, key=str):
        print(inst, "<-", reach[inst][0], f"(+{len(reach[inst]) - 1})")


# ---- batches and tables -----------------------------------------------------------------------------------------------
def _init_tables(m, name, d, rng):
    """Weights of an ordinary scale for every model: DistMult / ComplEx scores of order one (so that a hinge is not
    decided by values near 1e-4), TransH hyperplane vectors whose projection is not near the identity."""
    s = 0.8 * d ** (-1 / 6) if name in ("DistMult", "ComplEx") else 0.1
    with torch.no_grad():
        for tname in m.USER_TABLES + m.ENTITY_TABLES + m.RELATION_TABLES:
            w = getattr(m, tname).weight
            if name == "RotatE" and tname == "relation_embedding":
                x = rng.uniform(0, 2 * np.pi, tuple(w.shape))
            elif tname == "norm_vec":
                x = rng.normal(0, 0.5 / np.sqrt(d), tuple(w.shape))
            else:
                x = rng.normal(0, s, tuple(w.shape))
            w.copy_(torch.from_numpy(x.astype(np.float32)))
    m.invalidate_target_image()


def _tables(m):
    return {f: [getattr(m, n).weight.detach().cpu().numpy().copy() for n in names]
            for f, names in zip(FAMILIES, (m.USER_TABLES, m.ENTITY_TABLES, m.RELATION_TABLES))}


def _f64(tabs):
    return {f: [t.astype(np.float64) for t in ts] for f, ts in tabs.items()}


def _batch(rng, n_rec, n_kg, k_rec, k_kg, U_, I_, E_, R_, iso=True):
    """A compact K-negative batch over ids that avoid the isolated rows.  Planted: rec and KG pairs whose negative is
    their positive, KG anchors that are also the tail, and (K = 1, `iso`) each isolated entity row as both the
    positive and the negative of one KG pair."""
    e_hi = E_ - N_ISO
    b = {
        "user_id": rng.integers(1, U_, n_rec),
        "item_id": rng.integers(1, I_, n_rec),
        "neg_item_id": rng.integers(1, I_, n_rec * k_rec),
        "head_id": rng.integers(1, e_hi, n_kg),
        "relation_id": rng.integers(0, R_ - 1, n_kg),
        "tail_id": rng.integers(1, e_hi, n_kg),
        "neg_tail_id": rng.integers(1, e_hi, n_kg * k_kg),
    }
    j = np.arange(0, n_rec, 41)
    b["neg_item_id"][j] = b["item_id"][j]
    j = np.arange(3, n_kg, 37)
    b["neg_tail_id"][j] = b["tail_id"][j]
    j = np.arange(5, n_kg, 43)
    b["head_id"][j] = b["tail_id"][j]
    planted_kg = np.zeros(n_kg * k_kg, dtype=bool)
    planted_kg[np.arange(3, n_kg, 37)] = True
    if iso and k_kg == 1 and n_kg > 2 * N_ISO:
        j = np.arange(N_ISO) * (n_kg // N_ISO) + 1
        b["tail_id"][j] = b["neg_tail_id"][j] = np.arange(e_hi, E_)
        planted_kg[j] = True
    planted_rec = np.zeros(n_rec * k_rec, dtype=bool)
    planted_rec[np.arange(0, n_rec, 41)] = True
    return b, planted_rec, planted_kg


def _hinge_offset(name, tabs, h_fam, hid, rid, tpid, tnid):
    """z - margin of every (positive, negative) pair of a pairwise model, float64 (the hinge is open at z >= 0)."""
    h = [t[hid] for t in tabs[h_fam]]
    r = [t[rid] for t in tabs["relation"]]
    tp = [t[tpid] for t in tabs["entity"]]
    tn = [t[tnid] for t in tabs["entity"]]
    if name == "DistMult":
        q = h[0] * r[0]
        return -(q * tp[0]).sum(-1) + (q * tn[0]).sum(-1)
    if name == "TransH":
        c = 1.0 - r[1].sum(-1, keepdims=True) * r[1]
        proj = lambda e: e[0] * c   # noqa: E731
    elif name == "TransD":
        proj = lambda e: e[0] + r[1] * (e[0] * e[1]).sum(-1, keepdims=True)   # noqa: E731
    else:
        proj = lambda e: e[0]   # noqa: E731
    x = proj(h) + r[0]
    dist = lambda t: np.sqrt(((x - proj(t) + EPS_PAIRWISE) ** 2).sum(-1))   # noqa: E731
    return dist(tp) - dist(tn)


def _set_margin_and_resample(m, name, tabs, b, planted_rec, planted_kg, k_rec, k_kg, rng, I_, e_hi):
    """Pairwise models: a margin that leaves about half of the pairs inactive (and the planted pairs, whose z is the
    margin, active), then every negative whose float64 z lies within 1e-4 of 0 is drawn again -- which side of the
    hinge such a pair falls on is decided by fp32 rounding, not by the kernel being right."""
    if name not in HINGE:
        return float(np.float32(m.margin))
    n_rec, n_kg = len(b["user_id"]), len(b["head_id"])
    ui = m._ui_row(False)

    def offsets():
        tb = tile_batch(b, k_rec, k_kg)
        o_rec = _hinge_offset(name, tabs, "user", tb["user_id"], np.full(n_rec * k_rec, ui), tb["item_id"],
                              tb["neg_item_id"])
        o_kg = _hinge_offset(name, tabs, "entity", tb["head_id"], tb["relation_id"], tb["tail_id"], tb["neg_tail_id"])
        return o_rec, o_kg

    o_rec, o_kg = offsets()
    o = np.concatenate([o_rec[~planted_rec], o_kg[~planted_kg]])
    margin = float(np.float32(max(np.median(-o), 0.25 * np.std(o))))
    for _ in range(50):
        near_rec = (np.abs(margin + o_rec) < 1e-4) & ~planted_rec
        near_kg = (np.abs(margin + o_kg) < 1e-4) & ~planted_kg
        if not near_rec.any() and not near_kg.any():
            break
        b["neg_item_id"][near_rec] = rng.integers(1, I_, near_rec.sum())
        b["neg_tail_id"][near_kg] = rng.integers(1, e_hi, near_kg.sum())
        o_rec, o_kg = offsets()
    else:
        raise AssertionError("could not move every pair away from the hinge")
    m.margin = margin
    m._struct_cache = {}
    return margin


# ---- checks -------------------------------------------------------------------------------------------------------
def _ulp(x):
    return np.spacing(np.abs(np.asarray(x)).astype(np.float32)).astype(np.float64)


def _forward_state(m):
    st = m._state
    g = {f: [t.cpu().numpy().copy() for t in st[f]["g"]] for f in FAMILIES}
    marked = {f: st[f]["row_state"][:, 1].cpu().numpy() == m._step + 1 for f in FAMILIES}
    return g, marked


def _check_forward(m, name, tabs, b, k, margin, loss, err, iso_rows=None):
    """Loss, every gradient accumulator of every table and part, and the marked rows against the closed form."""
    n_rec, n_kg = len(b["user_id"]), len(b["head_id"])
    w_rec, w_kg = loss_weights(name, n_rec * k[0], n_kg * k[1])
    want_loss, want, a, active = closed_form_forward(name, _f64(tabs), tile_batch(b, *k), w_rec, w_kg,
                                                     m._ui_row(False), margin)
    np.testing.assert_allclose(float(loss), want_loss, rtol=1e-5, err_msg=f"{err} loss")
    got, marked = _forward_state(m)
    for f in FAMILIES:
        for p in range(len(want[f])):
            diff = np.abs(got[f][p].astype(np.float64) - want[f][p])
            # fp32 accumulation of the contributions, element by element: not a bound scaled by the table's largest
            # gradient, which would hide a lost column in a table of small values
            bound = 2e-5 * a[f][p] + 1e-7 * a[f][p].max()
            bad = diff > bound
            if bad.any():
                r_, c_ = np.unravel_index(np.argmax(diff - bound), diff.shape)
                raise AssertionError(
                    f"{err} {f}[{p}]: {bad.sum()} / {bad.size} elements beyond the bound; worst row {r_} col {c_}: "
                    f"got {got[f][p][r_, c_]!r} want {want[f][p][r_, c_]!r} A {a[f][p][r_, c_]!r} "
                    f"(bad columns {np.unique(np.nonzero(bad)[1])[:16]})")
        np.testing.assert_array_equal(marked[f], active[f], err_msg=f"{err} marked {f} rows")
    if iso_rows is not None:
        # positive and negative of one pair and nowhere else: two opposite terms by two atomics cancel exactly
        for p, g in enumerate(got["entity"]):
            assert not g[iso_rows].any(), f"{err} entity[{p}]: an isolated pos == neg row kept a gradient"
            assert active["entity"][iso_rows].all()
    return got, marked


def _check_adam_first_step(m, before, g, marked, err):
    """One Adam step from zero moments on the marked rows, against adam_dense_step fed the kernel's gradient; every
    other row bit-identical and every accumulator zeroed."""
    m._launch_apply(None)
    st = m._state
    for f, names in zip(FAMILIES, (m.USER_TABLES, m.ENTITY_TABLES, m.RELATION_TABLES)):
        t = marked[f]
        rs = st[f]["row_state"].cpu().numpy()
        assert (rs[t, 0] == m._step).all() and (rs[~t, 0] == -1).all(), f"{err} {f} last_step"
        for p, n in enumerate(names):
            w = getattr(m, n).weight.detach().cpu().numpy()
            mm, vv = st[f]["m"][p].cpu().numpy(), st[f]["v"][p].cpu().numpy()
            p0 = before[f][p][t].astype(np.float64)
            want_p, want_m, want_v = adam_dense_step(p0, 0.0, 0.0, g[f][p][t].astype(np.float64), 1, **ADAM)
            # a few ulp: the update's operations (sqrt_nonneg, div_pos_den: within 1 ulp each) and the final rounding
            tol_p = _ulp(want_p) + 8 * 2.0**-23 * np.abs(p0 - want_p)
            assert (np.abs(w[t] - want_p) <= tol_p).all(), f"{err} {f}[{p}] weights after Adam"
            assert (np.abs(mm[t] - want_m) <= 2 * _ulp(want_m)).all(), f"{err} {f}[{p}] m"
            assert (np.abs(vv[t] - want_v) <= 4 * _ulp(want_v)).all(), f"{err} {f}[{p}] v"
            assert np.array_equal(w[~t], before[f][p][~t]), f"{err} {f}[{p}] an unmarked row moved"
            assert not mm[~t].any() and not vv[~t].any(), f"{err} {f}[{p}] moments of an unmarked row"
            assert not st[f]["g"][p].any(), f"{err} {f}[{p}] accumulator not zeroed"


# ---- 2. the forward pass and the first Adam step at every layout, for every model ------------------------------
@gpu
@pytest.mark.parametrize("name,d", [(n, d) for n in MODELS for d in D_LADDER],
                         ids=[_fwd_id(n, d) for n in MODELS for d in D_LADDER])
def test_forward_and_adam_at_every_layout(name, d):
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    n_rec, n_kg = ladder_sizes(d, n_sm)
    k = ladder_k(d)
    assert fwd_instantiation(name, d, n_rec, n_kg, U + E, R, True, n_sm)[1] == pick_rowcfg(d)
    rng = np.random.default_rng(1000 + d + 7 * MODELS.index(name))
    m = make_product_model(name, U, I, E, R, d)
    _init_tables(m, name, d, rng)
    tabs = _tables(m)
    b, pr, pk = _batch(rng, n_rec, n_kg, *k, U, I, E, R)
    margin = _set_margin_and_resample(m, name, _f64(tabs), b, pr, pk, *k, rng, I, E - N_ISO)
    iso = np.arange(E - N_ISO, E) if (name in HINGE and k[1] == 1) else None
    loss = m._launch_forward(to_device_batch(b), with_grad=True)
    g, marked = _check_forward(m, name, tabs, b, k, margin, loss, f"{name} d={d}", iso)
    _check_adam_first_step(m, tabs, g, marked, f"{name} d={d}")


# ---- 3. two triples per warp -------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name,case", [(n, c) for n in ("TransE", "DistMult") for c in TWO_CASES],
                         ids=[_two_id(n, c) for n in ("TransE", "DistMult") for c in TWO_CASES])
def test_two_triples_per_warp(name, case):
    tag, d, R_, k, grad = case
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    n_rec, n_kg = two_sizes(tag, n_sm * 256)
    kind, layout, racc = fwd_instantiation(name, d, n_rec, n_kg, U + E, R_, grad, n_sm)
    assert layout == ((4, 32, 1) if tag == "below" else TWO_PER_WARP)
    assert racc == (grad and R_ == 22 and tag != "below")
    rng = np.random.default_rng(77 + d + R_ + n_kg)
    m = make_product_model(name, U, I, E, R_, d)
    _init_tables(m, name, d, rng)
    tabs = _tables(m)
    b, pr, pk = _batch(rng, n_rec, n_kg, *k, U, I, E, R_)
    margin = _set_margin_and_resample(m, name, _f64(tabs), b, pr, pk, *k, rng, I, E - N_ISO)
    err = f"{name} {tag} d={d} R={R_} k={k}"
    if not grad:
        m._ensure_state(torch.device("cuda"))   # (row states exist: a pass without gradient must not mark any)
        loss = m._launch_forward(to_device_batch(b), with_grad=False)
        w_rec, w_kg = loss_weights(name, n_rec * k[0], n_kg * k[1])
        want_loss = closed_form_forward(name, _f64(tabs), tile_batch(b, *k), w_rec, w_kg, m._ui_row(False), margin,
                                        families=())[0]
        np.testing.assert_allclose(float(loss), want_loss, rtol=1e-5, err_msg=err)
        for f in FAMILIES:
            assert not any(bool(t.any()) for t in m._state[f]["g"]), f"{err}: {f} gradient written"
            assert bool((m._state[f]["row_state"] == -1).all()), f"{err}: {f} row state written"
        return
    iso = np.arange(E - N_ISO, E) if k[1] == 1 and n_kg > 2 * N_ISO else None
    loss = m._launch_forward(to_device_batch(b), with_grad=True)
    g, marked = _check_forward(m, name, tabs, b, k, margin, loss, err, iso)
    _check_adam_first_step(m, tabs, g, marked, err)


# ---- 4. the optimisers over several steps: lazy replay, flush, the other learners ------------------------------
def _steps_batch(rng, rows, n, k):
    """A batch over the given id sets (rows: {"user", "entity", "relation"} arrays)."""
    pick = lambda ids, size: rng.choice(ids, size)   # noqa: E731
    items = rows["entity"][rows["entity"] < I]
    return {"user_id": pick(rows["user"], n), "item_id": pick(items, n), "neg_item_id": pick(items, n * k),
            "head_id": pick(rows["entity"], n), "relation_id": pick(rows["relation"], n),
            "tail_id": pick(rows["entity"], n), "neg_tail_id": pick(rows["entity"], n * k)}


def _dense_grads(m):
    return {f: [t.double().cpu().numpy() for t in m._state[f]["g"]] for f in FAMILIES}


def _run_three_steps(m, rng):
    """Step 1 references the rows A and B, step 2 A only, step 3 A and half of B; returns the gradients the kernel
    accumulated in every step (dense, zero on idle rows)."""
    ids = {"user": np.arange(1, U), "entity": np.arange(1, E), "relation": np.arange(0, R - 1)}
    half = {f: (x[: len(x) // 2], x[len(x) // 2 :]) for f, x in ids.items()}
    a_rows = {f: h[0] for f, h in half.items()}
    ab1 = {f: np.concatenate([h[0], h[1][: len(h[1]) // 2]]) for f, h in half.items()}
    grads = []
    for rows in (ids, a_rows, ab1):
        b = _steps_batch(rng, rows, 3000, 1)
        m._launch_forward(to_device_batch(b), with_grad=True)
        grads.append(_dense_grads(m))
        m._launch_apply(None)
    return grads


def _check_against_dense(m, want_w, want_v, move, err, want_m=None, m_scale=None):
    m.state_dict()   # flushes: every row brought to the last step
    st = m._state
    for f, names in zip(FAMILIES, (m.USER_TABLES, m.ENTITY_TABLES, m.RELATION_TABLES)):
        for p, n in enumerate(names):
            w = getattr(m, n).weight.detach().cpu().numpy()
            # a few ulp per step: the replayed and the real updates are within a few ulp of the float64 ones
            tol = 4 * _ulp(want_w[f][p]) + 2e-6 * move[f][p]
            bad = np.abs(w - want_w[f][p]) > tol
            assert not bad.any(), f"{err} {f}[{p}] weights: {bad.sum()} elements, rows {np.unique(np.nonzero(bad)[0])[:10]}"
            if want_v is not None:
                vv = st[f]["v"][p].cpu().numpy()
                np.testing.assert_allclose(vv, want_v[f][p], rtol=2e-6, atol=1e-38, err_msg=f"{err} {f}[{p}] v")
            if want_m is not None:
                # (m = b1 m + (1 - b1) g cancels where g turns against m: its rounding scales with the same recursion
                # on absolute values, not with |m|)
                mm = st[f]["m"][p].cpu().numpy()
                bad = np.abs(mm - want_m[f][p]) > 2e-6 * m_scale[f][p] + 1e-38
                assert not bad.any(), f"{err} {f}[{p}] m: {bad.sum()} elements"


def _dense_adam_step(p, mo, vo, move, m_abs, g, step):
    """float64 dense Adam on whole tables, in place; `move` sums |update| and `m_abs` runs m's recursion on |g|."""
    for f in FAMILIES:
        for i in range(len(p[f])):
            new, mo[f][i], vo[f][i] = adam_dense_step(p[f][i], mo[f][i], vo[f][i], g[f][i], step, **ADAM)
            m_abs[f][i] = ADAM["b1"] * m_abs[f][i] + (1 - ADAM["b1"]) * np.abs(g[f][i])
            move[f][i] += np.abs(new - p[f][i])
            p[f][i] = new


@gpu
@pytest.mark.parametrize("d", LAYOUT_D, ids=lambda d: f"d{d}")
def test_lazy_adam_replay_and_flush(d):
    """Rows idle in some steps: the next forward / Adam step replays the skipped zero-gradient steps, the flush brings
    the rest up; against float64 dense Adam on whole tables with zero gradients on idle rows."""
    name = MODELS[LAYOUT_D.index(d) % len(MODELS)]
    rng = np.random.default_rng(500 + d)
    m = make_product_model(name, U, I, E, R, d)
    _init_tables(m, name, d, rng)
    ref = _f64(_tables(m))
    mo = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    vo = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    move = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    m_abs = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    for step, g in enumerate(_run_three_steps(m, rng), start=1):
        _dense_adam_step(ref, mo, vo, move, m_abs, g, step)
    _check_against_dense(m, ref, vo, move, f"{name} d={d}", want_m=mo, m_scale=m_abs)


@gpu
@pytest.mark.parametrize("learner,lr", [("sgd", 0.5), ("adagrad", 0.05), ("rmsprop", 1e-3)])
@pytest.mark.parametrize("d", LAYOUT_D, ids=lambda d: f"d{d}")
def test_other_learners_at_every_layout(d, learner, lr):
    """SGD, Adagrad and RMSprop against torch.optim in float64 fed the kernel's gradients; RMSprop's second moments of
    idle rows decay through the replay and the flush."""
    name = MODELS[(LAYOUT_D.index(d) + 3) % len(MODELS)]
    rng = np.random.default_rng(600 + d)
    m = make_product_model(name, U, I, E, R, d, learner=learner, lr=lr)
    _init_tables(m, name, d, rng)
    init = _f64(_tables(m))
    params = {f: [torch.tensor(t, requires_grad=True) for t in ts] for f, ts in init.items()}
    flat = [t for f in FAMILIES for t in params[f]]
    lr32 = float(np.float32(lr))
    opt = {"sgd": lambda: torch.optim.SGD(flat, lr=lr32), "adagrad": lambda: torch.optim.Adagrad(flat, lr=lr32),
           "rmsprop": lambda: torch.optim.RMSprop(flat, lr=lr32, alpha=RMSPROP_ALPHA)}[learner]()
    move = {f: [np.zeros_like(t) for t in ts] for f, ts in init.items()}
    for g in _run_three_steps(m, rng):
        old = {f: [t.detach().numpy().copy() for t in params[f]] for f in FAMILIES}
        for f in FAMILIES:
            for p, t in enumerate(params[f]):
                t.grad = torch.from_numpy(g[f][p])
        opt.step()
        for f in FAMILIES:
            for p, t in enumerate(params[f]):
                move[f][p] += np.abs(t.detach().numpy() - old[f][p])
    want_w = {f: [t.detach().numpy() for t in params[f]] for f in FAMILIES}
    key = {"adagrad": "sum", "rmsprop": "square_avg"}.get(learner)
    want_v = None if key is None else {f: [opt.state[t][key].numpy() for t in params[f]] for f in FAMILIES}
    _check_against_dense(m, want_w, want_v, move, f"{learner} {name} d={d}")


@gpu
@pytest.mark.parametrize("win", [8, 16, 32])
def test_scan_windows(win):
    """Tables at the lower edge of the row-state scan's 8, 16 and 32-row windows (rows % 32 != 0): row 0, the last row
    and the first and last rows of windows are updated, every other row stays bit-identical; then a flush replays the
    rows a second step left idle."""
    n_sm = torch.cuda.get_device_properties(0).multi_processor_count
    rows = win * (n_sm * 32 - 1) + 1   # the smallest table with this window
    assert scan_window(rows, n_sm) == win and scan_window(rows - 1, n_sm) == win // 2 and rows % 32
    d, R_ = 8, 4
    m = make_product_model("ComplEx", rows, rows, rows, R_, d)   # (ComplEx: every referenced row gets a gradient)
    rng = np.random.default_rng(win)
    n_win = (rows + win - 1) // win
    wins = np.array([0, 1, n_win // 2, n_win - 2, n_win - 1])
    edge = np.unique(np.concatenate([wins * win, np.minimum(wins * win + win - 1, rows - 1), [0, rows - 1]]))
    touched = np.unique(np.concatenate([edge, rng.integers(0, rows, 300)]))
    before = _tables(m)
    ref = _f64(before)

    def step(ids):
        n = len(ids)
        b = {"user_id": ids, "item_id": ids[::-1].copy(), "neg_item_id": rng.permutation(ids), "head_id": ids,
             "relation_id": rng.integers(0, R_ - 1, n), "tail_id": rng.permutation(ids), "neg_tail_id": ids[::-1].copy()}
        m._launch_forward(to_device_batch(b), with_grad=True)
        g = _dense_grads(m)
        m._launch_apply(None)
        return g

    g1 = step(touched)
    for f in ("user", "entity"):
        rs = m._state[f]["row_state"].cpu().numpy()
        np.testing.assert_array_equal(np.flatnonzero(rs[:, 0] == 1), touched, err_msg=f"win {win} {f} rows updated")
        for p, n in enumerate(m.USER_TABLES if f == "user" else m.ENTITY_TABLES):
            w = getattr(m, n).weight.detach().cpu().numpy()
            want, _, _ = adam_dense_step(ref[f][p][touched], 0.0, 0.0, g1[f][p][touched], 1, **ADAM)
            tol = _ulp(want) + 8 * 2.0**-23 * np.abs(want - ref[f][p][touched])
            assert (np.abs(w[touched] - want) <= tol).all(), f"win {win} {f}[{p}]"
            idle = np.ones(rows, dtype=bool)
            idle[touched] = False
            assert np.array_equal(w[idle], before[f][p][idle]), f"win {win} {f}[{p}]: an idle row moved"
    # step 2 leaves the window edges idle: the flush replays them
    g2 = step(np.setdiff1d(touched, edge))
    mo = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    vo = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    move = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    m_abs = {f: [np.zeros_like(t) for t in ts] for f, ts in ref.items()}
    for s, g in ((1, g1), (2, g2)):
        _dense_adam_step(ref, mo, vo, move, m_abs, g, s)
    _check_against_dense(m, ref, vo, move, f"win {win}", want_m=mo, m_scale=m_abs)


# ---- 5. the row-sparse exchange on one GPU -------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("d", LAYOUT_D, ids=lambda d: f"d{d}")
def test_row_sparse_exchange(d):
    """kge_grad_pack hands out exactly the marked rows' accumulators and clears them; kge_grad_add into a twin with
    the same weights restores them bit for bit with the same marks, and the next Adam step of both is identical."""
    from hopwise_b200.distributed import FlatLayout, _cuda_add, _cuda_pack

    name = MODELS[(LAYOUT_D.index(d) + 5) % len(MODELS)]
    models = []
    for _ in range(2):
        m = make_product_model(name, U, I, E, R, d)
        _init_tables(m, name, d, np.random.default_rng(900 + d))
        models.append(m)
    m1, m2 = models
    rng = np.random.default_rng(901 + d)
    b, _, _ = _batch(rng, 2000, 3000, 1, 2, U, I, E, R)
    m1._launch_forward(to_device_batch(b), with_grad=True)
    g, marked = _forward_state(m1)
    rows_of = {"user": U, "entity": E, "relation": R}
    parts = [len(g[f]) for f in FAMILIES]
    lay = FlatLayout([rows_of[f] for f in FAMILIES], parts, d)
    buf = torch.zeros(lay.nbytes, dtype=torch.uint8, device="cuda")
    for which, f in enumerate(FAMILIES):
        count, ids, rows = lay.views(buf, which)
        _cuda_pack(m1, which, 1, count, ids, rows)
        n = int(count.item())
        got_ids = ids[:n].cpu().numpy()
        np.testing.assert_array_equal(np.sort(got_ids), np.flatnonzero(marked[f]), err_msg=f"{f} packed ids")
        packed = rows[:n].view(n, parts[which], d).cpu().numpy()
        for p in range(parts[which]):
            assert np.array_equal(packed[:, p], g[f][p][got_ids]), f"{f}[{p}] packed rows"
            assert not m1._state[f]["g"][p].any(), f"{f}[{p}] accumulator not zeroed by the pack"
        assert bool((m1._state[f]["row_state"][:, 1] == -1).all()), f"{f} marks not cleared"
    m2._ensure_state(torch.device("cuda"))
    for which, f in enumerate(FAMILIES):
        count, ids, rows = lay.views(buf, which)
        for m in (m1, m2):
            _cuda_add(m, which, 1, count, ids, rows)
        got, mk = _forward_state(m2)
        for p in range(parts[which]):
            assert np.array_equal(got[f][p], g[f][p]), f"{f}[{p}] accumulator after the add"
        np.testing.assert_array_equal(mk[f], marked[f], err_msg=f"{f} marks after the add")
    m2._pending = True
    for m in (m1, m2):
        m._launch_apply(None)
    for f, names in zip(FAMILIES, (m1.USER_TABLES, m1.ENTITY_TABLES, m1.RELATION_TABLES)):
        for p, n in enumerate(names):
            assert torch.equal(getattr(m1, n).weight, getattr(m2, n).weight), f"{n} after the step"
            for key in ("m", "v"):
                assert torch.equal(m1._state[f][key][p], m2._state[f][key][p]), f"{n} {key}"


# ---- 6. scoring at every layout ----------------------------------------------------------------------------------
def _score_abs(name, h, r, t, margin):
    """The scale of a score's fp32 rounding: the sum of the absolute terms of its contraction (distance models: the
    norm of the residual formed from absolute values)."""
    ab = np.abs
    if name == "DistMult":
        return (ab(h[0] * r[0] * t[0])).sum(-1)
    if name == "ComplEx":
        return (ab(h[0] * r[0] * t[0]) + ab(h[1] * r[0] * t[1]) + ab(h[0] * r[1] * t[1]) + ab(h[1] * r[1] * t[1])).sum(-1)
    if name == "RotatE":
        c, s = ab(np.cos(r[0])), ab(np.sin(r[0]))
        x = c * ab(h[0]) + s * ab(h[1]) + ab(t[0]) + c * ab(h[1]) + s * ab(h[0]) + ab(t[1])
        return abs(margin) + np.sqrt((x * x).sum(-1))
    if name == "TorusE":
        fr = lambda a: ab(a - np.trunc(a))   # noqa: E731
        return 4 * (2 * (fr(h[0]) + fr(r[0]) + fr(t[0])) ** 2 + 1).sum(-1)
    if name == "TransH":
        k = 1 + ab(r[1]).sum(-1, keepdims=True) * ab(r[1])
        x = (ab(h[0]) + ab(t[0])) * k + ab(r[0])
    elif name == "TransD":
        pr = lambda e: ab(e[0]) + ab(r[1]) * ab(e[0] * e[1]).sum(-1, keepdims=True)   # noqa: E731
        x = pr(h) + ab(r[0]) + pr(t)
    else:
        x = ab(h[0]) + ab(r[0]) + ab(t[0])
    return np.sqrt((x * x).sum(-1))


def _check_scores(got, name, h, r, t, margin, err, chunk=4):
    """got [n] or [n, n_targets] (then h / r: [n] rows, t: every target) against kge_numpy.score."""
    want, a = np.empty(got.shape), np.empty(got.shape)
    if got.ndim == 1:
        want[:] = score(name, h, r, t, margin)
        a[:] = _score_abs(name, h, r, t, margin)
    else:
        for s in range(0, got.shape[0], chunk):   # (the [rows, targets, d] temporaries stay small)
            hh = [x[s : s + chunk, None] for x in h]
            rr = [x[s : s + chunk, None] for x in r]
            tt = [x[None] for x in t]
            want[s : s + chunk] = score(name, hh, rr, tt, margin)
            a[s : s + chunk] = _score_abs(name, hh, rr, tt, margin)
    bad = np.abs(got - want) > 1e-5 * np.abs(want) + 1e-6 * a
    assert not bad.any(), f"{err}: {bad.sum()} / {bad.size} scores beyond the bound, first at {np.argwhere(bad)[0]}"


@gpu
@pytest.mark.parametrize("name,d", [(n, d) for n in MODELS for d in D_LADDER],
                         ids=[_fwd_id(n, d) for n in MODELS for d in D_LADDER])
def test_scores_at_every_layout(name, d):
    """predict / predict_kg / full_sort_predict / full_sort_predict_kg (where the model has them) against the float64
    scores, and the fused top-k against the canonical top-k of the dense masked scores, exactly."""
    U_, I_, E_, R_ = 60, 300, 700, 9
    rng = np.random.default_rng(3000 + d + 11 * MODELS.index(name))
    m = make_product_model(name, U_, I_, E_, R_, d)
    _init_tables(m, name, d, rng)
    tabs = _f64(_tables(m))
    margin = float(np.float32(m.margin))
    ui = m._ui_row(False)
    err = f"{name} d={d}"
    cuda = lambda x: torch.from_numpy(np.asarray(x)).cuda()   # noqa: E731
    rel = lambda ids: [t[ids] for t in tabs["relation"]]   # noqa: E731
    users, items = rng.integers(0, U_, 97), rng.integers(0, I_, 97)
    got = m.predict({"user_id": cuda(users), "item_id": cuda(items)}).cpu().numpy()
    _check_scores(got, name, [t[users] for t in tabs["user"]], rel(np.full(97, ui)),
                  [t[items] for t in tabs["entity"]], margin, f"{err} predict")
    if name != "TransH":
        heads, rels, tails = rng.integers(0, E_, 53), rng.integers(0, R_ - 1, 53), rng.integers(0, E_, 53)
        got = m.predict_kg({"head_id": cuda(heads), "relation_id": cuda(rels), "tail_id": cuda(tails)}).cpu().numpy()
        _check_scores(got, name, [t[heads] for t in tabs["entity"]], rel(rels), [t[tails] for t in tabs["entity"]],
                      margin, f"{err} predict_kg")
    qu = rng.integers(1, U_, 13)
    dense = m.full_sort_predict({"user_id": cuda(qu)}).cpu().numpy()
    ui_fs = m._ui_row(True)
    _check_scores(dense, name, [t[qu] for t in tabs["user"]], rel(np.full(13, ui_fs)),
                  [t[:I_] for t in tabs["entity"]], margin, f"{err} full_sort_predict")
    if name not in ("TransH", "TransD"):
        qh, qr = rng.integers(1, E_, 6), rng.integers(0, R_ - 1, 6)
        got = m.full_sort_predict_kg({"head_id": cuda(qh), "relation_id": cuda(qr)}).cpu().numpy()
        _check_scores(got, name, [t[qh] for t in tabs["entity"]], rel(qr), tabs["entity"], margin,
                      f"{err} full_sort_predict_kg")
    # the fused top-k: exactly the canonical top-k of the dense masked scores
    hist_u = np.repeat(np.arange(len(qu)), rng.integers(0, 40, len(qu)))
    hist_i = rng.integers(1, I_, len(hist_u))
    from hopwise_b200 import evaluator as ev

    hist_off, hist_items = ev.csr_from_pairs(hist_u, hist_i, len(qu), "cuda")
    k = 20
    ids, sc = m.full_sort_topk(cuda(qu), k, hist_off, hist_items, path="cuda")
    want_ids, want_sc = ofs.topk_canonical(ofs.mask_scores(dense, hist_u, hist_i), k)
    np.testing.assert_array_equal(ids.cpu().numpy(), want_ids, err_msg=f"{err} top-k ids")
    np.testing.assert_array_equal(sc.cpu().numpy(), want_sc, err_msg=f"{err} top-k scores")
