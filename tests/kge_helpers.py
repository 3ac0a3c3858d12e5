"""Shared helpers of the parity tests: build product models / oracle twins on given shapes."""

import numpy as np
import torch

from oracle.kge_torch import OracleKGE, Shapes

BATCH_KEYS = ("user_id", "item_id", "neg_item_id", "head_id", "relation_id", "tail_id", "neg_tail_id")

BASE_CONFIG = {
    "USER_ID_FIELD": "user_id",
    "ITEM_ID_FIELD": "item_id",
    "NEG_PREFIX": "neg_",
    "ENTITY_ID_FIELD": "entity_id",
    "RELATION_ID_FIELD": "relation_id",
    "HEAD_ENTITY_ID_FIELD": "head_id",
    "TAIL_ENTITY_ID_FIELD": "tail_id",
    "margin": 1.0,
    "learner": "adam",
    "learning_rate": 0.001,
    "weight_decay": 0.0,
}


class ShapeDataset:
    """The dataset attributes the model constructors read (SURVEY.md 8(b))."""

    def __init__(self, U, I, E, R, ui_token_id=None):
        self._num = {"user_id": U, "item_id": I, "entity_id": E, "relation_id": R}
        self.ui_relation = "[UI-Relation]"
        self.field2token_id = {"relation_id": {"[UI-Relation]": R - 1 if ui_token_id is None else ui_token_id}}

    def num(self, field):
        return self._num[field]


def make_product_model(name, U, I, E, R, d, device="cuda", margin=1.0, seed=2024, lr=1e-3, **cfg):
    import hopwise_b200

    config = dict(BASE_CONFIG, embedding_size=d, margin=margin, device=torch.device(device), learning_rate=lr, **cfg)
    torch.manual_seed(seed)
    model = hopwise_b200.MODELS[name](config, ShapeDataset(U, I, E, R))
    return model.to(device)


def make_oracle_model(name, U, I, E, R, d, margin=1.0, seed=2024):
    torch.manual_seed(seed)
    return OracleKGE(name, Shapes(U, I, E, R, d, margin=margin))


def random_batch(rng, U, I, E, R, n_rec, n_kg, k_rec=1, k_kg=1):
    return {
        "user_id": rng.integers(1, U, n_rec),
        "item_id": rng.integers(1, I, n_rec),
        "neg_item_id": rng.integers(1, I, n_rec * k_rec),
        "head_id": rng.integers(1, E, n_kg),
        "relation_id": rng.integers(1, R - 1, n_kg),
        "tail_id": rng.integers(1, E, n_kg),
        "neg_tail_id": rng.integers(1, E, n_kg * k_kg),
    }


def to_device_batch(b, device="cuda"):
    return {k: torch.as_tensor(np.asarray(v), dtype=torch.long).to(device) for k, v in b.items()}


def tile_batch(b, k_rec, k_kg):
    """The reference's K-negative layout: positives repeated K times (abstract_dataloader.py:192-198)."""
    out = dict(b)
    for key in ("user_id", "item_id"):
        out[key] = np.tile(b[key], k_rec)
    for key in ("head_id", "relation_id", "tail_id"):
        out[key] = np.tile(b[key], k_kg)
    return out


def to_cpu_batch(b):
    return {k: torch.as_tensor(np.asarray(v), dtype=torch.long) for k, v in b.items()}


def closed_form_forward(name, tabs, b, w_rec, w_kg, ui_row, margin=1.0, families=None, chunk=65536):
    """float64 closed form of one training forward pass (oracle.kge_numpy.pair_loss_and_grads on every pair).

    tabs: {"user" | "entity" | "relation": [float64 table per part]}; b: one entry per (positive, negative) pair
    (the tiled view of a K-negative batch, `tile_batch`); w_rec / w_kg: the weight of one pair in the scalar loss.
    Returns (loss, g, a, active): g and a are per family lists shaped like the tables -- the gradient, and the scale of
    its fp32 rounding: the sum over the contributing pairs of the pair's largest gradient term in that column (the
    head and relation gradients of the translation models are differences of the two tails' terms, which cancel in
    float64 where fp32 keeps their rounding; at d = 1 they cancel in every pair whose residuals share a sign) -- and
    active[family] is a bool [rows] of the rows of a pair with a gradient (pairwise models: the hinge is open; the
    user->item relation row belongs to every rec pair).  With `families`, g and a are accumulated for those families only."""
    from oracle.kge_numpy import pair_loss_and_grads

    g = {f: [np.zeros_like(t) for t in ts] for f, ts in tabs.items()}
    a = {f: [np.zeros_like(t) for t in ts] for f, ts in tabs.items()}
    active = {f: np.zeros(len(ts[0]), dtype=bool) for f, ts in tabs.items()}
    loss = 0.0
    n_rec = len(b["user_id"])
    segs = (("user", b["user_id"], np.full(n_rec, ui_row), b["item_id"], b["neg_item_id"], w_rec),
            ("entity", b["head_id"], b["relation_id"], b["tail_id"], b["neg_tail_id"], w_kg))
    for hfam, hid, rid, tpid, tnid, w in segs:
        fams = (hfam, "relation", "entity", "entity")
        for s in range(0, len(hid), chunk):   # (chunks keep the float64 temporaries small)
            ids = [np.asarray(x[s : s + chunk]) for x in (hid, rid, tpid, tnid)]
            rows = [[t[i] for t in tabs[f]] for f, i in zip(fams, ids)]
            l, *grads = pair_loss_and_grads(name, *rows, w, margin)
            loss += l
            act = np.any(np.stack([x != 0 for gs in grads for x in gs]), axis=(0, 2))
            scale = np.max(np.stack([np.abs(x) for gs in grads for x in gs]), axis=0)
            for f, i, gs in zip(fams, ids, grads):
                if families is not None and f not in families:
                    continue
                for p, x in enumerate(gs):
                    np.add.at(g[f][p], i, x)
                    np.add.at(a[f][p], i, scale)
                active[f][i[act]] = True
    return loss, g, a, active


def assert_weights_close(got, want, rtol=1e-5, atol=5e-7, outlier_frac=5e-4, outlier_atol=1e-4, err_msg=""):
    """Post-Adam weights: every element within rtol/atol, except a bounded few.

    Adam's update lr * m / (sqrt(v) + eps) amplifies rounding noise of a near-zero gradient
    (|g| ~ eps = 1e-8, e.g. duplicate rows whose contributions cancel): d(update)/dg peaks at
    lr / (4 eps) = 2.5e4, so two correct fp32 implementations that sum in a different order can
    differ by up to ~1e-5..1e-4 on such an element.  Those elements are allowed, but only
    `outlier_frac` of a table (two at least) and never beyond `outlier_atol` (a tenth of one Adam step).
    """
    got, want = np.asarray(got), np.asarray(want)
    assert got.shape == want.shape, err_msg
    diff = np.abs(got - want)
    bad = diff > atol + rtol * np.abs(want)
    assert np.isfinite(got).all(), err_msg
    # (at least two elements per table: the float atomics of the gradient scatter add in a different order every run, so
    # WHICH nearly cancelled element lands beyond the tolerance varies from run to run on small tables)
    allowed = max(2, int(outlier_frac * bad.size))
    assert bad.sum() <= allowed, f"{err_msg}: {bad.sum()} / {bad.size} elements beyond rtol={rtol}, atol={atol}"
    assert diff.max() <= outlier_atol, f"{err_msg}: max abs diff {diff.max()} > {outlier_atol}"
