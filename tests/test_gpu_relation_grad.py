"""Relation gradients of one training forward pass against the float64 closed form, and the relation rows it marks.

Batches of at least 148 * 256 triples with d = 68..128 run two triples per warp; TransE and DistMult there sum
relation gradients in per-warp shared-memory copies that leave once per CTA.  Relation layouts that make both
triples of a warp name the same row, or different rows, exercise the merge of the two groups; the other models,
a relation table too large for the copies and a pass without gradients take the per-triple atomics."""

import numpy as np
import pytest

from kge_helpers import closed_form_forward, make_product_model, to_device_batch
from oracle.kge_numpy import loss_weights

pytestmark = pytest.mark.gpu

U, I, E, D = 6041, 3001, 30001, 100
N = 262144   # the benchmark's cfg2 batch: N rec + N KG positives


def _batch(rng, R, n_rec, n_kg, layout="uniform"):
    i = np.arange(n_kg)
    rel = {
        "uniform": lambda: rng.integers(0, R - 1, n_kg),
        "one": lambda: np.full(n_kg, 3),
        "pairs": lambda: np.where((i // 2) % 2 == 0, 3, 7),      # both triples of a warp on one row, rows alternate
        "alternate": lambda: np.where(i % 2 == 0, 3, 7),         # the two triples of a warp on different rows
    }[layout]()
    return {
        "user_id": rng.integers(1, U, n_rec),
        "item_id": rng.integers(1, I, n_rec),
        "neg_item_id": rng.integers(1, I, n_rec),
        "head_id": rng.integers(1, E, n_kg),
        "relation_id": rel,
        "tail_id": rng.integers(1, E, n_kg),
        "neg_tail_id": rng.integers(1, E, n_kg),
    }


def _tables(m, names):
    sd = m.state_dict()
    return [sd[f"{n}.weight"].double().cpu().numpy() for n in names]


def _closed_form(m, name, b, R, margin=1.0):
    """float64 relation gradient [PR][R][d] of the scalar loss, and which relation rows got an active triple."""
    tabs = {"user": _tables(m, m.USER_TABLES), "entity": _tables(m, m.ENTITY_TABLES),
            "relation": _tables(m, m.RELATION_TABLES)}
    w_rec, w_kg = loss_weights(name, len(b["user_id"]), len(b["head_id"]))
    _, g, _, active = closed_form_forward(name, tabs, b, w_rec, w_kg, R - 1, margin, families=("relation",))
    return np.stack(g["relation"]), active["relation"]


def _forward(m, b):
    """One training forward pass: the relation gradient [PR][R][d] and the relation rows marked in its step."""
    m._launch_forward(to_device_batch(b), with_grad=True)
    st = m._state["relation"]
    g = np.stack([t.cpu().numpy() for t in st["g"]])
    marked = st["row_state"][:, 1].cpu().numpy() == m._step + 1
    return g, marked


def _check_grad(got, want, err):
    for p in range(want.shape[0]):
        scale = np.abs(want[p]).max()
        np.testing.assert_allclose(got[p], want[p], rtol=1e-4, atol=1e-4 * scale, err_msg=f"{err} part {p}")


CASES = [
    ("TransE", "uniform", N, N),
    ("TransE", "one", N, N),
    ("TransE", "pairs", N, N),
    ("TransE", "alternate", N, N - 1),     # odd KG half: the last warp's second group has no triple
    ("DistMult", "uniform", N, N),
    ("DistMult", "pairs", N - 3, N + 1),
]


@pytest.mark.parametrize("name,layout,n_rec,n_kg", CASES)
def test_relation_gradient_after_one_forward(name, layout, n_rec, n_kg):
    R = 22
    m = make_product_model(name, U, I, E, R, D)
    b = _batch(np.random.default_rng(11), R, n_rec, n_kg, layout)
    got, marked = _forward(m, b)
    want, active = _closed_form(m, name, b, R)
    _check_grad(got, want, f"{name} {layout}")
    np.testing.assert_array_equal(marked, active)


@pytest.mark.parametrize("name,R", [("TransH", 22), ("TransE", 400)])
def test_relation_gradient_of_the_per_triple_path(name, R):
    """Two relation parts (TransH) and a relation table whose per-warp copies do not fit shared memory."""
    m = make_product_model(name, U, I, E, R, D)
    b = _batch(np.random.default_rng(12), R, N, N)
    got, marked = _forward(m, b)
    want, active = _closed_form(m, name, b, R)
    _check_grad(got, want, name)
    np.testing.assert_array_equal(marked, active)


def test_forward_without_gradient_touches_nothing():
    R = 22
    m = make_product_model("TransE", U, I, E, R, D)
    rng = np.random.default_rng(13)
    m.train_step(to_device_batch(_batch(rng, R, N, N)))   # (creates the optimiser state)
    loss = m._launch_forward(to_device_batch(_batch(rng, R, N, N)), with_grad=False)
    assert float(loss) > 0
    st = m._state["relation"]
    assert not any(bool(t.any()) for t in st["g"])
    assert not bool((st["row_state"][:, 1] == m._step + 1).any())


def test_marked_relation_rows_follow_the_rule():
    """Marked = every row with an active triple, plus every lagging row a triple references (brought up to date by a
    zero-gradient step)."""
    R = 22
    margin = 0.0   # about half of the pairs are inactive
    m = make_product_model("TransE", U, I, E, R, D, margin=margin)
    rng = np.random.default_rng(14)
    # step 1 references every relation, steps 2-3 only relation 1: the others lag behind at step 4
    for step in range(3):
        b = _batch(rng, R, N, N)
        if step:
            b["relation_id"] = np.full(N, 1)
        m.train_step(to_device_batch(b))
    # relations 5..10 get one triple each at step 4: some of those triples are inactive
    b = _batch(rng, R, N, N)
    single = np.arange(5, 11)
    b["relation_id"][np.isin(b["relation_id"], single)] = 2
    b["relation_id"][: len(single)] = single
    got, marked = _forward(m, b)
    _, active = _closed_form(m, "TransE", b, R, margin)   # (state_dict brings the lagging rows to step 3)
    lagging = np.ones(R, dtype=bool)
    lagging[[1, R - 1]] = False
    referenced = np.isin(np.arange(R), b["relation_id"]) | (np.arange(R) == R - 1)
    assert (referenced & lagging & ~active).any()   # (the case the rule is about occurs)
    np.testing.assert_array_equal(marked, active | (referenced & lagging))
