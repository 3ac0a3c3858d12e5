"""Weight decay without a GPU: which learner / weight_decay pairs the models take, the kge_adam_t slot that carries the
decay, and the library's refusal of the decay it cannot apply row by row (coupled L2 under Adam, Adagrad, RMSprop)."""

import contextlib
import ctypes as C
import math

import pytest

from kge_helpers import make_product_model


def _model(**cfg):
    return make_product_model("TransE", 10, 8, 20, 5, 16, device="cpu", **cfg)


def test_learner_mapping_with_weight_decay():
    assert _model(learner="adamw").learner == "adam"                       # AdamW at weight decay 0 is Adam
    m = _model(learner="AdamW", weight_decay=0.01)
    assert (m.learner, m.weight_decay) == ("adamw", 0.01)
    m = _model(learner="sgd", weight_decay=0.5)
    assert (m.learner, m.weight_decay) == ("sgd", 0.5)
    a = m._adam_struct(3)
    assert a.optimizer == 1 and a.weight_decay == pytest.approx(0.5) and a.step == 3
    assert _model(learner="adamw", weight_decay=0.01)._adam_struct(1).optimizer == 4
    assert _model()._adam_struct(1).weight_decay == 0.0


@pytest.mark.parametrize("learner", ["adam", "adagrad", "rmsprop", "lion"])
def test_coupled_l2_is_refused_and_names_the_supported_learners(learner):
    with pytest.warns(UserWarning) if learner == "lion" else contextlib.nullcontext():
        with pytest.raises(NotImplementedError, match="adamw.*sgd"):
            _model(learner=learner, weight_decay=0.1)


@pytest.mark.parametrize("wd", [-0.1, math.inf, math.nan])
@pytest.mark.parametrize("learner", ["adamw", "sgd"])
def test_negative_or_non_finite_weight_decay_is_refused(learner, wd):
    with pytest.raises(NotImplementedError):
        _model(learner=learner, weight_decay=wd)


def test_clip_grad_norm_stays_refused_with_weight_decay():
    with pytest.raises(NotImplementedError):
        _model(learner="adamw", weight_decay=0.1, clip_grad_norm={"max_norm": 5})


def test_weight_decay_slot_of_kge_adam_t():
    from hopwise_b200 import _abi

    assert C.sizeof(_abi.kge_adam_t) == 32
    assert _abi.kge_adam_t.weight_decay.offset == 28 and _abi.kge_adam_t.weight_decay.size == 4
    assert _abi.kge_adam_t().weight_decay == 0.0   # a zeroed struct: no decay
    assert _abi.OPTIMIZERS["adamw"] == 4


def _fake_model():
    """A TransE struct whose pointers are never dereferenced: every call below is refused before any launch."""
    from hopwise_b200 import _abi

    m = _abi.kge_model_t()
    m.model, m.d = _abi.MODEL_KINDS["TransE"], 16
    for fam in ("user", "entity", "relation"):
        t = getattr(m, fam)
        t.rows, t.parts = 10, 1
        t.w[0] = t.m[0] = t.v[0] = t.g[0] = 256
        t.row_state = 256
    return m


def _adam(opt, wd):
    from hopwise_b200 import _abi

    a = _abi.kge_adam_t()
    a.lr, a.beta1, a.beta2, a.eps, a.step, a.replay_cap = 1e-3, 0.9, 0.999, 1e-8, 1, 200
    a.optimizer, a.weight_decay = opt, wd
    return a


@pytest.mark.parametrize("opt,wd", [(0, 0.1), (2, 0.1), (3, 1e-4), (4, -0.5), (1, math.inf), (4, math.nan)])
def test_library_refuses_weight_decay_it_cannot_apply(opt, wd):
    from hopwise_b200 import _abi

    lib = _abi.lib()
    m, a = C.byref(_fake_model()), C.byref(_adam(opt, wd))
    b = _abi.kge_batch_t()
    b.k_rec = b.k_kg = 1
    loss = 256
    calls = {
        "kge_train_forward": lambda: lib.kge_train_forward(m, C.byref(b), a, 1, loss, None),
        "kge_train_step": lambda: lib.kge_train_step(m, C.byref(b), a, 1.0, loss, None),
        "kge_adam_apply": lambda: lib.kge_adam_apply(m, a, 1.0, None, None),
        "kge_adam_flush": lambda: lib.kge_adam_flush(m, a, None),
        "kge_owner_adam_step": lambda: lib.kge_owner_adam_step(256, 256, 256, 256, 256, 256, 16, 0, 2, a, 1.0, 256, 0,
                                                               256, 1, None),
    }
    for name, call in calls.items():
        assert call() == -2, name   # KGE_E_UNSUPPORTED
        assert b"weight_decay" in lib.kge_last_error(), name


def test_owner_sharded_step_refuses_optimizers_other_than_adam_and_adamw():
    from hopwise_b200 import _abi

    lib = _abi.lib()
    for opt, wd in ((1, 0.1), (1, 0.0), (2, 0.0), (3, 0.0)):
        rc = lib.kge_owner_adam_step(256, 256, 256, 256, 256, 256, 16, 0, 2, C.byref(_adam(opt, wd)), 1.0, 256, 0, 256,
                                     1, None)
        assert rc == -2, (opt, wd)

