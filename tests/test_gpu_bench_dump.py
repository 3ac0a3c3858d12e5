"""bench.py --dump-outputs: the loss and the tables of the last timed train step as float32 .npy files, at most 64 MB
in all; the values are those of the oracle's train steps on the same seeded inputs."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

from kge_helpers import assert_weights_close, make_oracle_model, to_cpu_batch

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench(out_dir, *extra):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "1", "--warmup", "3", "--no-extras",
           "--no-cpu-baseline", "--dump-outputs", str(out_dir), *extra]
    res = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, res.stdout[:500]
    files = {f[: -len(".npy")]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}
    return json.loads(lines[0]), files


def test_dump_outputs_are_the_oracle_steps(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    from oracle.kge_torch import make_optimizer, train_step

    line, got = _bench(tmp_path)
    assert line["steps"] == 1
    w = bench.WORKLOADS["cfg2_transe_ml1m"]
    assert set(got) == {"loss", "user_embedding.weight", "entity_embedding.weight", "relation_embedding.weight"}
    assert got["loss"].shape == (1,) and float(got["loss"][0]) == line["final_loss"]
    # bench.py's headline on rank 0: model seed 2024, four batches of seed 2024, max(warmup, 3, 4) warm-up steps
    # cycling over them, then the timed step
    batches = [to_cpu_batch(b) for b in bench.synth_batches(w, 4, seed=2024)]
    ora = make_oracle_model(w["model"], w["U"], w["I"], w["E"], w["R"], w["d"])
    opt = make_optimizer(ora)
    for i in range(4 + 1):
        want_loss = float(train_step(ora, opt, batches[i % 4]))
    np.testing.assert_allclose(got["loss"][0], want_loss, rtol=1e-5)
    for k, v in ora.state_dict().items():
        assert got[k].dtype == np.float32, k
        # (a triple whose margin term sits at zero within fp32 rounding may count on either side: a few elements can
        # differ by up to the five lr = 1e-3 Adam steps taken)
        assert_weights_close(got[k], v.numpy(), outlier_atol=5e-3, err_msg=k)


def test_dump_outputs_sample_tables_beyond_64mb(tmp_path):
    _, a = _bench(tmp_path, "--workload", "cfg5_transe_alibaba_b2048")
    assert sum(v.nbytes for v in a.values()) <= 64 << 20
    assert a["relation_embedding.weight"].shape == (54, 128)                 # small tables whole
    assert 0 < a["entity_embedding.weight"].shape[0] < 1_000_001 and a["entity_embedding.weight"].shape[1] == 128
    assert all(v.dtype == np.float32 and np.isfinite(v).all() for v in a.values())
