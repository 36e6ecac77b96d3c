"""bench.py contract on CPU: the reference arm (oracle port on the host cores) prints ONE JSON line with the keys
the driver reads.  MPCF_BENCH_QUICK shrinks the calibration sample so this stays a few seconds."""
import json
import os
import subprocess
import sys

import pytest
from conftest import ROOT


def test_reference_arm_json_line():
    env = dict(os.environ, MPCF_BENCH_QUICK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0"],
                         capture_output=True, text=True, env=env, timeout=300, check=True).stdout.strip().splitlines()
    line = json.loads(out[-1])
    assert line["impl"] == "reference" and line["metric"] == "rollout_steps_per_s_with_jacobians"
    assert line["unit"] == "rollout-steps/s" and line["higher_is_better"] is True and line["dtype"] == "f64"
    assert line["value"] > 0 and line["steps"] == 1 and line["n_gpus"] == 1
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1 and line["cpu_baseline"]["value"] == line["value"]
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in line["config"] and "model" not in line["config"]


def test_flop_model_is_the_frozen_one():
    sys.path.insert(0, ROOT)
    import bench
    fm = bench.flop_model(6)
    assert (fm["aba"], fm["step_values"], fm["step_jac"], fm["bytes_values"], fm["bytes_jac"]) == (2067, 8580, 223080, 344, 3944)
    assert bench.flop_model(12)["step_values"] == 19188 and bench.flop_model(37)["step_values"] == 63388


@pytest.mark.gpu
def test_c1_headline_times_steps_and_dumps_its_outputs(tmp_path):
    """--config C1: --steps sets the timed launches, the line reports them and the warm-up actually run, and --dump-outputs
    writes every array the node evaluation returns."""
    import numpy as np
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--config", "C1", "--steps", "2", "--warmup", "0",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, check=True)
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["warmup"] == 3 and line["value"] > 0
    for name in ("tau", "q_next", "T_next"):
        a = np.load(tmp_path / (name + ".npy"))
        assert a.dtype == np.float64 and a.shape[0] == 3 and np.isfinite(a).all()


def test_dump_outputs_writes_a_fixed_bounded_sample(tmp_path, monkeypatch):
    """--dump-outputs: a chunked output over its byte share is cut to the same ascending unit columns in every run; a small
    one is written whole; everything is float64 and the files stay within DUMP_BYTES."""
    import numpy as np
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 2 * 1000 * 6 * 8)
    width = 5000
    big = [torch.arange(6 * width, dtype=torch.float64).reshape(2, 3, width) % width + i * width for i in range(3)]
    small = [torch.arange(40, dtype=torch.float32).reshape(4, 10)]
    runs = []
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"big": big, "small": small})
        runs.append({k: np.load(tmp_path / d / (k + ".npy")) for k in ("big", "small")})
    a, b = runs
    assert a["big"].dtype == np.float64 and a["big"].shape == (2, 3, 1000)
    cols = a["big"][0, 0]
    assert (np.diff(cols) > 0).all() and cols[0] >= 0 and cols[-1] < 3 * width and (a["big"] == cols).all()
    assert cols.max() >= 2 * width  # the sample spans the chunks
    assert np.array_equal(a["big"], b["big"]) and np.array_equal(a["small"], b["small"])
    assert a["small"].dtype == np.float64 and np.array_equal(a["small"], np.arange(40.0).reshape(4, 10))
    assert a["big"].nbytes + a["small"].nbytes <= bench.DUMP_BYTES
