"""bench.py's reference arm runs on the host alone: check that it prints exactly ONE JSON line with the contract's keys.
(The GPU arm needs a B200; its line is produced by the same code path for the shared keys.)"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_contract_line():
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, res.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline", "dtype",
              "data", "config", "cpu_baseline", "e2e"):
        assert k in d, k
    assert d["metric"] == "msckf_updates_per_sec" and d["unit"] == "updates/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and abs(d["value"] * d["ms_per_step"] - 1e3) < 1e-6 * 1e3
    assert "workload" in d["config"] and "400 MSCKF features" in d["config"]["workload"]
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] == 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"] and e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0
    assert d["vs_baseline"] is None and d["dtype"] == "f64" and d["data"] == "rpng_sim"


def test_reference_arm_honours_steps_and_dumps_outputs(tmp_path):
    """--steps K times exactly K updates; --dump-outputs writes what the last one returned to its caller, as float64 .npy files."""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "2", "--warmup", "1",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    d = json.loads(res.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2
    N, F = d["config"]["state_dim"], d["config"]["features_in"]
    shapes = {"status": (F,), "p_FinA": (F, 3), "p_FinG": (F, 3), "anchor_cam": (F,), "anchor_clone": (F,), "chi2": (F,), "dx": (N,), "P": (N, N)}
    assert sorted(p.name for p in tmp_path.iterdir()) == sorted(k + ".npy" for k in shapes)
    a = {k: np.load(tmp_path / (k + ".npy")) for k in shapes}
    for k, shape in shapes.items():
        assert a[k].dtype == np.float64 and a[k].shape == shape and np.isfinite(a[k]).all(), k
    used = a["status"] == 0
    assert int(used.sum()) == d["features_used"]
    # the captured case has rejected features; where one never got a point or a chi², the dump holds 0 instead of the ABI's NaN
    assert (~used).any() and np.all(a["chi2"][used] > 0) and np.all(a["p_FinG"][used].any(axis=1))
    assert np.array_equal(a["P"], a["P"].T) and np.abs(a["dx"]).max() > 0
