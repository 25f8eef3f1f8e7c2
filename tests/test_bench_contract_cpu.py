"""bench.py's reference arm (the CPU restatement timed on the host cores) honours the JSON-line contract; runs on the
CPU with a tiny sample.  Under torchrun only rank 0 prints."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL = ["--impl", "reference", "--steps", "3", "--warmup", "1", "--cpu-instances", "2", "--cpu-steps", "8", "--prefill", "40"]


def _run(extra_env=None):
    env = {k: v for k, v in os.environ.items() if k not in ("RANK", "WORLD_SIZE", "LOCAL_RANK")}
    env.update(extra_env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + SMALL, capture_output=True, text=True,
                          env=env, timeout=600)


def test_reference_arm_json_line():
    out = _run()
    assert out.returncode == 0, out.stderr[-2000:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference"
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
                "vs_baseline", "dtype", "data", "config", "e2e", "cpu_baseline"):
        assert key in line, key
    assert line["unit"] == "instance-steps/s" and line["higher_is_better"] is True and line["dtype"] == "f64"
    assert line["config"]["workload"] == "rm3_irregular_ensemble"
    assert line["value"] > 0 and line["cpu_baseline"]["value"] == line["value"]
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"] == {"value": line["value"], "unit": line["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_stay_silent():
    out = _run({"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert out.returncode == 0, out.stderr[-2000:]
    assert out.stdout.strip() == ""


def test_dump_outputs_keeps_a_fixed_sample_within_the_budget(tmp_path, monkeypatch):
    import numpy as np
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 4096)
    a = np.arange(1000 * 12, dtype=np.float64).reshape(1000, 12)
    for d in ("x", "y"):
        bench.dump_outputs(str(tmp_path / d), {"forces_device": a, "forces_host": -a})
    x, y = np.load(tmp_path / "x" / "forces_device.npy"), np.load(tmp_path / "x" / "forces_host.npy")
    assert 0 < x.nbytes + y.nbytes <= 4096 and x.shape[1] == 12
    np.testing.assert_array_equal(x, -y)                                             # the same rows of every array
    np.testing.assert_array_equal(x, np.load(tmp_path / "y" / "forces_device.npy"))  # ... and of every run
    assert np.all(np.diff(x[:, 0]) > 0)
    bench.dump_outputs(str(tmp_path / "z"), {"f": a[:10]})
    np.testing.assert_array_equal(np.load(tmp_path / "z" / "f.npy"), a[:10])        # within the budget: all of it
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs",
                          str(tmp_path / "r")], capture_output=True, text=True, timeout=600)
    assert out.returncode == 2 and "returns no forces" in out.stderr
