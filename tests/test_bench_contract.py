"""bench.py prints ONE JSON line with the contract's keys (both arms)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches"}


def _run(args, timeout=600):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1, out.stdout[-2000:]
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["unit"] == "env-steps/s" and d["higher_is_better"] is True and d["value"] > 0
    assert "workload" in d["config"] and d["vs_baseline"] is None
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


@pytest.mark.gpu
def test_our_arm_line(cuda_device):
    d = _run(["--steps", "4", "--warmup", "3", "--envs-per-gpu", "512"])
    assert BASE_KEYS <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] >= 3 and d["gpu_launches"] >= 4
    assert d["dtype"] == "f32" and d["data"] == "synthetic" and d["scaling"] == "weak"
    assert d["e2e"]["h2d_bytes_per_step"] == 512 * 80 * 4 and d["e2e"]["d2h_bytes_per_step"] > 0
    assert d["e2e"]["value"] > 0 and d["e2e"]["value"] != d["value"]
    rf = d["roofline"]
    for key in ("bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert key in rf
    assert 0 < rf["frac"] < 1.5
    assert {"sm_mhz", "sm_max_mhz", "reasons"} <= set(d["clocks"])
    cb = d["cpu_baseline"]
    assert cb["kind"] == "port" and cb["cores"] >= 1 and cb["value"] > 0


DUMPED = {"yaw": (80,), "wind_speed": (80,), "wind_direction": (80,), "power": (80,), "load": (80, 4), "reward": (),
          "freewind": (2,), "truncated": ()}


@pytest.mark.gpu
def test_dump_outputs_repeat_run_to_run(cuda_device, tmp_path):
    """--dump-outputs writes the last timed step's outputs; the inputs are seeded, so a second run writes the same arrays."""
    runs = []
    for name in ("a", "b"):
        d = _run(["--steps", "3", "--warmup", "2", "--envs-per-gpu", "256", "--quick", "--no-cpu-baseline",
                  "--dump-outputs", str(tmp_path / name)])
        assert d["steps"] == 3
        assert sorted(os.listdir(tmp_path / name)) == sorted(f"{k}.npy" for k in DUMPED)
        runs.append({k: np.load(tmp_path / name / f"{k}.npy") for k in DUMPED})
    for k, shape in DUMPED.items():
        a, b = runs[0][k], runs[1][k]
        assert a.dtype == np.float32 and a.shape == (256,) + shape, (k, a.dtype, a.shape)
        assert np.array_equal(a, b), k
    assert np.all(runs[0]["power"] >= 0) and runs[0]["power"].max() > 0 and np.all(np.isfinite(runs[0]["reward"]))


def test_dump_outputs_samples_envs_over_the_size_limit(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", 20000)
    rng = np.random.default_rng(1)
    out = {"power": rng.random((300, 5)), "load": rng.random((300, 5, 4)).astype(np.float32),
           "truncated": (rng.random(300) < 0.5).astype(np.uint8)}
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), out)
    got = {k: np.load(tmp_path / "a" / f"{k}.npy") for k in ("power", "load", "truncated", "env_index")}
    assert sum(a.nbytes for a in got.values()) <= 20000
    idx = got["env_index"].astype(np.int64)
    assert got["env_index"].dtype == np.float64 and 0 < len(idx) < 300 and np.all(np.diff(idx) > 0)
    assert got["power"].dtype == np.float64 and np.array_equal(got["power"], out["power"][idx])
    assert got["load"].dtype == np.float32 and np.array_equal(got["load"], out["load"][idx])
    assert got["truncated"].dtype == np.float32 and np.array_equal(got["truncated"], out["truncated"][idx])
    assert np.array_equal(np.load(tmp_path / "b" / "env_index.npy"), got["env_index"])
