"""The bench.py output contract (one JSON line on stdout, the keys the driver reads) for both arms."""
import json
import pathlib
import subprocess
import sys

import pytest

ROOT = pathlib.Path(__file__).resolve().parent.parent
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling", "vs_baseline",
             "dtype", "data", "config", "e2e", "cpu_baseline"}


def _run(args, timeout):
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), *args], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [l for l in res.stdout.splitlines() if l.strip()]
    assert len(lines) == 1, lines                       # exactly ONE line on stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"], 600)
    assert BASE_KEYS <= set(d) and d["impl"] == "reference"
    assert d["metric"] == "env_steps_per_sec_incl_q_updates" and d["unit"] == "env-steps/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and "workload" in d["config"]


@pytest.mark.gpu
def test_our_arm_line():
    d = _run(["--steps", "3", "--warmup", "3", "--no-extra"], 900)
    assert BASE_KEYS | {"roofline", "gpu_launches", "clocks"} <= set(d) and "impl" not in d
    assert d["n_gpus"] == 1 and d["steps"] == 3 and d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f32"
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and r["traffic"]
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 0
    assert d["gpu_launches"] > 0 and d["cpu_baseline"]["cores"] == 1 and d["cpu_baseline"]["kind"] == "port"
    assert d["value"] > 1e9 and "workload" in d["config"]


def test_steps_must_be_positive():
    res = subprocess.run([sys.executable, str(ROOT / "bench.py"), "--steps", "0"], capture_output=True, text=True, timeout=120, cwd=ROOT)
    assert res.returncode == 2 and "--steps" in res.stderr


@pytest.mark.gpu
def test_dump_outputs_repeatable(tmp_path):
    """--dump-outputs: float32 / float64 arrays, 64 MB at most, the same arrays from two runs with the same arguments, and trainer
    state that counts exactly the ramp, warm-up and --steps global steps."""
    import numpy as np
    import bench
    runs = [tmp_path / "a", tmp_path / "b"]
    for d in runs:
        assert _run(["--steps", "2", "--warmup", "3", "--no-extra", "--no-cpu", "--dump-outputs", str(d)], 900)["steps"] == 2
    names = sorted(p.name for p in runs[0].iterdir())
    assert {"q_a.npy", "q_b.npy", "count.npy", "env_body.npy", "population_total_steps.npy"} <= set(names)
    assert names == sorted(p.name for p in runs[1].iterdir()) and sum(p.stat().st_size for p in runs[0].iterdir()) <= 64 << 20
    for n in names:
        a, b = np.load(runs[0] / n), np.load(runs[1] / n)
        assert a.dtype in (np.float32, np.float64) and np.array_equal(a, b, equal_nan=True), n
    steps = np.load(runs[0] / "population_total_steps.npy")
    assert np.all(steps == bench.ENVS_PER_POPULATION * (32 * bench.RAMP_LAUNCHES + 3 + 2)) and np.load(runs[0] / "count.npy").sum() > 0
