"""bench.py keeps the driver's contract: one JSON line with the agreed keys, for both arms."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BASE_KEYS = {"metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better", "scaling",
             "vs_baseline", "dtype", "data", "config", "e2e", "gpu_launches", "cpu_baseline"}


def _run(args, timeout):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                         timeout=timeout, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    return json.loads(lines[0])


def test_reference_arm_line():
    d = _run(["--impl", "reference", "--steps", "1", "--warmup", "0"], 300)
    assert d["impl"] == "reference" and BASE_KEYS <= set(d)
    assert d["metric"] == "candidate schedules/sec" and d["unit"] == "candidates/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["e2e"]["value"] == d["value"] and d["e2e"]["h2d_bytes_per_step"] == 0
    assert d["steps"] == 1
    assert d["cpu_baseline"]["kind"] == "port" and d["cpu_baseline"]["cores"] >= 1 and d["gpu_launches"] == 0
    assert "workload" in d["config"] and "model" not in d["config"]
    # both arms print the same `config` object for the headline run
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.static_config(True)
    assert d["cpu_baseline"]["cores"] <= (os.cpu_count() or 1) and "physical cores" in d["run"]["cores_how"]


@pytest.mark.gpu
def test_our_arm_line():
    d = _run(["--steps", "4", "--warmup", "3", "--batch", str(148 * 16 * 32 * 2), "--no-cpu"], 600)
    assert BASE_KEYS <= set(d) and {"roofline", "clocks"} <= set(d)
    assert d["metric"] == "candidate schedules/sec" and d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] >= 3
    assert d["scaling"] == "weak" and d["vs_baseline"] is None and d["dtype"] == "f32" and d["data"] == "synthetic"
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and 0 < r["frac"] < 1.2 and r["peak"] > 1000
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9
    assert d["e2e"]["h2d_bytes_per_step"] > 0 and d["e2e"]["d2h_bytes_per_step"] > 0 and d["e2e"]["value"] > 0
    assert d["gpu_launches"] == 4 and d["value"] > 1e8
    assert set(d["clocks"]) >= {"sm_mhz", "sm_max_mhz", "reasons"}
    sys.path.insert(0, ROOT)
    import bench
    assert d["config"] == bench.static_config(True)
    assert d["e2e"]["candidates_per_gpu_per_step"] == d["run"]["candidates_per_gpu_per_step"]   # same batch as `value`


def test_bad_arguments_are_refused(tmp_path):
    for args in (["--steps", "0"], ["--impl", "reference", "--dump-outputs", str(tmp_path)]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, capture_output=True, text=True,
                             timeout=120, cwd=ROOT)
        assert out.returncode == 2 and "error" in out.stderr, args
    assert not any(tmp_path.iterdir())


@pytest.mark.gpu
def test_dump_outputs(tmp_path):
    """--dump-outputs writes the last timed step's makespans and arg-min; the inputs are seeded, so runs with a
    different step count produce the same arrays."""
    import numpy as np
    B = 148 * 16 * 32 * 2
    runs = []
    for steps in (2, 5):
        d = _run(["--steps", str(steps), "--warmup", "3", "--batch", str(B), "--no-cpu", "--no-e2e",
                  "--dump-outputs", str(tmp_path / str(steps))], 600)
        assert d["steps"] == steps and d["gpu_launches"] == steps
        runs.append({n: np.load(tmp_path / str(steps) / (n + ".npy"))
                     for n in ("makespan", "candidate_id", "best_makespan", "best_candidate_id")})
    a, b = runs
    assert a["makespan"].dtype == np.float32 and a["candidate_id"].dtype == np.float64
    assert a["makespan"].shape == (B,) and np.array_equal(a["candidate_id"], np.arange(B))
    assert np.isfinite(a["makespan"]).all() and a["best_makespan"][0] == a["makespan"].min()
    assert a["makespan"][int(a["best_candidate_id"][0])] == a["best_makespan"][0]
    assert sum(x.nbytes for x in a.values()) <= 64 << 20
    for n in a:
        assert np.array_equal(a[n], b[n]), n
