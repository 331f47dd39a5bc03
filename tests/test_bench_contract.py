"""CPU test of the bench.py contract: the reference arm (oracle port on host
threads) must print ONE JSON line with the keys the driver reads."""

import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_prints_one_json_line():
    env = dict(os.environ, OMP_NUM_THREADS="2")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=900, env=env)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [ln for ln in r.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    j = json.loads(lines[0])
    for k in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step",
              "higher_is_better", "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e"):
        assert k in j, k
    assert j["impl"] == "reference" and j["value"] > 0 and j["unit"] == "grid-cell-timesteps/s"
    assert j["cpu_baseline"]["kind"] == "port" and j["cpu_baseline"]["cores"] >= 1
    assert j["e2e"]["h2d_bytes_per_step"] == 0 and j["e2e"]["value"] == j["value"]
    assert "workload" in j["config"] and "1440x720x8760" in j["config"]["workload"]  # the north-star cutout
    assert j["scaling"] == "strong"


def test_reference_arm_other_ranks_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2",
                        "--steps", "1", "--warmup", "0"], capture_output=True, text=True, timeout=300, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.parametrize("argv", [["--steps", "0"], ["--warmup", "-1"],
                                  ["--impl", "reference", "--dump-outputs", "out"]])
def test_bad_arguments_are_refused(argv, tmp_path):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + argv, capture_output=True, text=True,
                       timeout=120, cwd=tmp_path)
    assert r.returncode == 2 and "error" in r.stderr
    assert not os.listdir(tmp_path)


def test_dump_outputs_fits_the_budget_with_a_fixed_sample(tmp_path, monkeypatch):
    import bench

    monkeypatch.setattr(bench, "DUMP_BYTES", 1 << 20)
    rng = np.random.default_rng(3)
    results = {"pv": rng.random((1000, 300)), "wind": rng.random((1000, 300), dtype=np.float32),
               "heat_demand": rng.random((40, 300), dtype=np.float32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), results)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == sorted(f"{k}{s}.npy" for k in results for s in ("", "_time_index"))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= bench.DUMP_BYTES
    for k, v in results.items():
        got, rows = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "a" / f"{k}_time_index.npy")
        assert got.dtype == np.float32 and rows.dtype == np.float64
        assert np.array_equal(got, v[rows.astype(np.int64)].astype(np.float32))
        assert np.array_equal(got, np.load(tmp_path / "b" / f"{k}.npy"))  # the same sample on every run
    assert len(np.load(tmp_path / "a" / "heat_demand_time_index.npy")) == 40  # small results stay whole
    assert 0 < len(np.load(tmp_path / "a" / "pv_time_index.npy")) < 1000
