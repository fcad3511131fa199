"""bench.py --dump-outputs (what the timed path returned in its last step, as .npy files by which two builds can be compared) and
the timed steps of the reference arm."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_dump_writes_every_output_whole_when_it_fits(tmp_path):
    arrays = {"obs": np.arange(40, dtype=np.float32).reshape(10, 4), "reward": np.ones(10, np.float32)}
    bench.dump_outputs(str(tmp_path / "d"), arrays)
    assert sorted(os.listdir(tmp_path / "d")) == ["obs.npy", "reward.npy"]
    for name, a in arrays.items():
        got = np.load(tmp_path / "d" / (name + ".npy"))
        assert got.dtype == a.dtype and np.array_equal(got, a)


def test_dump_samples_the_same_rows_of_every_output_within_the_limit(tmp_path):
    n, limit = 1000, 20000
    obs = np.arange(n * 6, dtype=np.float64).reshape(n, 6)
    reward = -np.arange(n, dtype=np.float64)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"obs": obs, "reward": reward}, limit=limit)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == ["env_index.npy", "obs.npy", "reward.npy"]
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= limit
    idx = np.load(tmp_path / "a" / "env_index.npy")
    assert idx.dtype == np.float64 and len(idx) > 100 and np.all(np.diff(idx) > 0)
    rows = idx.astype(np.int64)
    assert np.array_equal(np.load(tmp_path / "a" / "obs.npy"), obs[rows])
    assert np.array_equal(np.load(tmp_path / "a" / "reward.npy"), reward[rows])
    for f in files:                                    # a fixed seed: the same sample on every run
        assert np.array_equal(np.load(tmp_path / "a" / f), np.load(tmp_path / "b" / f))


def _bench(cwd, *args):
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True, cwd=str(cwd))


def test_reference_arm_times_steps_env_steps_per_core(tmp_path):
    p = _bench(tmp_path, "--impl", "reference", "--steps", "30", "--warmup", "2")
    assert p.returncode == 0, p.stderr[-3000:]
    line = json.loads(p.stdout)
    cores = line["cpu_baseline"]["cores"]
    assert line["steps"] == 30 and line["warmup"] == 2 and line["config"]["timed_env_steps"] == 30 * cores
    assert line["value"] > 0 and line["ms_per_step"] > 0


def test_dump_outputs_is_refused_for_the_reference_arm(tmp_path):
    p = _bench(tmp_path, "--impl", "reference", "--dump-outputs", str(tmp_path / "d"))
    assert p.returncode == 2 and "does not apply" in p.stderr and not (tmp_path / "d").exists()


@pytest.mark.gpu
def test_bench_dump_outputs_are_reproducible_and_follow_steps(tmp_path):
    """The dump is what the last timed step returned: a run whose e2e leg steps the batch further afterwards dumps the same
    outputs as one without that leg.  One more timed step changes them."""
    def run(steps, d, *extra):
        p = _bench(tmp_path, "--gpus", "1", "--steps", str(steps), "--warmup", "3", "--settle", "40", "--envs-per-gpu", "512",
                   "--no-cpu-baseline", "--no-extra", "--dump-outputs", str(tmp_path / d), *extra)
        assert p.returncode == 0, p.stderr[-3000:]
        line = json.loads(p.stdout)
        return line, {f[:-4]: np.load(tmp_path / d / f) for f in os.listdir(tmp_path / d)}

    la, a = run(5, "a")
    lb, b = run(5, "b", "--no-e2e")
    lc, c = run(6, "c", "--no-e2e")
    assert la["e2e"]["steps"] >= 10 and lb["e2e"] is None
    assert la["steps"] == 5 and lc["steps"] == 6
    assert sorted(a) == ["obs", "reward", "terminated", "truncated"]
    assert a["obs"].shape == (512, 24) and all(a[k].shape == (512,) for k in ("reward", "terminated", "truncated"))
    assert all(x.dtype == np.float32 for x in a.values()) and np.isfinite(a["obs"]).all()
    for k in a:
        assert np.array_equal(a[k], b[k]), k
    assert not np.array_equal(a["obs"], c["obs"])
