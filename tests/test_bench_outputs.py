"""bench.py --dump-outputs: what the timed step computed, written so that two builds can be compared output for output."""
import os
import subprocess
import sys

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_dump_outputs_writes_float_arrays_and_samples_within_the_limit(tmp_path):
    rng = np.random.default_rng(3)
    arrays = {"obs": rng.standard_normal((1000, 2, 60)).astype(np.float32), "reward": rng.standard_normal((1000, 2)),
              "term": rng.integers(0, 2, (1000, 3)).astype(np.uint8)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    full = _load(tmp_path / "all")
    assert sorted(full) == ["env_index", "obs", "reward", "term"]
    assert full["obs"].dtype == np.float32 and full["reward"].dtype == np.float64 and full["term"].dtype == np.float32
    assert np.array_equal(full["env_index"], np.arange(1000)) and np.array_equal(full["term"], arrays["term"])
    limit = 200_000
    for name in ("a", "b"):
        bench.dump_outputs(str(tmp_path / name), arrays, limit=limit)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= limit
    rows = a["env_index"].astype(np.int64)
    assert 0 < len(rows) < 1000 and np.all(np.diff(rows) > 0)
    assert all(np.array_equal(a[k], b[k]) for k in a)   # the sample is fixed
    assert np.array_equal(a["obs"], arrays["obs"][rows]) and np.array_equal(a["reward"], arrays["reward"][rows])


@pytest.mark.gpu
def test_bench_dump_is_reproducible_and_follows_steps(tmp_path):
    env = dict(os.environ, MJB_BENCH_ENVS="256", MJB_BENCH_SETTLE="5")

    def run(name, steps):
        out = tmp_path / name
        cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1", "--no-cpu", "--no-configs",
               "--dump-outputs", str(out)]
        res = subprocess.run(cmd, env=env, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, res.stdout + res.stderr
        return _load(out)

    a, b, c = run("a", 3), run("b", 3), run("c", 4)
    assert sorted(a) == ["env_index", "obs", "reward", "term", "trunc"]
    assert a["obs"].shape == (256, 2, 60) and a["reward"].shape == (256, 2) and a["term"].shape == a["trunc"].shape == (256, 3)
    assert all(v.dtype == np.float32 for k, v in a.items() if k != "env_index")
    assert np.isfinite(a["obs"]).all() and set(np.unique(a["term"])) <= {0.0, 1.0}
    assert all(np.array_equal(a[k], b[k]) for k in a)   # same arguments, same inputs, same outputs
    assert not np.array_equal(a["obs"], c["obs"])        # one more timed step moves the state on
