"""bench.py --dump-outputs: what the last timed step computed, identical from run to run with the same arguments, and
--steps taken as given."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")
pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUTPUTS = ("agent", "target", "best_dir", "reward", "terminated", "truncated")


def _bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--no-extras", "--no-cpu-baseline",
                          "--e2e-steps", "3", *args], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    return json.loads(lines[0])


def _load(d):
    return {f[:-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d))}


def test_headline_dump_is_a_fixed_sample_and_repeats_bit_for_bit(tmp_path):
    """The default 4 096 000 envs are more than 64 MB of outputs: a seeded sample of envs, the same in both runs."""
    runs = []
    for name in ("a", "b"):
        line = _bench("--steps", "7", "--warmup", "3", "--dump-outputs", str(tmp_path / name))
        assert line["steps"] == 7 and line["gpu_launches"] == 7
        runs.append(_load(tmp_path / name))
    a, b = runs
    assert set(a) == set(OUTPUTS) | {"rows"}
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 64 * 10**6
    rows = a["rows"].astype(np.int64)
    assert (np.diff(rows) > 0).all() and rows[0] >= 0 and rows[-1] < 4096000 and len(rows) > 10**6
    for k in a:
        assert a[k].dtype in (np.float32, np.float64) and len(a[k]) == len(rows), k
        np.testing.assert_array_equal(a[k], b[k], err_msg=k)
    assert a["reward"].dtype == np.float64
    assert ((a["agent"] >= 0) & (a["agent"] < 81)).all() and ((a["target"] >= 0) & (a["target"] < 81)).all()
    assert np.isin(a["terminated"], (0, 1)).all() and np.isin(a["truncated"], (0, 1)).all()
    # best dir = agent - next cell on the shortest path: one step along one axis, or (0, 0) on the goal
    assert np.isin(np.abs(a["best_dir"]).sum(1), (0, 1)).all()


def test_steps_are_taken_as_given_and_a_small_batch_is_dumped_whole(tmp_path):
    """--steps 2000 --warmup 500 equal the configs1 defaults; another workload still runs exactly that many steps."""
    line = _bench("--workload", "toroidal-regen", "--envs-per-gpu", "4096", "--steps", "2000", "--warmup", "500",
                  "--dump-outputs", str(tmp_path / "d"))
    assert line["steps"] == 2000 and line["gpu_launches"] == 2000 * 4
    d = _load(tmp_path / "d")
    assert set(d) == set(OUTPUTS)
    assert all(len(v) == 4096 for v in d.values())
