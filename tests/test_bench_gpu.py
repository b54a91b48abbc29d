"""bench.py --dump-outputs on the device: what the last timed step computed depends on the arguments alone (two runs write
bit-identical files) and follows exactly max(--warmup, 3) + --steps lockstep iterations with one update each."""
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT

pytestmark = pytest.mark.gpu

ARGS = ["--gpus", "1", "--steps", "7", "--warmup", "4", "--envs", "256", "--replay", "4096", "--pool", "64",
        "--no-e2e", "--no-configs", "--no-cpu-baseline"]


def _dump(out_dir):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + ARGS + ["--dump-outputs", str(out_dir)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-3000:]
    return {f[:-len(".npy")]: np.load(os.path.join(out_dir, f)) for f in sorted(os.listdir(out_dir))}


def test_bench_dump_outputs_reproducible(tmp_path):
    a, b = _dump(tmp_path / "a"), _dump(tmp_path / "b")
    assert sorted(a) == sorted(b)
    for k in a:
        assert a[k].dtype in (np.float32, np.float64), k
        assert np.array_equal(a[k], b[k]), k
    assert a["env_obs"].shape == (256, 100) and a["env_px"].shape == (256,) and np.isfinite(a["learner_q_local"]).all()
    assert a["learner_counters"].tolist() == [4 + 7, 4 + 7]          # epochs, Adam steps
