"""bench.dump_outputs with stand-ins for the device objects: a batch above the row limit is cut to a fixed, sorted sample
of envs, every per-env array keeps the same rows, and everything is written as float32 / float64."""
import os
import types

import numpy as np

import bench


class _Host:
    def __init__(self, a):
        self.a = a

    def cpu(self):
        return self

    def numpy(self):
        return self.a


class _Env:
    n = 1000

    def get_state(self):
        out = {k: np.arange(self.n, dtype=np.float64) for k in ("px", "py", "pz", "vx", "vy", "V", "score", "total_score",
                                                                  "path_len", "reward64")}
        out.update({k: np.arange(self.n, dtype=np.int32) for k in ("step", "cursor", "scenario")})
        out["done"] = (np.arange(self.n) % 2).astype(np.uint8)
        return out

    def observe(self):
        return _Host(np.repeat(np.arange(self.n, dtype=np.float32)[:, None], 100, 1))


class _Learner:
    def get_params(self, which):
        return np.full(50, which, np.float32)

    def counters(self):
        return 9, 8


def _load(d):
    return {f[:-len(".npy")]: np.load(os.path.join(d, f)) for f in os.listdir(d)}


def test_dump_outputs_samples_envs_above_the_limit(tmp_path):
    wl = types.SimpleNamespace(env=_Env(), L=_Learner())
    bench.dump_outputs(wl, str(tmp_path / "a"), max_envs=300)
    bench.dump_outputs(wl, str(tmp_path / "b"), max_envs=300)
    a, b = _load(tmp_path / "a"), _load(tmp_path / "b")
    rows = a["env_index"]
    assert rows.shape == (300,) and np.all(np.diff(rows) > 0) and np.array_equal(rows, b["env_index"])
    for k, v in a.items():
        assert v.dtype in (np.float32, np.float64), k
        if k.startswith("env_") and k not in ("env_done", "env_obs"):
            assert np.array_equal(v, rows), k
    assert np.array_equal(a["env_obs"], np.repeat(rows.astype(np.float32)[:, None], 100, 1))
    assert np.array_equal(a["env_done"], rows % 2)
    assert np.array_equal(a["learner_grad"], np.full(50, 4, np.float32)) and a["learner_counters"].tolist() == [9, 8]


def test_dump_outputs_keeps_small_batches_whole(tmp_path):
    bench.dump_outputs(types.SimpleNamespace(env=_Env(), L=_Learner()), str(tmp_path))
    a = _load(tmp_path)
    assert np.array_equal(a["env_index"], np.arange(1000)) and a["env_obs"].shape == (1000, 100)
