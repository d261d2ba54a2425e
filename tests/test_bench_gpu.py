"""bench.py --dump-outputs on the device: the last timed step's outputs equal the oracle's after the same number of steps
from the same seeds, and are identical from run to run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

from oracle import flappy_oracle as fo  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NAMES = ("reward", "terminal", "score", "env_index", "obs", "obs_env_index", "state")
ENVS, DECORRELATE, CHECKED = 4096, 200, 24


def _bench(out_dir, steps):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "2",
                        "--envs-per-gpu", str(ENVS), "--decorrelate", str(DECORRELATE), "--no-learner", "--no-cpu-baseline",
                        "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert r.returncode == 0, r.stderr[-2000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == steps
    return line, {n: np.load(os.path.join(out_dir, n + ".npy")) for n in NAMES}


def _check_against_oracle(line, d):
    """bench's env: GameState(seed=42), every step Bernoulli(0.5) actions from stream_word(1234, 1, env, step); all
    steps taken = the decorrelation steps + the warm-up steps + the timed steps"""
    T = DECORRELATE + line["warmup"] + line["steps"]
    assert d["reward"].shape == d["terminal"].shape == d["score"].shape == (ENVS,) and d["state"].shape == (ENVS, 16)
    assert np.array_equal(d["env_index"], np.arange(ENVS))
    assert d["obs"].shape == (512, 80, 80) and d["obs_env_index"].shape == (512,)
    want_obs = np.zeros(T, np.uint8)
    want_obs[-1] = 1
    for j in range(0, 512, 512 // CHECKED):
        e = int(d["obs_env_index"][j])
        acts = np.array([fo.stream_word(1234, 1, e, t) < 2**31 for t in range(T)], np.uint8)
        r, term, sc, st, obs = fo.OracleEnvs(1, seed=42, first_env_id=e).run(0, acts, want_obs)
        assert (d["reward"][e], d["terminal"][e], d["score"][e]) == (r[-1], term[-1], sc[-1]), e
        np.testing.assert_array_equal(d["state"][e], st[-1], err_msg=f"env {e}")
        np.testing.assert_array_equal(d["obs"][j], obs[0], err_msg=f"env {e}")


def test_dump_outputs_are_the_last_step_and_reproducible(tmp_path):
    torch = pytest.importorskip("torch")
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    (la, a), (_, b), (lc, c) = _bench(tmp_path / "a", 5), _bench(tmp_path / "b", 5), _bench(tmp_path / "c", 6)
    for n in NAMES:
        assert a[n].dtype == np.float32 and np.array_equal(a[n], b[n]), n
    _check_against_oracle(la, a)
    _check_against_oracle(lc, c)                  # one more --steps: the oracle one step further still agrees
