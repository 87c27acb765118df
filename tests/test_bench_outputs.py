"""bench.py --steps / --dump-outputs: exactly K timed steps, and what the last one returned written as .npy files that are
the same on every run with the same arguments (so that two builds can be compared output for output)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
import bench  # noqa: E402


def _load(d, name):
    return np.load(os.path.join(str(d), name + ".npy"))


def test_dump_outputs_writes_every_array_and_samples_the_same_rows_above_the_limit(tmp_path):
    n = 1000
    obs = torch.arange(4 * n, dtype=torch.float64).reshape(n, 4)
    arrays = {"obs": obs, "reward": torch.arange(n, dtype=torch.float64), "done": torch.zeros(n)}
    bench.dump_outputs(str(tmp_path / "all"), arrays)
    assert sorted(os.listdir(tmp_path / "all")) == ["done.npy", "obs.npy", "reward.npy"]
    assert np.array_equal(_load(tmp_path / "all", "obs"), obs.numpy())
    row_bytes = 4 * 8 + 8 + 4 + 8                 # obs, reward, done and the row index
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays, limit_bytes=100 * row_bytes)
    idx = _load(tmp_path / "a", "env_index")
    assert idx.dtype == np.float64 and idx.shape == (100,) and np.all(np.diff(idx) > 0)
    rows = idx.astype(np.int64)
    assert np.array_equal(_load(tmp_path / "a", "obs"), obs.numpy()[rows])
    assert np.array_equal(_load(tmp_path / "a", "reward"), rows.astype(np.float64))
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in os.listdir(tmp_path / "a")) <= 100 * row_bytes + 4 * 128
    for name in ("env_index", "obs", "reward", "done"):
        assert np.array_equal(_load(tmp_path / "a", name), _load(tmp_path / "b", name))


def _bench(out_dir, dtype, steps, warmup, envs, batches):
    cmd = [sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", str(warmup),
           "--envs", str(envs), "--batches", str(batches), "--dtype", dtype, "--no-extras", "--no-cpu-baseline",
           "--dump-outputs", str(out_dir)]
    res = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=600)
    assert res.returncode == 0, res.stderr[-3000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


@pytest.mark.gpu
def test_bench_times_k_steps_and_dumps_the_same_outputs_on_every_run(tmp_path):
    a = _bench(tmp_path / "a", "float32", 7, 2, 8192, 3)
    b = _bench(tmp_path / "b", "float32", 7, 2, 8192, 3)
    assert a["steps"] == a["timing"]["steps_timed"] == a["gpu_launches"] == 7
    assert sorted(os.listdir(tmp_path / "a")) == ["done.npy", "obs.npy", "reward.npy"]
    obs, reward, done = (_load(tmp_path / "a", name) for name in ("obs", "reward", "done"))
    assert obs.shape == (8192, 4) and obs.dtype == np.float32 and reward.dtype == np.float32 and done.dtype == np.float32
    for name in ("obs", "reward", "done"):
        assert np.array_equal(_load(tmp_path / "a", name), _load(tmp_path / "b", name)), name


@pytest.mark.gpu
def test_bench_dump_is_the_last_timed_step_of_its_batch(tmp_path):
    """The dump equals the C oracle run through bench.py's seeded schedule for batch b = (K - 1) % R: reset at tick 0,
    the warm-up steps i = b, b + R, ... < max(W, 3) eagerly, then the K-step graph's steps i = b, b + R, ... < K, captured
    twice (single stream, then R branches) and each capture replayed twice with the ticks it was captured at.  Batch b
    holds envs [b n, (b + 1) n) with seed 0 and takes actions renv_random_actions_u8(seed 0, step (i // R) % 8)."""
    from oracle import c_oracle
    K, W, n, R = 7, 2, 4096, 3
    _bench(tmp_path, "float64", K, W, n, R)
    obs, reward, done = (_load(tmp_path, name) for name in ("obs", "reward", "done"))
    b = (K - 1) % R
    lo, hi = np.array(bench.SEARCH[0::2]), np.array(bench.SEARCH[1::2])
    ids = range(b * n, (b + 1) * n)
    st = np.ascontiguousarray(np.stack([c_oracle.init_state(0, i, 0) for i in ids]).T)
    xi = np.ascontiguousarray(np.stack([c_oracle.xi_uniform(0, i, 0, lo, hi) for i in ids]).T)
    el, ep = np.zeros(n, np.int32), np.ones(n, np.uint32)
    acts = [c_oracle.random_actions(n, b * n, 0, k) for k in range(8)]

    def run(tick0, steps):
        out = c_oracle.closed_loop(st, xi, el, ep, 0, b * n, tick0, len(steps), actions=np.stack(
            [acts[(i // R) % 8] for i in steps]), lo=lo, hi=hi, log=True)
        return out["done"][-1]

    warm, timed = list(range(b, max(W, 3), R)), list(range(b, K, R))
    if warm:
        run(1, warm)
    tick = 1 + len(warm)
    for _ in range(2):                      # the single-stream graph, then the R-branch graph: two replays each
        for _ in range(2):
            last_done = run(tick, timed)
        tick += len(timed)
    assert np.max(np.abs(obs - st.T)) <= 1e-9 and np.array_equal(done, last_done.astype(np.float32))
    assert np.all(reward == 1.0)
