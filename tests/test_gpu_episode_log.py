"""Episode log on the GPU: every record equals what a host-side reconstruction of the episode gives, the fused rollout
logs exactly what K single steps log, logging perturbs nothing, and the ring / overflow / sharding contracts hold."""
import numpy as np
import pytest
import torch

import random_envs_b200 as random_envs

pytestmark = pytest.mark.gpu

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
SURVIVE = (0.1, 0.1, 1.0, 0.3)
FIELDS = ("xi", "final_state", "length", "truncated", "end_tick", "count")


def _dr_env(n, dtype="float32", seed=0, **kw):
    env = random_envs.RandomCartPoleVecEnv(n, dtype=dtype, seed=seed, **kw)
    env.set_dr_distribution("uniform", SEARCH)
    env.set_dr_training(True)
    return env


def _policy_actions(env, w, b):
    s = env.obs.double()
    acc = s @ torch.tensor(w, dtype=torch.float64, device=s.device) + b
    return (acc > 0).to(torch.uint8)


def _assert_logs_equal(a, b):
    for f in FIELDS:
        assert torch.equal(getattr(a, f), getattr(b, f)), f


def _assert_envs_equal(a, b):
    assert torch.equal(a.obs, b.obs) and torch.equal(a.get_task(), b.get_task())
    assert torch.equal(a.elapsed, b.elapsed) and torch.equal(a.episode, b.episode)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
@pytest.mark.parametrize("integrator", ["euler", "semi-implicit"])
def test_step_records_equal_a_host_reconstruction(dtype, integrator):
    """For every done env the record in slot (count - 1) mod R is the episode that just ended: the xi and elapsed
    snapshot taken before the step, the truncated flag of the step, its tick, and the state a twin env without
    auto-reset reaches from the same state, task and action."""
    n, R, K = 10000, 4, 200
    env = _dr_env(n, dtype, seed=3, max_episode_steps=40, kinematics_integrator=integrator)
    twin = random_envs.RandomCartPoleVecEnv(n, dtype=dtype, seed=3, auto_reset=False, max_episode_steps=0,
                                            kinematics_integrator=integrator)
    env.reset()
    log = env.start_episode_log(R)
    dones = torch.zeros(n, dtype=torch.int32, device="cuda")
    truncations = 0
    for _ in range(K):
        xi0, el0, st0, tick = env.get_task().clone(), env.elapsed.clone(), env.state.clone(), env._tick
        act = env.sample_actions().clone()
        twin.set_state(st0); twin.set_task(xi0)
        twin.step(act)
        _, _, done, info = env.step(act)
        dones += done.to(torch.int32)
        idx = done.nonzero().squeeze(1)
        slot = ((log.count[idx] - 1) % R).long()
        assert torch.equal(log.xi[slot, idx], xi0[idx])
        assert torch.equal(log.length[slot, idx], el0[idx] + 1)
        assert torch.equal(log.truncated[slot, idx], info["TimeLimit.truncated"][idx])
        assert bool((log.end_tick[slot, idx] == tick).all())
        assert torch.equal(log.final_state[slot, idx], twin.state[idx])
        truncations += int(info["TimeLimit.truncated"].sum())
    assert torch.equal(log.count, dones)
    assert int(dones.sum()) > 2 * truncations > 0             # both kinds of ending are covered


def _rollout_vs_steps(dtype, w, b, K, pre=0, R=8, n=5000, limit=60):
    fused, stepped = _dr_env(n, dtype, seed=4, max_episode_steps=limit), _dr_env(n, dtype, seed=4, max_episode_steps=limit)
    for e in (fused, stepped):
        e.reset()
        for _ in range(pre):
            e.step(e.sample_actions())
    lf, ls = fused.start_episode_log(R), stepped.start_episode_log(R)
    fused.rollout(w, b, K)
    for _ in range(K):
        stepped.step(stepped.sample_actions() if w is None else _policy_actions(stepped, w, b))
    _assert_envs_equal(fused, stepped)
    _assert_logs_equal(lf, ls)
    assert int(lf.count.sum()) > 0
    # two half rollouts == one full rollout
    halves = _dr_env(n, dtype, seed=4, max_episode_steps=limit)
    halves.reset()
    for _ in range(pre):
        halves.step(halves.sample_actions())
    lh = halves.start_episode_log(R)
    halves.rollout(w, b, K // 2); halves.rollout(w, b, K - K // 2)
    _assert_envs_equal(halves, fused)
    _assert_logs_equal(lh, lf)
    assert torch.equal(halves.stats_tensor, fused.stats_tensor)


@pytest.mark.parametrize("w,b", [((0.0, 0.0, 1.0, 0.0), 0.0), ((0.0, 0.0, 0.0, 0.0), 1.0), ((0.0, 0.0, 0.0, 0.0), -1.0),
                                 (SURVIVE, 0.0)])
def test_fp32_pair_rollout_logs_what_repeated_steps_log(w, b):
    _rollout_vs_steps("float32", w, b, K=150)


@pytest.mark.parametrize("w,b", [((0.0, 0.0, 1.0, 0.0), 0.0), (SURVIVE, 0.0)])
def test_fp64_rollout_logs_what_repeated_steps_log(w, b):
    _rollout_vs_steps("float64", w, b, K=150)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_random_policy_rollout_logs_what_step_with_sample_actions_logs(dtype):
    _rollout_vs_steps(dtype, None, 0.0, K=90, pre=100)         # ticks 100 .. 189 cross the 128-step action block


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_logging_does_not_perturb_the_run(dtype):
    plain, logged = _dr_env(3000, dtype, seed=8, max_episode_steps=50), _dr_env(3000, dtype, seed=8, max_episode_steps=50)
    logged.start_episode_log(2)
    for e in (plain, logged):
        e.reset()
        for _ in range(30):
            e.step(e.sample_actions())
        e.rollout(SURVIVE, 0.0, 70)
        e.rollout(None, 0.0, 70)
    _assert_envs_equal(plain, logged)
    assert torch.equal(plain.stats_tensor, logged.stats_tensor)
    # a detached log stays readable and is no longer written
    log = logged.episode_log
    logged.stop_episode_log()
    count = log.count.clone()
    for _ in range(40):
        logged.step(logged.sample_actions())
    assert logged.episode_log is None and torch.equal(log.count, count) and int(count.sum()) > 0


def test_unsupported_attribute_changes_with_a_log_attached_raise():
    """auto_reset and noisy are plain attributes: flipping them while a log is attached must not route silently to the
    logged entry points, which imply auto-reset and take no noise block."""
    env = _dr_env(512, seed=2)
    env.reset()
    log = env.start_episode_log(2)
    env.step(env.sample_actions())
    for attr, value in (("auto_reset", False), ("noisy", True)):
        setattr(env, attr, value)
        with pytest.raises(ValueError, match="episode log"):
            env.step(env.sample_actions())
        with pytest.raises(ValueError, match="episode log"):
            env.rollout(SURVIVE, 0.0, 5)
        setattr(env, attr, not value)
    env.step(env.sample_actions())
    env.auto_reset = False
    env.stop_episode_log()                                    # detaching always works
    env.step(env.sample_actions())
    assert env.episode_log is None and log.count.shape == (512,)


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_episodes_reproduce_episode_stats(dtype):
    env = _dr_env(4000, dtype, seed=6, max_episode_steps=100)
    env.reset()
    log = env.start_episode_log(64)
    env.rollout(None, 0.0, 300)
    env.rollout(SURVIVE, 0.0, 200)
    st = env.episode_stats()
    ep = log.episodes()
    ret = ep["length"].double()
    assert ep["length"].numel() == st["episodes"] > 0
    assert abs(float(ret.mean()) - st["mean_return"]) < 1e-9 and abs(float(ret.mean()) - st["mean_length"]) < 1e-9
    assert float(ret.min()) == st["min_return"] and float(ret.max()) == st["max_return"]
    assert bool((ep["length"] >= 1).all()) and bool((ep["length"] <= 100).all())
    # (env, chronological) order: env ids non-decreasing, end ticks increasing within an env
    ids, ticks = ep["env_id"], ep["end_tick"]
    assert bool((ids[1:] >= ids[:-1]).all())
    same = ids[1:] == ids[:-1]
    assert bool((ticks[1:][same] > ticks[:-1][same]).all())
    assert ep["xi"].shape == (ret.numel(), 4) and ep["final_state"].shape == (ret.numel(), 4)
    assert ep["truncated"].dtype == torch.bool and bool(ep["truncated"].any())


@pytest.mark.parametrize("R", [1, 3])
def test_ring_keeps_the_latest_episodes_and_overflow_raises(R):
    n, big = 2000, 64
    ring, full = _dr_env(n, seed=11, max_episode_steps=30), _dr_env(n, seed=11, max_episode_steps=30)
    lr, lf = ring.start_episode_log(R), full.start_episode_log(big)
    for e in (ring, full):
        e.reset()
        for _ in range(40):
            e.step(e.sample_actions())
        e.rollout(None, 0.0, 100)
    assert torch.equal(lr.count, lf.count)
    count = lf.count.long()
    assert int(count.max()) <= big and int(count.min()) > R
    env_idx = torch.arange(n, device="cuda")
    for j in range(R):
        # the latest episode c of each env with c % R == j
        c = count - 1 - ((count - 1 - j) % R)
        for f in ("xi", "final_state", "length", "truncated", "end_tick"):
            assert torch.equal(getattr(lr, f)[j], getattr(lf, f)[c, env_idx]), (j, f)
    with pytest.raises(OverflowError, match="overwrote %d episodes" % int((count - R).sum())):
        lr.episodes()
    lr.clear()
    assert int(lr.count.sum()) == 0 and lr.episodes()["length"].numel() == 0
    ring.step(ring.sample_actions())
    assert int(lr.count.sum()) > 0                             # still attached after clear()


@pytest.mark.parametrize("dtype", ["float32", "float64"])
def test_log_is_invariant_to_sharding_and_tile_ordering(dtype):
    def run(env):
        env.reset()
        log = env.start_episode_log(16)
        for _ in range(50):
            env.step(env.sample_actions())
        env.rollout(SURVIVE, 0.0, 60)
        env.rollout(None, 0.0, 60)
        return log.episodes()
    whole = run(_dr_env(6000, dtype, seed=9, max_episode_steps=45))
    a = run(_dr_env(1000, dtype, seed=9, env_id0=0, max_episode_steps=45))
    b = run(_dr_env(5000, dtype, seed=9, env_id0=1000, max_episode_steps=45))
    for k in whole:
        assert torch.equal(whole[k], torch.cat([a[k], b[k]])), k
    tiled = run(_dr_env(6000, dtype, seed=9, max_episode_steps=45, tile_ordering=True))
    untiled = run(_dr_env(6000, dtype, seed=9, max_episode_steps=45, tile_ordering=False))
    for k in whole:
        assert torch.equal(tiled[k], untiled[k]) and torch.equal(tiled[k], whole[k]), k


def test_robustness_map_over_a_task_grid():
    """set_task over a 16 x 16 (gravity, pole_length) grid, reset, one 500-step rollout with R = 1: every env reports
    its first episode under its own grid point (a survivor is truncated at step 500)."""
    g, l = torch.meshgrid(torch.linspace(2.0, 20.0, 16), torch.linspace(0.1, 1.0, 16), indexing="ij")
    grid = torch.stack([g.reshape(-1), torch.full((256,), 1.0), torch.full((256,), 0.1), l.reshape(-1)], 1)
    env = random_envs.RandomCartPoleVecEnv(256, seed=1)
    env.set_task(grid)
    env.reset()
    log = env.start_episode_log(1)
    env.rollout(SURVIVE, 0.0, 500)
    assert bool((log.count >= 1).all())
    first = log.count == 1
    assert bool((log.length[0] >= 1).all()) and bool((log.length[0] <= 500).all())
    assert torch.equal(log.xi[0][first], grid.to("cuda")[first])
    assert torch.equal(log.truncated[0], log.length[0] == 500)
