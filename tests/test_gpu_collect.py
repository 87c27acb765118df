"""Trajectory collection on the GPU: sampled actions against the host Philox oracle and float64 logits, calibration,
collect(K) against K x {obs; policy_actions(sample, return_logp); step} bit for bit, the episode log, greedy collect
against rollout(policy), chaining, sharding and buffer reuse, and the rejections."""
import math

import numpy as np
import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from oracle import c_oracle
from random_envs_b200 import MLPPolicy

pytestmark = pytest.mark.gpu

PURPOSE_POLICY_SAMPLE = 5          # include/renv.h: Philox purpose of the MLP policy's sampled action
SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
BOX = torch.tensor([2.4, 3.0, 0.21, 3.5])
TRAJ_FIELDS = ("obs", "actions", "logp", "dones", "truncated")


def _net(act=nn.Tanh, h1=64, h2=64, o=2, scale=1.0, seed=0):
    torch.manual_seed(seed)
    net = nn.Sequential(nn.Linear(4, h1), act(), nn.Linear(h1, h2), act(), nn.Linear(h2, o))
    with torch.no_grad():
        for p in net.parameters():
            p.mul_(scale)
    return net


def _env(n, seed=0, dr="uniform", **kw):
    env = random_envs.RandomCartPoleVecEnv(n, seed=seed, **kw)
    if dr == "uniform":
        env.set_dr_distribution("uniform", SEARCH)
    elif dr == "truncnorm":
        env.set_dr_distribution("truncnorm", [9.8, 1.0, 1.0, 0.2, 0.1, 0.03, 0.5, 0.1])
    env.set_dr_training(dr is not None)
    return env


def _mid_episode_start(envs, n, max_steps, seed=11):
    g = torch.Generator(device="cuda").manual_seed(seed)
    mid = (torch.rand((n, 4), generator=g, device="cuda") * 2 - 1) * BOX.cuda() * 0.5
    el = torch.randint(0, max_steps, (n,), generator=g, device="cuda")
    for e in envs:
        e.reset()
        e.set_state(mid, elapsed=el)


def _assert_envs_equal(a, b):
    assert torch.equal(a.state, b.state) and torch.equal(a.get_task(), b.get_task())
    assert torch.equal(a.elapsed, b.elapsed) and torch.equal(a.episode, b.episode) and a._tick == b._tick


def _stepped(env, policy, K, sample):
    """K x {obs; policy_actions(sample, return_logp); step}: the trajectory collect(K) must record, and the statistics
    a rollout accumulates over the episodes that end."""
    rows = {f: [] for f in TRAJ_FIELDS}
    stats = [0.0, 0.0, 0.0, math.inf, -math.inf, 0.0]
    for _ in range(K):
        rows["obs"].append(env.obs.clone())
        el0 = env.elapsed.clone()
        actions, logp = env.policy_actions(policy, sample=sample, return_logp=True)
        rows["actions"].append(actions.clone())
        rows["logp"].append(logp.clone())
        _, _, done, info = env.step(actions)
        rows["dones"].append(done.clone())
        rows["truncated"].append(info["TimeLimit.truncated"].clone())
        r = (el0 + 1)[done].double()
        if len(r):
            stats[0] += len(r); stats[1] += float(r.sum()); stats[2] += float((r * r).sum())
            stats[3] = min(stats[3], float(r.min())); stats[4] = max(stats[4], float(r.max())); stats[5] += float(r.sum())
    return {f: torch.stack(v) for f, v in rows.items()}, stats


def _log_sigmoid64(d):
    return -torch.nn.functional.softplus(-d)


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
@pytest.mark.parametrize("o", [2, 1])
@pytest.mark.parametrize("scale", [1.0, 4.0])
def test_sampled_actions_and_logp_against_the_host_oracle(act, o, scale):
    n, K, seed, env_id0 = 8192, 24, 21, 1000
    net = _net(act, 64, 64, o, scale, seed=o + int(scale))
    policy = MLPPolicy.from_module(net, "cuda")
    env = _env(n, seed, max_episode_steps=15, env_id0=env_id0)
    env.reset()
    traj = env.collect(policy, K, sample=True)
    g = torch.Generator().manual_seed(3)
    ks, iis = torch.randint(0, K, (4000,), generator=g), torch.randint(0, n, (4000,), generator=g)
    obs = traj.obs[ks.cuda(), iis.cuda()]
    l64 = policy.reference_logits(obs).cpu()
    d64 = l64[:, 1] - l64[:, 0]
    p64 = torch.sigmoid(d64)
    u = torch.tensor([float(c_oracle.uniforms(seed, env_id0 + int(i), traj.tick0 + int(k), PURPOSE_POLICY_SAMPLE, 0, 1,
                                              np.float32)[0]) for k, i in zip(ks, iis)], dtype=torch.float64)
    actions = traj.actions[ks.cuda(), iis.cuda()].cpu()
    logp = traj.logp[ks.cuda(), iis.cuda()].cpu().double()
    big = max(1.0, float(l64.abs().max()))
    clear = (u - p64).abs() > 1e-5 * big + 1e-6
    assert int(clear.sum()) > 3900
    assert torch.equal(actions[clear], (u < p64)[clear].to(torch.uint8))
    logp64 = torch.where(actions == 1, _log_sigmoid64(d64), _log_sigmoid64(-d64))
    err = float((logp - logp64).abs().max())
    assert err <= 2e-5 * big + 1e-6, (err, big)
    assert bool((traj.logp <= 0).all())


def test_sampled_actions_are_calibrated_over_the_whole_buffer():
    n, K = 1 << 20, 4
    policy = MLPPolicy.from_module(_net(nn.Tanh, seed=2), "cuda")
    env = _env(n, 5)
    env.reset()
    traj = env.collect(policy, K, sample=True)
    with torch.no_grad():
        l64 = policy.reference_logits(traj.obs.reshape(-1, 4))
    p64 = torch.sigmoid(l64[:, 1] - l64[:, 0])
    got = float(traj.actions.double().sum())
    want, sd = float(p64.sum()), math.sqrt(float((p64 * (1 - p64)).sum()))
    assert abs(got - want) <= 6 * sd, (got, want, sd)
    assert 0.05 < want / p64.numel() < 0.95                  # a policy that really samples both actions


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
@pytest.mark.parametrize("dr", ["uniform", "truncnorm"])
@pytest.mark.parametrize("integrator", ["euler", "semi-implicit"])
@pytest.mark.parametrize("sample", [True, False])
def test_collect_equals_k_steps_of_sampled_policy_actions(act, dr, integrator, sample):
    n, K, max_steps = 5000 + 37, 120, 40          # not a multiple of 32 or 128
    policy = MLPPolicy.from_module(_net(act, 48, 64, 2, scale=2.0, seed=3), "cuda")
    fused, stepped = (_env(n, 5, dr, max_episode_steps=max_steps, kinematics_integrator=integrator) for _ in range(2))
    _mid_episode_start((fused, stepped), n, max_steps)
    traj = fused.collect(policy, K, sample=sample)
    want, stats = _stepped(stepped, policy, K, sample)
    for f in TRAJ_FIELDS:
        assert torch.equal(getattr(traj, f), want[f]), f
    assert traj.num_steps == K and traj.tick0 == stepped._tick - K
    assert bool(traj.dones.any()) and bool(traj.truncated.any()) and bool((traj.dones & ~traj.truncated).any())
    _assert_envs_equal(fused, stepped)
    assert torch.equal(fused.obs, stepped.obs)
    assert fused.stats_tensor.tolist() == stats and stats[0] > n


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
def test_collect_agrees_with_the_episode_log(act):
    n, K, R = 4000, 150, 64
    policy = MLPPolicy.from_module(_net(act, 64, 32, 1, seed=8), "cuda")
    fused, stepped = (_env(n, 2, max_episode_steps=10) for _ in range(2))       # terminations and truncations
    for e in (fused, stepped):
        e.reset()
    lf, ls = fused.start_episode_log(R), stepped.start_episode_log(R)
    traj = fused.collect(policy, K, sample=True)
    _, stats = _stepped(stepped, policy, K, True)
    for f in ("xi", "final_state", "length", "truncated", "end_tick", "count"):
        assert torch.equal(getattr(lf, f), getattr(ls, f)), f
    _assert_envs_equal(fused, stepped)
    assert fused.stats_tensor.tolist() == stats
    ep = lf.episodes()                                             # (env, chronological) order
    env_k = traj.dones.t().nonzero()                              # (E, 2): env, step -- the same order
    assert len(env_k) == len(ep["length"]) > n and bool(ep["truncated"].any())
    i, k = env_k[:, 0], env_k[:, 1]
    assert torch.equal(ep["end_tick"], traj.tick0 + k)
    assert torch.equal(traj.final_obs[k, i], ep["final_state"])
    assert torch.equal(traj.truncated[k, i], ep["truncated"])
    first = torch.ones_like(i, dtype=torch.bool)
    first[1:] = i[1:] != i[:-1]
    prev = torch.where(first, torch.full_like(k, -1), torch.roll(k, 1))
    assert torch.equal((k - prev).to(torch.int32), ep["length"])   # every env starts at elapsed 0 after reset()


def test_greedy_collect_equals_policy_actions_and_rollout():
    n, K = 3000, 150
    policy = MLPPolicy.from_module(_net(nn.ReLU, seed=4, scale=2.0), "cuda")
    fused, rolled, stepped = (_env(n, 6, max_episode_steps=30) for _ in range(3))
    _mid_episode_start((fused, rolled, stepped), n, 30)
    lf, lr = fused.start_episode_log(8), rolled.start_episode_log(8)
    traj = fused.collect(policy, K, sample=False)
    rolled.rollout(policy, 0.0, K)
    for k in range(K):
        actions = stepped.policy_actions(policy)                  # today's argmax kernel
        assert torch.equal(traj.actions[k], actions), k
        stepped.step(actions)
    _assert_envs_equal(fused, rolled)
    _assert_envs_equal(fused, stepped)
    assert torch.equal(fused.stats_tensor, rolled.stats_tensor)
    for f in ("xi", "final_state", "length", "truncated", "end_tick", "count"):
        assert torch.equal(getattr(lf, f), getattr(lr, f)), f


def _copy(traj):
    out = {f: getattr(traj, f).clone() for f in TRAJ_FIELDS}
    out["final_obs"] = torch.where(traj.dones[..., None], traj.final_obs, torch.zeros_like(traj.final_obs))
    return out


def test_chained_sharded_and_reused_collects_equal_one_collect():
    n, K1, K2 = 3000, 35, 55
    policy = MLPPolicy.from_module(_net(nn.Tanh, seed=5), "cuda")
    whole, chained, reused = (_env(n, 9, max_episode_steps=60) for _ in range(3))
    halves = [_env(n // 2, 9, max_episode_steps=60, env_id0=k * (n // 2)) for k in range(2)]
    for e in [whole, chained, reused] + halves:
        e.reset()
    w = _copy(whole.collect(policy, K1 + K2))
    c = [_copy(chained.collect(policy, K)) for K in (K1, K2)]
    for f in w:
        assert torch.equal(w[f], torch.cat([c[0][f], c[1][f]])), f
    _assert_envs_equal(whole, chained)
    assert torch.equal(whole.stats_tensor, chained.stats_tensor)
    buf = reused.trajectory_buffer(K1 + K2)
    r = [_copy(reused.collect(policy, K, out=buf)) for K in (K1, K2)]
    for f in w:
        assert torch.equal(torch.cat([r[0][f], r[1][f]]), w[f]), f
    _assert_envs_equal(whole, reused)
    h = [_copy(e.collect(policy, K1 + K2)) for e in halves]
    for f in w:
        assert torch.equal(torch.cat([h[0][f], h[1][f]], dim=1), w[f]), f
    assert torch.equal(torch.cat([e.state for e in halves]), whole.state)
    assert torch.equal(torch.cat([e.get_task() for e in halves]), whole.get_task())


def test_buffers_without_logp_or_final_obs():
    n, K = 1000, 40
    policy = MLPPolicy.from_module(_net(nn.Tanh, seed=6), "cuda")
    a, b = _env(n, 3, max_episode_steps=20), _env(n, 3, max_episode_steps=20)
    for e in (a, b):
        e.reset()
    full = a.collect(policy, K)
    slim = b.collect(policy, K, out=b.trajectory_buffer(K, logp=False, final_obs=False))
    assert slim.logp is None and slim.final_obs is None
    for f in ("obs", "actions", "dones", "truncated"):
        assert torch.equal(getattr(full, f), getattr(slim, f)), f
    _assert_envs_equal(a, b)
    assert torch.equal(full.rewards, torch.ones((K, n), device="cuda"))


@pytest.mark.parametrize("kw", [dict(dtype="float64"), dict(noisy=True), dict(lean=True)])
def test_unsupported_envs_raise(kw):
    policy = MLPPolicy.from_module(_net(), "cuda")
    env = random_envs.RandomCartPoleVecEnv(64, **kw)
    env.reset()
    with pytest.raises(ValueError):
        env.collect(policy, 5)


def test_wrong_buffers_raise():
    policy = MLPPolicy.from_module(_net(), "cuda")
    env, other = random_envs.RandomCartPoleVecEnv(64), random_envs.RandomCartPoleVecEnv(96)
    env.reset()
    with pytest.raises(ValueError):
        env.collect(policy, 5, out=other.trajectory_buffer(5))
    with pytest.raises(ValueError):
        env.collect(policy, 6, out=env.trajectory_buffer(5))
    with pytest.raises(ValueError):
        env.collect(policy, 0)
    env.start_episode_log(2)
    env.auto_reset = False                     # the log's precondition no longer holds
    with pytest.raises(ValueError):
        env.collect(policy, 5)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="a policy on another device needs a second GPU")
def test_policy_or_buffer_on_another_device_raises():
    env = random_envs.RandomCartPoleVecEnv(64, device="cuda:0")
    env.reset()
    with pytest.raises(ValueError):
        env.collect(MLPPolicy.from_module(_net(), "cuda:1"), 5)
    far = random_envs.RandomCartPoleVecEnv(64, device="cuda:1")
    with pytest.raises(ValueError):
        env.collect(MLPPolicy.from_module(_net(), "cuda:0"), 5, out=far.trajectory_buffer(5))
