"""Advantage estimation on the GPU: the kernel's values against policy_actions' logits bit for bit, its advantages and
returns against a float32 replay of the recurrence bit for bit and against float64 GAE within a derived bound,
independence from sharding and repetition, no side effects, and the rejections."""
import math

import numpy as np
import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from random_envs_b200 import MLPPolicy

pytestmark = pytest.mark.gpu

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
BOX = torch.tensor([2.4, 3.0, 0.21, 3.5])
GAMMA_LAMBDA = [(0.99, 0.95), (1.0, 1.0), (0.9, 0.0)]
U = 2.0 ** -24


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


def _mid_episode_start(env, n, max_steps, seed=11):
    g = torch.Generator(device="cuda").manual_seed(seed)
    mid = (torch.rand((n, 4), generator=g, device="cuda") * 2 - 1) * BOX.cuda() * 0.5
    el = torch.randint(0, max_steps, (n,), generator=g, device="cuda")
    env.reset()
    env.set_state(mid, elapsed=el)


def _collected(n, K, act=nn.Tanh, dr="uniform", sample=True, max_steps=20, seed=5, env_id0=0, mid=True):
    """An env and the trajectory of a K-step collect under a 2-output policy, starting mid-episode."""
    env = _env(n, seed, dr, max_episode_steps=max_steps, env_id0=env_id0)
    if mid:
        _mid_episode_start(env, n, max_steps)
    else:
        env.reset()
    policy = MLPPolicy.from_module(_net(act, 48, 64, 2, scale=2.0, seed=3), "cuda")
    return env, env.collect(policy, K, sample=sample)


def _critic(act=nn.Tanh, h1=64, h2=64, seed=7, scale=1.0):
    return MLPPolicy.from_module(_net(act, h1, h2, 1, scale, seed), "cuda")


def _probe_values(critic, rows):
    """V of each (N, 4) row block as policy_actions(critic, return_logits=True) computes it: column 1 of the logits."""
    probe = random_envs.RandomCartPoleVecEnv(rows[0].shape[0])
    probe.reset()
    out = []
    for r in rows:
        probe.set_state(r)
        out.append(probe.policy_actions(critic, return_logits=True)[1][:, 1].clone())
    return torch.stack(out)


def _replay32(values, done, trunc, v_final, v_last, gamma, lam):
    """The contract of include/renv.h renv_cartpole_gae_mlp_f32 in numpy float32: one rounding per operation."""
    K, n = values.shape
    g = np.float32(gamma)
    gl = np.float32(g * np.float32(lam))
    one, zero = np.float32(1.0), np.zeros(n, np.float32)
    adv, ret = np.empty((K, n), np.float32), np.empty((K, n), np.float32)
    a, v_next = zero, v_last
    for k in range(K - 1, -1, -1):
        v = values[k]
        nv = np.where(done[k], np.where(trunc[k], v_final[k], zero), v_next)
        delta = (one + g * nv) - v
        a = np.where(done[k], delta, delta + gl * a)
        adv[k], ret[k] = a, a + v
        v_next = v
    return adv, ret


def _check_replay(env, traj, critic, gamma, lam):
    v_final = _probe_values(critic, list(traj.final_obs)).cpu().numpy()
    v_last = _probe_values(critic, [env.obs])[0].cpu().numpy()
    adv, ret = _replay32(traj.values.cpu().numpy(), traj.dones.cpu().numpy(), traj.truncated.cpu().numpy(), v_final,
                         v_last, gamma, lam)
    got_a, got_r = traj.advantages.cpu().numpy(), traj.returns.cpu().numpy()
    assert np.array_equal(got_a, adv), int((got_a != adv).sum())
    assert np.array_equal(got_r, ret), int((got_r != ret).sum())


@pytest.mark.parametrize("act,h1,h2", [(nn.Tanh, 64, 64), (nn.ReLU, 64, 64), (nn.Tanh, 32, 48)])
def test_values_equal_policy_actions_logits(act, h1, h2):
    n, K = 3000 + 37, 40
    env, traj = _collected(n, K, act)
    critic = _critic(act, h1, h2, seed=h1 + h2)
    assert critic.outputs == 1
    env.gae(traj, critic)
    want = _probe_values(critic, list(traj.obs))
    assert torch.equal(traj.values, want)
    assert traj.values.shape == (K, n) and traj.advantages.shape == (K, n) and traj.returns.shape == (K, n)


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
@pytest.mark.parametrize("dr", ["uniform", "truncnorm"])
@pytest.mark.parametrize("sample", [True, False])
def test_advantages_and_returns_equal_a_float32_replay(act, dr, sample):
    n, K = 2000 + 5, 48
    env, traj = _collected(n, K, act, dr, sample, max_steps=12)
    assert bool(traj.truncated.any()) and bool(traj.truncated[K - 1].any())         # some truncate on the last step
    assert bool((traj.dones & ~traj.truncated).any())
    critic = _critic(act, seed=9, scale=1.5)
    for gamma, lam in GAMMA_LAMBDA:
        env.gae(traj, critic, gamma, lam)
        _check_replay(env, traj, critic, gamma, lam)


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
def test_a_single_step_bootstraps_from_the_observation_after_it(act):
    n = 4000
    env, traj = _collected(n, 1, act, max_steps=3)
    critic = _critic(act, seed=4)
    env.gae(traj, critic, 0.97, 0.9)
    assert bool(traj.truncated.any()) and bool((~traj.dones).any())           # both bootstraps: V(final_obs), V(s_K)
    _check_replay(env, traj, critic, 0.97, 0.9)


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
@pytest.mark.parametrize("gamma,lam", [(0.99, 0.95), (0.9, 0.0)])
def test_agrees_with_float64_gae(act, gamma, lam):
    n, K = 4096, 64
    env, traj = _collected(n, K, act, max_steps=30)
    critic = _critic(act, seed=12, scale=2.0)
    env.gae(traj, critic, gamma, lam)
    with torch.no_grad():
        v64 = critic.reference_logits(traj.obs.reshape(-1, 4))[:, 1].reshape(K, n)
        vf64 = critic.reference_logits(traj.final_obs.reshape(-1, 4))[:, 1].reshape(K, n)
        vl64 = critic.reference_logits(env.obs)[:, 1]
    done, trunc = traj.dones, traj.truncated
    g, gl = float(np.float32(gamma)), float(np.float32(gamma)) * float(np.float32(lam))
    a64, r64 = torch.empty_like(v64), torch.empty_like(v64)
    a, v_next = torch.zeros_like(vl64), vl64
    for k in range(K - 1, -1, -1):
        nv = torch.where(done[k], torch.where(trunc[k], vf64[k], torch.zeros_like(a)), v_next)
        delta = 1.0 + g * nv - v64[k]
        a = torch.where(done[k], delta, delta + gl * a)
        a64[k], r64[k] = a, a + v64[k]
        v_next = v64[k]
    # Bound.  Every V the kernel uses is within eps_v = 1e-5 max(1, M) of float64 (the logit contract; M = max |V64|
    # over obs, final_obs and s_K).  A step's delta = (1 + g nv) - v carries (1 + g) eps_v from its two V.  Its own
    # roundings: g*nv (<= M), 1 + . (<= 1 + M), - v (|delta| <= 1 + 2M), gl*A and the rounding of gl itself (<= |A|),
    # + (<= |A|): at most 9 u S with u = 2^-24 and S = max(1, M, max |A64|) -- c = 9.  The recurrence multiplies what
    # it carries by g*l per step, so the advantage error is at most [(1 + g) eps_v + 9 u S] / (1 - g l), and the return
    # adds eps_v of its v and one rounding u |R| <= 2 u S.
    M = max(float(v64.abs().max()), float(vf64[trunc].abs().max()) if bool(trunc.any()) else 0.0,
            float(vl64.abs().max()))
    eps_v = 1e-5 * max(1.0, M)
    S = max(1.0, M, float(a64.abs().max()))
    tol_a = ((1 + g) * eps_v + 9 * U * S) / (1 - gl)
    tol_r = tol_a + eps_v + 2 * U * S
    err_a = float((traj.advantages.double() - a64).abs().max())
    err_r = float((traj.returns.double() - r64).abs().max())
    assert err_a <= tol_a, (err_a, tol_a)
    assert err_r <= tol_r, (err_r, tol_r)
    assert float(a64.abs().max()) > 0.5                                              # a non-trivial recurrence


def test_sharding_repetition_and_a_second_critic():
    n, K = 3000, 50
    whole_env, whole = _collected(n, K, mid=False)
    halves = [_collected(n // 2, K, env_id0=h * (n // 2), mid=False) for h in range(2)]
    critic, other = _critic(seed=1), _critic(nn.Tanh, seed=2)
    whole_env.gae(whole, critic)
    for e, tr in halves:
        e.gae(tr, critic)
    for f in ("values", "advantages", "returns"):
        assert torch.equal(torch.cat([getattr(tr, f) for _, tr in halves], dim=1), getattr(whole, f)), f
    first = {f: getattr(whole, f).clone() for f in ("values", "advantages", "returns")}
    storage = whole._values.data_ptr()
    whole_env.gae(whole, critic)
    for f, v in first.items():
        assert torch.equal(getattr(whole, f), v), f
    whole_env.gae(whole, other)
    assert whole._values.data_ptr() == storage                                      # the same buffers, overwritten
    halves[0][0].gae(halves[0][1], other)
    assert not torch.equal(whole.values, first["values"])
    assert torch.equal(whole.values[:, :n // 2], halves[0][1].values)
    assert torch.equal(whole.advantages[:, :n // 2], halves[0][1].advantages)
    _check_replay(whole_env, whole, other, 0.99, 0.95)


def test_gae_changes_nothing_else():
    n, K = 2500, 40
    env, traj = _collected(n, K)
    env.start_episode_log(4)
    before = dict(state=env.state.clone(), xi=env.get_task().clone(), elapsed=env.elapsed.clone(),
                  episode=env.episode.clone(), stats=env.stats_tensor.clone(), tick=env._tick)
    fields = ("obs", "actions", "logp", "dones", "truncated", "final_obs")
    rows = {f: getattr(traj, f).clone() for f in fields}
    env.gae(traj, _critic())
    torch.cuda.synchronize()
    assert torch.equal(env.state, before["state"]) and torch.equal(env.get_task(), before["xi"])
    assert torch.equal(env.elapsed, before["elapsed"]) and torch.equal(env.episode, before["episode"])
    assert torch.equal(env.stats_tensor, before["stats"]) and env._tick == before["tick"]
    assert int(env.episode_log.count.sum()) == 0
    for f in fields:
        assert torch.equal(getattr(traj, f), rows[f]), f
    assert traj.num_steps == K and traj.tick0 == env._tick - K


def test_rejections():
    n, K = 256, 10
    env, traj = _collected(n, K, mid=False)
    critic = _critic()
    with pytest.raises(ValueError):
        env.gae(traj, MLPPolicy.from_module(_net(o=2), "cuda"))                     # 2-output
    with pytest.raises(ValueError):
        env.gae(random_envs.RandomCartPoleVecEnv(n + 32).trajectory_buffer(K), critic)
    with pytest.raises(ValueError):
        env.gae(env.trajectory_buffer(K), critic)                                   # nothing collected into it
    slim = env.collect(MLPPolicy.from_module(_net(), "cuda"), K, out=env.trajectory_buffer(K, final_obs=False))
    with pytest.raises(ValueError):
        env.gae(slim, critic)
    env2, traj2 = _collected(n, K, mid=False)
    for gamma, lam in ((1.5, 0.9), (0.9, -0.1), (math.nan, 0.9)):
        with pytest.raises(ValueError):
            env2.gae(traj2, critic, gamma, lam)
    env2.gae(traj2, critic)                                                        # the clock stands after the collect
    env2.step(env2.policy_actions(critic))                                         # step after collect
    with pytest.raises(ValueError):
        env2.gae(traj2, critic)
    env3, traj3 = _collected(n, K, mid=False)
    env3.reset()                                                                   # reset after collect
    with pytest.raises(ValueError):
        env3.gae(traj3, critic)
    env4, traj4 = _collected(n, K, mid=False)
    env4.rollout(MLPPolicy.from_module(_net(), "cuda"), 0.0, 3)                    # rollout after collect
    with pytest.raises(ValueError):
        env4.gae(traj4, critic)
    for kw in (dict(dtype="float64"), dict(noisy=True)):
        other = random_envs.RandomCartPoleVecEnv(n, **kw)
        other.reset()
        with pytest.raises(ValueError):
            other.gae(traj, critic)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="a critic on another device needs a second GPU")
def test_critic_on_another_device_raises():
    env = random_envs.RandomCartPoleVecEnv(64, device="cuda:0")
    env.reset()
    traj = env.collect(MLPPolicy.from_module(_net(), "cuda:0"), 4)
    with pytest.raises(ValueError):
        env.gae(traj, MLPPolicy.from_module(_net(o=1), "cuda:1"))
