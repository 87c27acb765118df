"""MLP policy on the GPU: logits against float64 torch, the fused rollout against K x step(policy_actions) bit for bit
(buffers, statistics, episode log, chaining, sharding), a closed loop against the float64 torch module, and the
rejections."""
import math

import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from random_envs_b200 import MLPPolicy

pytestmark = pytest.mark.gpu

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
BOX = torch.tensor([2.4, 3.0, 0.21, 3.5], dtype=torch.float64)


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


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
@pytest.mark.parametrize("scale", [1.0, 4.0])
@pytest.mark.parametrize("h1,h2,o", [(64, 64, 2), (48, 32, 2), (64, 64, 1), (48, 32, 1)])
def test_logits_meet_the_fp32_accuracy_contract(act, scale, h1, h2, o):
    n = 1 << 20
    net = _net(act, h1, h2, o, scale, seed=h1 + h2 + o)
    policy = MLPPolicy.from_module(net, "cuda")
    env = _env(n, seed=1, dr=None)
    g = torch.Generator(device="cuda").manual_seed(7)
    obs = (torch.rand((n, 4), generator=g, device="cuda", dtype=torch.float64) * 2 - 1) * BOX.cuda()
    env.set_state(obs.float())
    actions, logits = env.policy_actions(policy, return_logits=True)
    x = env.state.double()
    with torch.no_grad():
        ref = net.double().cuda()(x)
    if o == 1:
        ref = torch.cat([torch.zeros_like(ref), ref], dim=1)
    bound = 1e-5 * max(1.0, float(ref.abs().max()))
    err = float((logits.double() - ref).abs().max())
    assert err <= bound, (err, bound)
    margin = ref[:, 1] - ref[:, 0]
    want = (margin > 0).to(torch.uint8)
    clear = margin.abs() > 2 * bound
    assert torch.equal(actions[clear], want[clear])
    assert torch.equal(actions, (logits[:, 1] > logits[:, 0]).to(torch.uint8))


def _stepped_stats(env, policy, K, stats):
    for _ in range(K):
        el0 = env.elapsed.clone()
        _, _, done, _ = env.step(env.policy_actions(policy))
        r = (el0 + 1)[done].double()
        if len(r):
            stats[0] += len(r); stats[1] += float(r.sum()); stats[2] += float((r * r).sum())
            stats[3] = min(stats[3], float(r.min())); stats[4] = max(stats[4], float(r.max())); stats[5] += float(r.sum())
    return stats


def _assert_envs_equal(a, b):
    assert torch.equal(a.state, b.state) and torch.equal(a.get_task(), b.get_task())
    assert torch.equal(a.elapsed, b.elapsed) and torch.equal(a.episode, b.episode)


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
@pytest.mark.parametrize("dr", ["uniform", "truncnorm"])
@pytest.mark.parametrize("integrator", ["euler", "semi-implicit"])
def test_rollout_equals_k_steps_of_policy_actions(act, dr, integrator):
    n, K = 5000 + 37, 120        # not a multiple of 32 or 128
    policy = MLPPolicy.from_module(_net(act, 48, 64, 2, scale=2.0, seed=3), "cuda")
    fused, stepped = (_env(n, 5, dr, max_episode_steps=40, kinematics_integrator=integrator) for _ in range(2))
    g = torch.Generator(device="cuda").manual_seed(11)
    mid = (torch.rand((n, 4), generator=g, device="cuda") * 2 - 1) * BOX.float().cuda() * 0.5
    el = torch.randint(0, 40, (n,), generator=g, device="cuda")
    for e in (fused, stepped):
        e.reset()
        e.set_state(mid, elapsed=el)          # an injected mid-episode start
    fused.rollout(policy, 0.0, K)
    want = _stepped_stats(stepped, policy, K, [0.0, 0.0, 0.0, math.inf, -math.inf, 0.0])
    _assert_envs_equal(fused, stepped)
    assert fused.stats_tensor.tolist() == want
    assert want[0] > n and fused._tick == stepped._tick


def test_chained_and_sharded_rollouts_equal_one_rollout():
    n = 3000
    policy = MLPPolicy.from_module(_net(nn.Tanh, seed=5), "cuda")
    whole, chained = _env(n, 9, max_episode_steps=60), _env(n, 9, max_episode_steps=60)
    halves = [_env(n // 2, 9, max_episode_steps=60, env_id0=k * (n // 2)) for k in range(2)]
    for e in [whole, chained] + halves:
        e.reset()
    whole.rollout(policy, 0.0, 90)
    chained.rollout(policy, 0.0, 35)
    chained.rollout(policy, 0.0, 55)
    _assert_envs_equal(whole, chained)
    assert torch.equal(whole.stats_tensor, chained.stats_tensor)
    for h in halves:
        h.rollout(policy, 0.0, 90)
    assert torch.equal(torch.cat([h.state for h in halves]), whole.state)
    assert torch.equal(torch.cat([h.get_task() for h in halves]), whole.get_task())
    assert torch.equal(torch.cat([h.elapsed for h in halves]), whole.elapsed)


@pytest.mark.parametrize("act", [nn.Tanh, nn.ReLU])
def test_logged_rollout_writes_what_logged_steps_write(act):
    n, K, R = 4000, 150, 16
    policy = MLPPolicy.from_module(_net(act, 64, 32, 1, seed=8), "cuda")
    fused, stepped, plain = (_env(n, 2, max_episode_steps=10) for _ in range(3))     # terminations and truncations
    for e in (fused, stepped, plain):
        e.reset()
    lf, ls = fused.start_episode_log(R), stepped.start_episode_log(R)
    fused.rollout(policy, 0.0, K)
    plain.rollout(policy, 0.0, K)
    for _ in range(K):
        stepped.step(stepped.policy_actions(policy))
    for f in ("xi", "final_state", "length", "truncated", "end_tick", "count"):
        assert torch.equal(getattr(lf, f), getattr(ls, f)), f
    assert int(lf.count.sum()) > n and bool(lf.truncated.any())
    _assert_envs_equal(fused, stepped)
    _assert_envs_equal(fused, plain)
    assert torch.equal(fused.stats_tensor, plain.stats_tensor)


def test_closed_loop_against_the_float64_module():
    """Per env, the trajectory driven by the float64 torch module equals the fused rollout's bit for bit at every step
    before the env's first step whose float64 margin |l1 - l0| is below 1e-4; no env diverges without such a tie."""
    n, K = 4096, 300
    net = _net(nn.Tanh, seed=12, scale=2.0)
    policy = MLPPolicy.from_module(net, "cuda")
    ref_net = net.double().cuda()
    fused, torch_driven, stepped = _env(n, 4), _env(n, 4), _env(n, 4)
    for e in (fused, torch_driven, stepped):
        e.reset()
    tied = torch.full((n,), K, dtype=torch.int64, device="cuda")       # step of the first near-tie, K = none
    ref_traj, fused_traj = [], []
    for k in range(K):
        with torch.no_grad():
            logits = ref_net(torch_driven.state.double())
        margin = (logits[:, 1] - logits[:, 0]).abs()
        tied = torch.where((margin < 1e-4) & (tied == K), torch.full_like(tied, k), tied)
        torch_driven.step((logits[:, 1] > logits[:, 0]).to(torch.uint8))
        stepped.step(stepped.policy_actions(policy))       # the fused trajectory, one step at a time
        ref_traj.append(torch_driven.state.clone())
        fused_traj.append(stepped.state.clone())
    fused.rollout(policy, 0.0, K)
    assert torch.equal(fused.state, stepped.state)         # stepped IS the fused rollout's trajectory
    ref_traj, fused_traj = torch.stack(ref_traj), torch.stack(fused_traj)          # (K, n, 4): state after step k
    before_tie = torch.arange(K, device="cuda")[:, None] < tied[None, :]          # (K, n): step k precedes the tie
    same = (ref_traj == fused_traj).all(dim=2)
    assert bool(same[before_tie].all()), "an env diverged before its first near-tie"
    assert int((tied == K).sum()) > n // 2                 # most envs never meet a near-tie: a strong check


@pytest.mark.parametrize("kw", [dict(dtype="float64"), dict(noisy=True), dict(lean=True)])
def test_unsupported_envs_raise(kw):
    policy = MLPPolicy.from_module(_net(), "cuda")
    env = random_envs.RandomCartPoleVecEnv(64, **kw)
    env.reset()
    with pytest.raises(ValueError):
        env.rollout(policy, 0.0, 5)
    if "lean" not in kw:
        with pytest.raises(ValueError):
            env.policy_actions(policy)


def test_bias_with_a_policy_raises():
    policy = MLPPolicy.from_module(_net(), "cuda:0")
    env = random_envs.RandomCartPoleVecEnv(64, device="cuda:0")
    env.reset()
    with pytest.raises(ValueError):
        env.rollout(policy, 0.5, 5)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="a policy on another device needs a second GPU")
def test_policy_on_another_device_raises():
    env = random_envs.RandomCartPoleVecEnv(64, device="cuda:0")
    env.reset()
    far = MLPPolicy.from_module(_net(), "cuda:1")
    with pytest.raises(ValueError):
        env.rollout(far, 0.0, 5)
    with pytest.raises(ValueError):
        env.policy_actions(far)
