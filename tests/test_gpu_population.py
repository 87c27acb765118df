"""Population evaluation on the GPU: every member's statistics against a reference reset() + rollout() of a fresh twin
env, bit for bit (linear and MLP policies, DR off and every DR law, both integrators, two TimeLimits), common random
numbers and independence from the population, a population past 65,535 members, sharding, the absence of side effects
on the env, and the rejections."""
import math

import numpy as np
import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from random_envs_b200 import MLPPolicy, MLPPopulation, combine_stats

pytestmark = pytest.mark.gpu

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
DR = {
    "uniform": SEARCH,
    "truncnorm": [9.8, 1.0, 1.0, 0.2, 0.1, 0.03, 0.5, 0.1],
    "gaussian": [9.8, 1.0, 1.0, 0.2, 0.3, 0.03, 0.5, 0.1],
    "fullgaussian": {"mean": [2.0, 1.5, 2.5, 2.0],
                     "cov": [[0.30, 0.05, 0.00, 0.02], [0.05, 0.20, 0.03, 0.00],
                             [0.00, 0.03, 0.25, 0.04], [0.02, 0.00, 0.04, 0.30]]},
}
TICK = 7


def _table(seed, rows=4096):
    g = torch.Generator().manual_seed(seed)
    lo, hi = torch.tensor(SEARCH[0::2]), torch.tensor(SEARCH[1::2])
    return (lo + (hi - lo) * torch.rand((rows, 4), generator=g)).float()


def _env(E, dr="uniform", seed=5, env_id0=0, limit=500, integrator="euler", table_seed=0):
    env = random_envs.RandomCartPoleVecEnv(E, seed=seed, env_id0=env_id0, max_episode_steps=limit,
                                           kinematics_integrator=integrator)
    if dr == "table":           # DR off: xi is the env's per-env table
        env.set_task(_table(table_seed)[env_id0:env_id0 + E].cuda())
    else:
        env.set_dr_distribution(dr, DR[dr])
        env.set_dr_training(True)
    env._tick = TICK
    return env


def _linear(P, seed):
    g = torch.Generator().manual_seed(seed)
    scale = torch.tensor([0.5, 0.5, 3.0, 1.0, 0.2])
    shift = torch.tensor([0.0, 0.0, 1.0, 0.5, 0.0])
    return (torch.randn((P, 5), generator=g) * scale + shift).float().cuda()


def _mlps(P, act, outputs, seed):
    nets = []
    for p in range(P):
        torch.manual_seed(seed + p)
        nets.append(nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 48), act(), nn.Linear(48, outputs)))
    return MLPPopulation.from_modules(nets, "cuda")


def _population(kind, P, seed=0):
    if kind == "linear":
        return _linear(P, seed)
    act, outputs = {"tanh2": (nn.Tanh, 2), "relu2": (nn.ReLU, 2), "tanh1": (nn.Tanh, 1), "relu1": (nn.ReLU, 1)}[kind]
    return _mlps(P, act, outputs, seed)


def _member(pop, p):
    return pop.member(p) if isinstance(pop, MLPPopulation) else pop[p]


def _reference(policy, E, K, **cfg):
    """stats of reset() at TICK, then rollout(policy, K), on a fresh env of that configuration"""
    env = _env(E, **cfg)
    env.reset()
    if isinstance(policy, MLPPolicy):
        env.rollout(policy, num_steps=K)
    else:
        row = policy.double().cpu().tolist()
        env.rollout(row[:4], row[4], K)
    stats = env.stats_tensor.clone()
    env.check_dr_violations()
    return stats


CASES = [   # kind, P, E, K, TimeLimit, integrator, DR
    ("linear", 1, 1, 1, 500, "euler", "table"),
    ("linear", 3, 31, 17, 20, "semi-implicit", "uniform"),
    ("linear", 37, 129, 500, 500, "euler", "truncnorm"),
    ("linear", 3, 1000, 500, 20, "euler", "gaussian"),
    ("linear", 37, 128, 17, 500, "semi-implicit", "fullgaussian"),
    ("linear", 3, 1, 500, 20, "semi-implicit", "table"),
    ("linear", 37, 31, 500, 500, "euler", "uniform"),
    ("linear", 1, 1000, 500, 500, "semi-implicit", "table"),
    ("tanh2", 3, 129, 500, 500, "euler", "uniform"),
    ("relu2", 37, 31, 17, 20, "semi-implicit", "table"),
    ("tanh1", 1, 1000, 500, 20, "semi-implicit", "truncnorm"),
    ("relu1", 3, 1, 17, 500, "euler", "gaussian"),
    ("tanh2", 3, 128, 1, 20, "euler", "fullgaussian"),
    ("relu2", 1, 1000, 500, 500, "euler", "table"),
    ("tanh1", 37, 129, 17, 500, "euler", "table"),
    ("relu1", 3, 1000, 500, 20, "semi-implicit", "fullgaussian"),
]


@pytest.mark.parametrize("kind,P,E,K,limit,integrator,dr", CASES)
def test_every_member_equals_a_reset_and_rollout_of_a_fresh_twin(kind, P, E, K, limit, integrator, dr):
    cfg = dict(dr=dr, limit=limit, integrator=integrator)
    pop = _population(kind, P, seed=P + E + K)
    env = _env(E, **cfg)
    stats = env.evaluate_population(pop, K)
    assert stats.dtype == torch.float64 and tuple(stats.shape) == (P, 6) and stats.device == env.device
    env.check_dr_violations()
    for p in range(P):
        want = _reference(_member(pop, p), E, K, **cfg)
        assert torch.equal(stats[p], want), (p, stats[p].tolist(), want.tolist())
    if K >= 17 and E * P >= 31:
        assert float(stats[:, 0].sum()) > 0       # episodes did end


@pytest.mark.parametrize("kind", ["linear", "tanh2"])
def test_common_random_numbers_and_independence_from_the_population(kind):
    E, K = 129, 200
    base = _population(kind, 37, seed=11)
    if kind == "linear":
        def make(order):
            return base[list(order)].contiguous()
    else:
        def make(order):
            return MLPPopulation(base.params[list(order)], base.activation, "cuda")

    def run(order):
        return _env(E, dr="uniform", limit=50).evaluate_population(make(order), K)

    # identical members: identical rows
    twins = run([0, 0, 1, 0])
    assert torch.equal(twins[0], twins[1]) and torch.equal(twins[0], twins[3]) and not torch.equal(twins[0], twins[2])
    # member 5 alone, in a pair, and at three positions of a population of 37
    alone = run([5])[0]
    assert torch.equal(run([5, 6])[0], alone) and torch.equal(run([6, 5])[1], alone)
    for pos in (0, 18, 36):
        order = [q for q in range(37) if q != 5]
        order.insert(pos, 5)
        assert torch.equal(run(order)[pos], alone), pos
    # two identical calls
    everyone = list(range(37))
    assert torch.equal(run(everyone), run(everyone))


def test_a_population_of_70000_linear_policies_on_one_env_each():
    P, E, K = 70000, 1, 50
    pop = _linear(P, seed=3)
    stats = _env(E, dr="uniform", limit=20).evaluate_population(pop, K)
    assert float(stats[:, 0].sum()) > 0
    for p in np.random.default_rng(0).choice(P, 20, replace=False).tolist() + [0, P - 1]:
        assert torch.equal(stats[p], _reference(pop[p], E, K, dr="uniform", limit=20)), p


def test_a_population_of_66000_mlp_policies_runs_on_the_one_dimensional_grid():
    P, E, K = 66000, 1, 3
    one = _mlps(1, nn.ReLU, 2, seed=4)
    pop = MLPPopulation(one.params.repeat(P, 1), one.activation, "cuda")
    pop.params[P - 1, 4608] += 1.0          # the last member differs: its own row must reach its own CTA
    stats = _env(E, dr="uniform", limit=2).evaluate_population(pop, K)
    for p in (0, 65535, 65536, P - 1):
        assert torch.equal(stats[p], _reference(pop.member(p), E, K, dr="uniform", limit=2)), p


@pytest.mark.parametrize("kind", ["linear", "relu2"])
def test_shards_combine_per_member_to_the_unsharded_rows(kind):
    E, K, P = 1000, 300, 5
    pop = _population(kind, P, seed=9)
    whole = _env(E, dr="uniform", limit=100).evaluate_population(pop, K).cpu().numpy()
    lo = _env(E // 2, dr="uniform", limit=100).evaluate_population(pop, K).cpu().numpy()
    hi = _env(E - E // 2, dr="uniform", limit=100, env_id0=E // 2).evaluate_population(pop, K).cpu().numpy()
    for p in range(P):
        assert np.array_equal(combine_stats(np.stack([lo[p], hi[p]])), whole[p]), p
    # the table variant: the shard holds its slice of the table
    whole = _env(E, dr="table").evaluate_population(pop, K).cpu().numpy()
    lo = _env(E // 2, dr="table").evaluate_population(pop, K).cpu().numpy()
    hi = _env(E - E // 2, dr="table", env_id0=E // 2).evaluate_population(pop, K).cpu().numpy()
    for p in range(P):
        assert np.array_equal(combine_stats(np.stack([lo[p], hi[p]])), whole[p]), p


def _history(env):
    env.reset()
    for _ in range(7):
        env.step(env.sample_actions())
    env.rollout((0.1, 0.2, 2.0, 0.4), 0.0, 60)


def _snapshot(env):
    b = env._buffers
    out = {k: b[k].clone() for k in ("state", "xi", "elapsed", "episode", "beyond", "stats")}
    if b["progress"] is not None:
        out["progress"] = b["progress"].clone()
    log = env.episode_log
    if log is not None:
        for f in ("_xi", "_final_state", "_length", "_truncated", "_end_tick", "_count"):
            out["log" + f] = getattr(log, f).clone()
    return out


@pytest.mark.parametrize("kind", ["linear", "tanh1"])
def test_the_env_is_left_untouched_except_for_its_clock(kind):
    E, K = 300, 40
    env, twin = _env(E, dr="uniform", limit=30), _env(E, dr="uniform", limit=30)
    env.start_episode_log(4)
    _history(env)
    _history(twin)
    before, tick = _snapshot(env), env._tick
    assert int(env.episode_log.count.sum()) > 0 and float(before["stats"][0]) > 0
    env.evaluate_population(_population(kind, 6, seed=1), K)
    after = _snapshot(env)
    assert before.keys() == after.keys()
    for k in before:
        assert torch.equal(before[k], after[k]), k
    assert env._tick == tick + K + 1
    twin._tick += K + 1
    for _ in range(3):
        a = env.sample_actions().clone()
        assert torch.equal(a, twin.sample_actions())
        o, r, d, info = env.step(a)
        o2, r2, d2, info2 = twin.step(a)
        assert torch.equal(o, o2) and torch.equal(d, d2)
        assert torch.equal(info["TimeLimit.truncated"], info2["TimeLimit.truncated"])
    assert torch.equal(env.get_task(), twin.get_task())
    env.check_dr_violations()


def test_consecutive_calls_draw_new_tasks():
    env = _env(64, dr="uniform", limit=500)
    pop = _linear(4, seed=2)
    first, second = env.evaluate_population(pop, 100), env.evaluate_population(pop, 100)
    assert not torch.equal(first, second)
    again = _env(64, dr="uniform", limit=500)
    again._tick = TICK + 101
    assert torch.equal(again.evaluate_population(pop, 100), second)


def test_a_gaussian_failure_is_raised_at_the_next_synchronising_call():
    env = random_envs.RandomCartPoleVecEnv(64, seed=1)
    env.set_dr_distribution("gaussian", [9.8, 1.0, 1.0, 0.1, -3.0, 0.1, 0.5, 0.05])
    env.set_dr_training(True)
    env.evaluate_population(_linear(3, seed=0), 10)            # no synchronisation, no error yet
    with pytest.raises(Exception, match="Not all samples were above > 0.1 after 2 attempts"):
        env.episode_stats()


def test_rejections():
    pop = _linear(3, seed=0)
    with pytest.raises(ValueError):
        random_envs.RandomCartPoleVecEnv(16, dtype="float64").evaluate_population(pop, 10)
    with pytest.raises(ValueError):
        random_envs.RandomCartPoleVecEnv(16, noisy=True).evaluate_population(pop, 10)
    env = _env(16)
    tick = env._tick
    for bad in (pop.double(), pop[:, :4].contiguous(), pop[:0], pop.reshape(-1), pop.cpu()):
        with pytest.raises(ValueError):
            env.evaluate_population(bad, 10)
    with pytest.raises(ValueError):
        env.evaluate_population(MLPPopulation(_mlps(2, nn.Tanh, 2, 0).params.cpu(), 0, "cpu"), 10)
    mlp = MLPPopulation(_mlps(2, nn.Tanh, 2, 0).params, 0, "cuda")          # "cuda" without an index is the env's device
    assert mlp.device == env.device and tuple(env.evaluate_population(mlp, 1).shape) == (2, 6)
    tick = env._tick
    with pytest.raises(TypeError):
        env.evaluate_population(_mlps(1, nn.Tanh, 2, 0).member(0), 10)
    for K in (0, -1):
        with pytest.raises(ValueError):
            env.evaluate_population(pop, K)
    assert env._tick == tick
    assert math.isinf(float(env.evaluate_population(pop, 1)[0, 3]))      # a 1-step run ends no episode from a reset
