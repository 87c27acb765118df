"""Evaluation grids on the GPU: every cell (p, c) against evaluate_population of a twin env configured with scenario c,
bit for bit (linear and MLP policies, fixed tasks, every DR law and mixes of them, both integrators, two TimeLimits),
independence from C, P, a cell's position and repetition, a 128 x 128 task map, sharding, the absence of side effects
on the env, and the rejections."""
import math

import numpy as np
import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from random_envs_b200 import MLPPopulation, Scenarios, combine_stats

pytestmark = pytest.mark.gpu

SEARCH = np.array([2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0])
LO, HI = SEARCH[0::2], SEARCH[1::2]
COV = [[0.30, 0.05, 0.00, 0.02], [0.05, 0.20, 0.03, 0.00], [0.00, 0.03, 0.25, 0.04], [0.02, 0.00, 0.04, 0.30]]
TICK = 7
LAWS = ("uniform", "truncnorm", "gaussian", "fullgaussian")


def _interleave(a, b):
    return np.stack([a, b], axis=1).ravel().tolist()


def _scenario_list(kind, C, seed):
    """C (kind, value) pairs: kind "task" (a (4,) task) or a DR law (its set_dr_distribution distr)."""
    rng = np.random.default_rng(seed)
    out = []
    for c in range(C):
        k = kind if kind != "mix" else ("task",) + LAWS
        k = k[c % len(k)] if isinstance(k, tuple) else k
        u = rng.random(4)
        if k == "task":
            out.append((k, LO + (HI - LO) * u))
        elif k == "uniform":
            lo = LO + (HI - LO) * 0.5 * u
            hi = lo + (HI - lo) * rng.random(4)
            if c % 3 == 1:
                hi[c % 4] = lo[c % 4]           # an ADR boundary: the dim pinned at lo
            out.append((k, _interleave(lo, hi)))
        elif k in ("truncnorm", "gaussian"):
            # means >= 4 std above the gaussian floor 0.1: no dim exhausts its three draws
            mean = np.array([9.8, 1.0, 0.5, 0.5]) * (0.8 + 0.4 * u)
            std = np.array([1.0, 0.1, 0.05, 0.05]) * (0.5 + rng.random(4))
            out.append((k, _interleave(mean, std)))
        else:
            out.append((k, {"mean": (np.array([2.0, 1.5, 2.5, 2.0]) + 0.5 * (u - 0.5)).tolist(), "cov": COV}))
    return out


def _scenarios(pairs):
    """Scenarios of (kind, value) pairs, each its own part, joined in order."""
    parts = [Scenarios.tasks([v], "cuda") if k == "task" else Scenarios.distributions(k, [v], "cuda") for k, v in pairs]
    return Scenarios.cat(*parts)


def _env(E, seed=5, env_id0=0, limit=500, integrator="euler"):
    env = random_envs.RandomCartPoleVecEnv(E, seed=seed, env_id0=env_id0, max_episode_steps=limit,
                                           kinematics_integrator=integrator)
    env._tick = TICK
    return env


def _twin(pair, E, tick, **cfg):
    """A fresh env of that configuration, set to scenario `pair`, its clock at `tick`."""
    env = _env(E, **cfg)
    kind, value = pair
    if kind == "task":
        env.set_task(*[float(v) for v in value])
    else:
        env.set_dr_distribution(kind, value)
        env.set_dr_training(True)
    env._tick = tick
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


def _policies(kind, P, seed=0):
    if kind == "linear":
        return _linear(P, seed)
    act, outputs = {"tanh2": (nn.Tanh, 2), "relu2": (nn.ReLU, 2), "tanh1": (nn.Tanh, 1), "relu1": (nn.ReLU, 1)}[kind]
    return _mlps(P, act, outputs, seed)


def _subset(policies, order):
    if isinstance(policies, MLPPopulation):
        return MLPPopulation(policies.params[list(order)], policies.activation, "cuda")
    return policies[list(order)].contiguous()


def _check_against_twins(grid, policies, pairs, E, K, tick, cells=None, **cfg):
    """grid[p, c] == twin(c).evaluate_population(policies)[p] for every cell (or the given ones)."""
    by_c = {}
    for p, c in cells if cells is not None else [(p, c) for c in range(len(pairs)) for p in range(grid.shape[0])]:
        by_c.setdefault(c, []).append(p)
    for c, ps in by_c.items():
        twin = _twin(pairs[c], E, tick, **cfg)
        want = twin.evaluate_population(policies if cells is None else _subset(policies, ps), K)
        twin.check_dr_violations()
        for q, p in enumerate(ps):
            row = p if cells is None else q
            assert torch.equal(grid[p, c], want[row]), (p, c, pairs[c][0], grid[p, c].tolist(), want[row].tolist())


def _run(env, policies, scen, K):
    tick = env._tick
    out = env.evaluate_grid(policies, scen, K)
    env.check_dr_violations()
    return out, tick


CASES = [   # policies, P, scenarios, C, E, K, TimeLimit, integrator
    ("linear", 1, "task", 1, 1, 1, 500, "euler"),
    ("linear", 3, "uniform", 5, 31, 17, 20, "semi-implicit"),
    ("linear", 37, "truncnorm", 5, 129, 500, 500, "euler"),
    ("linear", 3, "gaussian", 5, 1000, 500, 20, "euler"),
    ("linear", 37, "fullgaussian", 5, 128, 17, 500, "semi-implicit"),
    ("linear", 3, "mix", 33, 31, 500, 500, "euler"),
    ("linear", 1, "task", 33, 128, 500, 20, "semi-implicit"),
    ("tanh2", 3, "uniform", 33, 1, 500, 20, "euler"),
    ("relu2", 37, "task", 5, 31, 17, 500, "semi-implicit"),
    ("tanh1", 1, "truncnorm", 5, 1000, 500, 20, "semi-implicit"),
    ("relu1", 3, "gaussian", 1, 129, 17, 500, "euler"),
    ("tanh2", 3, "fullgaussian", 5, 128, 1, 20, "euler"),
    ("relu2", 3, "mix", 33, 1, 500, 500, "semi-implicit"),
    ("tanh1", 37, "mix", 5, 129, 17, 500, "euler"),
    ("relu1", 1, "task", 33, 1000, 500, 20, "euler"),
]


@pytest.mark.parametrize("kind,P,scen,C,E,K,limit,integrator", CASES)
def test_every_cell_equals_evaluate_population_of_a_twin(kind, P, scen, C, E, K, limit, integrator):
    cfg = dict(limit=limit, integrator=integrator)
    policies = _policies(kind, P, seed=P + E + K)
    pairs = _scenario_list(scen, C, seed=C + E)
    env = _env(E, **cfg)
    grid, tick = _run(env, policies, _scenarios(pairs), K)
    assert grid.dtype == torch.float64 and tuple(grid.shape) == (P, C, 6) and grid.device == env.device
    _check_against_twins(grid, policies, pairs, E, K, tick, **cfg)
    if K >= 17 and E * P * C >= 31:
        assert float(grid[:, :, 0].sum()) > 0       # episodes did end


@pytest.mark.parametrize("kind", ["linear", "tanh2"])
def test_a_cell_depends_on_neither_C_P_nor_its_position(kind):
    E, K = 31, 200
    base = _policies(kind, 5, seed=11)
    pairs = _scenario_list("mix", 10, seed=3)

    def run(order, cs):
        env = _env(E, limit=50)
        return env.evaluate_grid(_subset(base, order), _scenarios([pairs[c] for c in cs]), K)

    alone = run([2], [4])[0, 0]
    assert torch.equal(run([2], [4, 0, 1])[0, 0], alone)                 # more scenarios
    assert torch.equal(run([2], [0, 1, 4])[0, 2], alone)                 # another position
    assert torch.equal(run([0, 1, 2, 3, 4], [9, 4])[2, 1], alone)         # more policies
    assert torch.equal(run([4, 2], list(range(10)))[1, 4], alone)
    everything = (list(range(5)), list(range(10)))
    assert torch.equal(run(*everything), run(*everything))               # repetition
    # common random numbers: one scenario twice gives equal columns
    twice = run([0, 1], [3, 7, 3])
    assert torch.equal(twice[:, 0], twice[:, 2])


def test_a_16384_task_map_with_32_envs_each():
    P, E, K = 2, 32, 100
    g = torch.linspace(2.0, 20.0, 128, dtype=torch.float64)
    length = torch.linspace(0.1, 1.0, 128, dtype=torch.float64)
    gg, ll = torch.meshgrid(g, length, indexing="ij")
    tasks = torch.stack([gg.ravel(), torch.full_like(gg.ravel(), 1.0), torch.full_like(gg.ravel(), 0.1), ll.ravel()], 1)
    pairs = [("task", row) for row in tasks.numpy()]
    policies = _mlps(P, nn.ReLU, 2, seed=21)
    env = _env(E, limit=500)
    grid, tick = _run(env, policies, Scenarios.tasks(tasks, "cuda"), K)
    assert tuple(grid.shape) == (P, 128 * 128, 6) and float(grid[:, :, 0].sum()) > 0
    rng = np.random.default_rng(5)
    cells = [(int(rng.integers(P)), int(rng.integers(128 * 128))) for _ in range(6)] + [(0, 0), (P - 1, 128 * 128 - 1)]
    _check_against_twins(grid, policies, pairs, E, K, tick, cells=cells, limit=500)


def test_a_grid_of_2_to_the_31_triples_is_rejected():
    env = _env(1 << 11)
    scen = Scenarios.tasks(np.tile([9.8, 1.0, 0.1, 0.5], (1 << 10, 1)), "cuda")
    tick = env._tick
    with pytest.raises(ValueError):
        env.evaluate_grid(_linear(1 << 10, seed=0), scen, 10)
    assert env._tick == tick


@pytest.mark.parametrize("kind", ["linear", "relu2"])
def test_shards_combine_per_cell_to_the_unsharded_grid(kind):
    E, K, P = 1000, 300, 3
    policies = _policies(kind, P, seed=9)
    scen = _scenarios(_scenario_list("mix", 5, seed=8))
    whole = _env(E, limit=100).evaluate_grid(policies, scen, K).cpu().numpy()
    lo = _env(E // 2, limit=100).evaluate_grid(policies, scen, K).cpu().numpy()
    hi = _env(E - E // 2, limit=100, env_id0=E // 2).evaluate_grid(policies, scen, K).cpu().numpy()
    for p in range(P):
        for c in range(5):
            assert np.array_equal(combine_stats(np.stack([lo[p, c], hi[p, c]])), whole[p, c]), (p, c)


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
    env, twin = _env(E, limit=30), _env(E, limit=30)
    for e in (env, twin):
        e.set_dr_distribution("uniform", SEARCH.tolist())
        e.set_dr_training(True)
    env.start_episode_log(4)
    _history(env)
    _history(twin)
    before, tick = _snapshot(env), env._tick
    assert int(env.episode_log.count.sum()) > 0 and float(before["stats"][0]) > 0
    env.evaluate_grid(_policies(kind, 4, seed=1), _scenarios(_scenario_list("mix", 5, seed=2)), K)
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


def test_a_gaussian_failure_is_raised_at_the_next_synchronising_call():
    env = random_envs.RandomCartPoleVecEnv(64, seed=1)
    scen = Scenarios.distributions("gaussian", [[9.8, 1.0, 1.0, 0.1, -3.0, 0.1, 0.5, 0.05]], "cuda")
    env.evaluate_grid(_linear(3, seed=0), scen, 10)            # no synchronisation, no error yet
    with pytest.raises(Exception, match="Not all samples were above > 0.1 after 2 attempts"):
        env.episode_stats()


def test_rejections():
    pop = _linear(3, seed=0)
    scen = _scenarios(_scenario_list("mix", 5, seed=0))
    with pytest.raises(ValueError):
        random_envs.RandomCartPoleVecEnv(16, dtype="float64").evaluate_grid(pop, scen, 10)
    with pytest.raises(ValueError):
        random_envs.RandomCartPoleVecEnv(16, noisy=True).evaluate_grid(pop, scen, 10)
    env = _env(16)
    tick = env._tick
    with pytest.raises(ValueError):
        Scenarios.tasks(np.zeros((0, 4)), "cuda")
    with pytest.raises(ValueError):
        env.evaluate_grid(pop, Scenarios(scen.rows.cpu()), 10)               # scenarios on another device
    with pytest.raises(TypeError):
        env.evaluate_grid(pop, scen.rows, 10)
    for bad in (pop.double(), pop[:0], pop.cpu()):
        with pytest.raises(ValueError):
            env.evaluate_grid(bad, scen, 10)
    for K in (0, -1):
        with pytest.raises(ValueError):
            env.evaluate_grid(pop, scen, K)
    assert env._tick == tick
    out = env.evaluate_grid(pop, scen, 1)
    assert tuple(out.shape) == (3, 5, 6) and math.isinf(float(out[0, 0, 3]))   # a 1-step run ends no episode
