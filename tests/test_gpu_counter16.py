"""The default fp32 env keeps its TimeLimit counter as uint16 and takes the 54-byte step: everything it computes equals
what the same env with the int32 counter computes, bit for bit -- step (tile and grid ordering, eager and under CUDA
graph replay, across TimeLimit truncations), the linear, random and MLP rollouts, collect, population evaluation and
the episode log -- and its state_dict loads into either layout."""
import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from random_envs_b200 import MLPPolicy, MLPPopulation

pytestmark = pytest.mark.gpu

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
SURVIVE = (0.1, 0.1, 1.0, 0.3)


def _pair(n, seed=3, **kw):
    """(default env, the same env with the int32 counter), reset, uniform DR on."""
    out = []
    for int32 in (False, True):
        env = random_envs.RandomCartPoleVecEnv(n, seed=seed, env_id0=77, _int32_counter=int32, **kw)
        env.set_dr_distribution("uniform", SEARCH)
        env.set_dr_training(True)
        env.reset()
        out.append(env)
    a, b = out
    assert a._buffers["elapsed16"] is not None and a._buffers["elapsed"] is a._buffers["elapsed16"]
    assert b._buffers["elapsed"] is not None and b._buffers["elapsed16"] is None
    return a, b


def _net(seed=0, act=nn.Tanh):
    torch.manual_seed(seed)
    return nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2))


def _assert_same(a, b):
    assert torch.equal(a.obs, b.obs) and torch.equal(a.get_task(), b.get_task())
    assert torch.equal(a.elapsed, b.elapsed) and torch.equal(a.episode, b.episode)
    assert torch.equal(a.stats_tensor, b.stats_tensor)


def test_layout_follows_the_settings():
    for kw, c16 in ((dict(), True), (dict(max_episode_steps=65535), True), (dict(dtype="float64"), False),
                    (dict(noisy=True), False), (dict(auto_reset=False), False), (dict(max_episode_steps=0), False),
                    (dict(max_episode_steps=65536), False)):
        env = random_envs.RandomCartPoleVecEnv(64, **kw)
        env.reset()
        assert (env._buffers["elapsed16"] is not None) == c16, kw
        assert env._buffers["elapsed"].dtype == (torch.int16 if c16 else torch.int32), kw
    env = random_envs.RandomCartPoleVecEnv(64)
    env.reset()
    _, reward, _, _ = env.step(env.sample_actions())
    assert env._step_plan()["name"] == "renv_cartpole_step_lean_f32"        # no reward argument, 54 B per env-step
    assert reward.data_ptr() == env._buffers["reward"].data_ptr() and float(reward.min()) == 1.0 == float(reward.max())


@pytest.mark.parametrize("tile_ordering", [True, False])
def test_step_equals_the_int32_layout_across_two_timelimits(tile_ordering):
    n = 1 << 20
    a, b = _pair(n, tile_ordering=tile_ordering)
    for k in range(1100):                      # 500-step TimeLimit: envs that survive are truncated at 500 and 1000
        act = a.sample_actions().clone()
        if k % 2:                              # half the steps under a surviving policy, so that truncations happen
            act = ((a.obs @ torch.tensor(SURVIVE, device="cuda")) > 0).to(torch.uint8)
        oa, ra, da, ia = a.step(act)
        ob, rb, db, ib = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(da, db), k
        assert torch.equal(ia["TimeLimit.truncated"], ib["TimeLimit.truncated"]), k
        if k % 50 == 0 or k in (499, 500, 999, 1000):
            assert torch.equal(ra, rb) and torch.equal(a.elapsed, b.elapsed) and torch.equal(a.get_task(), b.get_task())
            assert torch.equal(a.episode, b.episode)
    assert int(a.elapsed.max()) < 500
    _assert_same(a, b)


def test_step_equals_the_int32_layout_under_graph_replay():
    n = 1 << 20
    a, b = _pair(n)
    act = a.sample_actions().clone()
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for _ in range(60):
                a.step(act)
                b.step(act)
    torch.cuda.current_stream().wait_stream(side)
    for _ in range(10):                        # 600 steps: one TimeLimit
        g.replay()
    torch.cuda.synchronize()
    _assert_same(a, b)


@pytest.mark.parametrize("w", [SURVIVE, None], ids=["linear", "random"])
def test_rollout_equals_the_int32_layout(w):
    n = 300_001
    a, b = _pair(n)
    for env in (a, b):
        env.rollout(w, 0.0, 700)
        env.step(env.sample_actions())
        env.rollout(w, 0.0, 333)
    _assert_same(a, b)


def test_mlp_rollout_and_collect_equal_the_int32_layout():
    n = 70_001
    a, b = _pair(n)
    policy = MLPPolicy.from_module(_net(1), "cuda")
    for env in (a, b):
        env.rollout(policy, 0.0, 520)
    _assert_same(a, b)
    ta, tb = a.collect(policy, 64), b.collect(policy, 64)
    for f in ("obs", "actions", "logp", "dones", "truncated", "final_obs"):
        assert torch.equal(getattr(ta, f), getattr(tb, f)), f
    _assert_same(a, b)


def test_population_equals_the_int32_layout():
    a, b = _pair(4099)
    lin = torch.tensor([SURVIVE + (0.0,), (0.0, 0.0, 1.0, 0.5, 0.0)], dtype=torch.float32, device="cuda")
    pop = MLPPopulation.from_modules([_net(2), _net(3)], "cuda")
    for policies in (lin, pop):
        assert torch.equal(a.evaluate_population(policies, 600), b.evaluate_population(policies, 600))
    _assert_same(a, b)


def test_episode_log_equals_the_int32_layout():
    a, b = _pair(50_003)
    la, lb = a.start_episode_log(4), b.start_episode_log(4)
    policy = MLPPolicy.from_module(_net(4), "cuda")
    for env in (a, b):
        for _ in range(30):
            env.step(env.sample_actions())
        env.rollout(SURVIVE, 0.0, 600)
        env.rollout(None, 0.0, 50)
        env.rollout(policy, 0.0, 40)
        env.collect(policy, 20)
    for f in ("xi", "final_state", "length", "truncated", "end_tick", "count"):
        assert torch.equal(getattr(la, f), getattr(lb, f)), f
    assert int(la.count.sum()) > 50_003
    _assert_same(a, b)


def test_state_dict_loads_into_either_layout():
    a, b = _pair(5000)
    a.rollout(SURVIVE, 0.0, 321)
    b.rollout(SURVIVE, 0.0, 321)
    sa, sb = a.state_dict(), b.state_dict()
    assert "elapsed16" in sa and "elapsed" in sb
    c, d = _pair(5000, seed=9)
    c.load_state_dict(sb)                     # int32 counter -> uint16 layout
    d.load_state_dict(sa)                     # uint16 counter -> int32 layout
    _assert_same(c, a)
    _assert_same(d, b)
    for env in (a, b, c, d):
        env.rollout(SURVIVE, 0.0, 300)
    _assert_same(a, c)
    _assert_same(b, d)
    _assert_same(a, b)


def test_settings_that_rule_out_the_uint16_counter_widen_it():
    a, b = _pair(4096)
    for env in (a, b):
        env.rollout(SURVIVE, 0.0, 450)
        env.max_episode_steps = 0             # no TimeLimit from now on: the counter must count past 65535
        env.rollout(SURVIVE, 0.0, 100)
    assert a._buffers["elapsed16"] is None
    _assert_same(a, b)
    for env in (a, b):
        env.max_episode_steps = 500
        env.step(env.sample_actions())
    _assert_same(a, b)
