"""Per-env task scenarios on the GPU: an env whose envs are assigned to a mix of DR laws and fixed tasks, against one
twin env per scenario configured with it (set_dr_distribution + set_dr_training(True), or set_task without DR), bit for
bit: reset, step in its three layouts (and logged, tile-ordered, under CUDA-graph replay), the linear, random and MLP
rollouts, collect, both integrators.  Also the per-scenario statistics against the twins' episode logs, C = 1 against
the env's own config, independence from the other envs' assignment and from C, sharding, checkpoints, and the
refusals."""
import numpy as np
import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from random_envs_b200 import MLPPolicy, Scenarios

pytestmark = pytest.mark.gpu

COV = [[0.30, 0.05, 0.00, 0.02], [0.05, 0.20, 0.03, 0.00], [0.00, 0.03, 0.25, 0.04], [0.02, 0.00, 0.04, 0.30]]
# (kind, value): the four laws (gaussian means well above its 0.1 floor), an ADR boundary and two fixed tasks
PAIRS = [
    ("uniform", [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]),
    ("truncnorm", [9.8, 1.0, 1.0, 0.2, 0.5, 0.05, 0.5, 0.1]),
    ("gaussian", [9.8, 1.0, 1.0, 0.1, 0.5, 0.05, 0.5, 0.05]),
    ("fullgaussian", {"mean": [2.0, 1.5, 2.5, 2.0], "cov": COV}),
    ("uniform", [2.0, 20.0, 3.0, 3.0, 0.05, 0.3, 0.1, 1.0]),
    ("task", [15.5, 0.75, 0.2, 0.25]),
    ("task", [4.0, 2.5, 0.05, 0.9]),
]
N = 3000            # not a multiple of the step tile (1024) nor of 32
SEED, ID0 = 11, 5


def _scenarios(pairs):
    return Scenarios.cat(*[Scenarios.tasks([v], "cuda") if k == "task" else Scenarios.distributions(k, [v], "cuda")
                           for k, v in pairs])


def _assignment(n=N, C=len(PAIRS), seed=0):
    return torch.from_numpy(np.random.default_rng(seed).integers(0, C, n)).cuda()


def _env(n=N, env_id0=ID0, **kw):
    kw.setdefault("seed", SEED)
    return random_envs.RandomCartPoleVecEnv(n, device="cuda", env_id0=env_id0, **kw)


def _configure(env, pair):
    kind, value = pair
    if kind == "task":
        env.set_task(*[float(v) for v in value])
    else:
        env.set_dr_distribution(kind, value)
        env.set_dr_training(True)
    return env


def _pair(pairs=PAIRS, assign_seed=0, n=N, env_id0=ID0, **kw):
    """(env with scenarios, assignment, [twin per scenario]) of the same settings."""
    env = _env(n, env_id0, **kw)
    a = _assignment(n, len(pairs), assign_seed)
    env.set_scenarios(_scenarios(pairs), a)
    return env, a, [_configure(_env(n, env_id0, **kw), p) for p in pairs]


def _snap(env):
    """Every per-env buffer a step or rollout leaves, as one dict of (N, ...) tensors."""
    return dict(state=env.state.clone(), xi=env.get_task().clone(), elapsed=env.elapsed.clone(),
                episode=env.episode.clone())


def _assert_rows(got, twins_got, a, what=""):
    """got[i] == twins_got[a[i]][i] for every env i (dicts of (N, ...) tensors)."""
    for c, want in enumerate(twins_got):
        m = a == c
        for k in got:
            assert torch.equal(got[k][m], want[k][m]), (what, k, c)


def _check_all(env, twins, a, what=""):
    env.check_dr_violations()
    for t in twins:
        t.check_dr_violations()
    _assert_rows(_snap(env), [_snap(t) for t in twins], a, what)


# ---- reset and step ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["lean", "int32", "logged"])
@pytest.mark.parametrize("limit", [17, 500])
@pytest.mark.parametrize("tile_ordering", [False, True])
def test_reset_and_step_equal_the_twins(layout, limit, tile_ordering):
    kw = dict(max_episode_steps=limit, tile_ordering=tile_ordering, _int32_counter=layout == "int32")
    env, a, twins = _pair(**kw)
    logs = [e.start_episode_log(8) for e in [env] + twins] if layout == "logged" else None
    env.reset()
    for t in twins:
        t.reset()
    _check_all(env, twins, a, "reset")
    for k in range(60):
        out = env.step(env.sample_actions())
        got = dict(obs=out[0].clone(), done=out[2].clone(), trunc=out[3]["TimeLimit.truncated"].clone())
        if layout == "int32":
            got["reward"] = out[1].clone()
        want = []
        for t in twins:
            o = t.step(t.sample_actions())
            want.append(dict(obs=o[0].clone(), done=o[2].clone(), trunc=o[3]["TimeLimit.truncated"].clone()))
            if layout == "int32":
                want[-1]["reward"] = o[1].clone()
        _assert_rows(got, want, a, "step %d" % k)
    _check_all(env, twins, a, "after steps")
    if logs:
        for name in ("_xi", "_final_state", "_length", "_truncated", "_end_tick"):
            _assert_rows({name: getattr(logs[0], name)[:, :N].transpose(0, 1)},
                         [{name: getattr(g, name)[:, :N].transpose(0, 1)} for g in logs[1:]], a, name)
        _assert_rows({"count": logs[0]._count[:N]}, [{"count": g._count[:N]} for g in logs[1:]], a, "count")


def test_step_under_cuda_graph_replay_equals_the_twins():
    env, a, twins = _pair(max_episode_steps=23)
    envs = [env] + twins
    for e in envs:
        e.reset()
    graphs = []
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for e in envs:
            e.step(e.sample_actions())          # warm up: the step plan and the action buffer
    torch.cuda.current_stream().wait_stream(s)
    for e in envs:
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            e.step(e._own_action_view())        # the env's own actions: re-drawn outside the graph
        graphs.append(g)
    for k in range(40):
        for e, g in zip(envs, graphs):
            e.sample_actions()
            g.replay()
    torch.cuda.synchronize()
    for e in envs:
        e._tick = envs[0]._tick
    _check_all(env, twins, a, "graph replay")


# ---- fused rollouts and collect ------------------------------------------------------------------------------------
def _net(act, seed):
    torch.manual_seed(seed)
    net = nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2))
    with torch.no_grad():
        net[-1].weight.mul_(3.0)
    return MLPPolicy.from_module(net, "cuda")


def _episode_rows(log, n):
    """(N, capacity) lengths and a validity mask of every record in the log."""
    count = log._count[:n].long()
    cap = log.capacity
    assert int(count.max()) <= cap, "the log wrapped: records were overwritten"
    length = log._length[:, :n].transpose(0, 1).double()
    valid = torch.arange(cap, device=count.device).view(1, -1) < count.view(-1, 1)
    return length, valid


def _stats_from_logs(twin_logs, a, C, n=N):
    """(C, 6) exact statistics of the episodes the twins' logs recorded for the envs assigned to each scenario."""
    out = torch.tensor([[0.0, 0.0, 0.0, np.inf, -np.inf, 0.0]] * C, dtype=torch.float64, device="cuda")
    for c, log in enumerate(twin_logs):
        length, valid = _episode_rows(log, n)
        valid = valid & (a == c).view(-1, 1)
        if bool(valid.any()):
            v = length[valid]
            out[c] = torch.stack([v.new_tensor(float(v.numel())), v.sum(), (v * v).sum(), v.min(), v.max(), v.sum()])
    return out


@pytest.mark.parametrize("policy", ["linear", "random", "tanh", "relu", "collect-sample", "collect-greedy"])
@pytest.mark.parametrize("integrator", ["euler", "semi-implicit"])
def test_rollouts_and_collect_equal_the_twins(policy, integrator):
    kw = dict(max_episode_steps=40, kinematics_integrator=integrator, _int32_counter=True)
    env, a, twins = _pair(**kw)
    K = 120
    mlp = _net(nn.Tanh if policy == "tanh" else nn.ReLU, 3) if policy not in ("linear", "random") else None
    for e in [env] + twins:
        e.reset()
        e.step(e.sample_actions())                  # mid-episode start
        e.reset_stats()
    logs = [t.start_episode_log(64) for t in twins]
    trajs = []
    for e in [env] + twins:
        if policy == "linear":
            e.rollout((0.1, 0.3, 2.0, 0.4), 0.01, K)
        elif policy == "random":
            e.rollout(None, 0.0, K)
        elif policy.startswith("collect"):
            trajs.append(e.collect(mlp, K, sample=policy == "collect-sample"))
        else:
            e.rollout(mlp, 0.0, K)
    _check_all(env, twins, a, policy)
    for name in ("obs", "actions", "logp", "dones", "truncated", "final_obs") if trajs else ():
        got = getattr(trajs[0], name).transpose(0, 1)
        for c, t in enumerate(trajs[1:]):
            m = a == c
            assert torch.equal(got[m], getattr(t, name).transpose(0, 1)[m]), (name, c)
    want = _stats_from_logs(logs, a, len(PAIRS))
    assert torch.equal(env.scenario_stats(), want)
    combined = random_envs.combine_stats(env.scenario_stats().cpu().numpy())
    assert np.array_equal(env.stats_tensor.cpu().numpy(), combined)
    assert env.episode_stats()["episodes"] == int(want[:, 0].sum())


def test_logged_rollouts_write_the_twins_records():
    env, a, twins = _pair(max_episode_steps=30, _int32_counter=True)
    mlp = _net(nn.ReLU, 4)
    for e in [env] + twins:
        e.reset()
    logs = [e.start_episode_log(32) for e in [env] + twins]
    for e in [env] + twins:
        e.rollout((0.0, 0.0, 1.0, 0.0), 0.0, 50)
        e.rollout(None, 0.0, 50)
        e.rollout(mlp, 0.0, 50)
        e.collect(mlp, 50)
    _check_all(env, twins, a, "logged")
    for name in ("_xi", "_final_state", "_length", "_truncated", "_end_tick"):
        _assert_rows({name: getattr(logs[0], name)[:, :N].transpose(0, 1)},
                     [{name: getattr(g, name)[:, :N].transpose(0, 1)} for g in logs[1:]], a, name)


# ---- C = 1, independence, sharding, checkpoints ----------------------------------------------------------------------
@pytest.mark.parametrize("pair", [PAIRS[0], PAIRS[3], PAIRS[5]])
def test_one_scenario_of_the_envs_own_config_changes_nothing(pair):
    kw = dict(max_episode_steps=25, _int32_counter=True)
    env = _configure(_env(**kw), pair)
    plain = _configure(_env(**kw), pair)
    env.set_scenarios(_scenarios([pair]), torch.zeros(N, dtype=torch.int64))
    mlp = _net(nn.Tanh, 5)
    for e in (env, plain):
        e.reset()
        for _ in range(30):
            e.step(e.sample_actions())
        e.rollout((0.0, 0.2, 1.5, 0.3), 0.0, 60)
        e.rollout(None, 0.0, 60)
        e.rollout(mlp, 0.0, 60)
        e.collect(mlp, 60)
    a = torch.zeros(N, dtype=torch.int64, device="cuda")
    _check_all(env, [plain], a)
    assert torch.equal(env.scenario_stats()[0], plain.stats_tensor)
    assert torch.equal(env.stats_tensor, plain.stats_tensor)


def _run_mix(env, K=80):
    env.reset()
    for _ in range(20):
        env.step(env.sample_actions())
    env.rollout((0.0, 0.2, 1.5, 0.3), 0.0, K)
    env.collect(_net(nn.ReLU, 6), K)
    env.check_dr_violations()
    return _snap(env)


def test_an_env_depends_on_its_own_row_only():
    base, a, _ = _pair(max_episode_steps=30, _int32_counter=True)
    want = _run_mix(base)
    # permute the assignment of the other envs, and append rows that nobody uses
    keep = torch.arange(N, device="cuda") % 3 == 0
    b = torch.where(keep, a, a[torch.randperm(N, device="cuda")])
    other = _env(max_episode_steps=30, _int32_counter=True)
    other.set_scenarios(Scenarios.cat(_scenarios(PAIRS), Scenarios.adr_boundaries([2, 0.5, 0.05, 0.1], [20, 3, 0.3, 1],
                                                                                  device="cuda")), b)
    got = _run_mix(other)
    for k in want:
        assert torch.equal(got[k][keep], want[k][keep]), k


def test_two_shards_equal_the_whole():
    whole, a, _ = _pair(max_episode_steps=30, _int32_counter=True)
    want = _run_mix(whole)
    half = N // 2 + 7
    parts, stats = [], []
    for lo, hi in ((0, half), (half, N)):
        e = _env(hi - lo, ID0 + lo, max_episode_steps=30, _int32_counter=True)
        e.set_scenarios(_scenarios(PAIRS), a[lo:hi])
        parts.append(_run_mix(e))
        stats.append(e.scenario_stats())
    for k in want:
        assert torch.equal(torch.cat([p[k] for p in parts]), want[k]), k
    combined = np.stack([random_envs.combine_stats(np.stack([s[c].cpu().numpy() for s in stats]))
                         for c in range(len(PAIRS))])
    assert np.array_equal(combined, whole.scenario_stats().cpu().numpy())


def test_state_dict_round_trip_and_clearing_restore_behaviour():
    env, a, _ = _pair(max_episode_steps=30, _int32_counter=True)
    _run_mix(env)
    sd = env.state_dict()
    other = _env(max_episode_steps=30, _int32_counter=True)
    other.load_state_dict(sd)
    assert torch.equal(other.scenarios[1], a) and torch.equal(other.scenarios[0], env.scenarios[0])
    assert torch.equal(other.scenario_stats(), env.scenario_stats())
    assert torch.equal(_run_mix(env)["state"], _run_mix(other)["state"])
    assert torch.equal(other.scenario_stats(), env.scenario_stats())
    # set_scenarios(None): the env's own config decides again, the statistics fold into the env-wide row
    before = env.stats_tensor.clone()
    env.set_scenarios(None)
    assert torch.equal(env.stats_tensor, before) and env.scenarios is None
    plain = _env(max_episode_steps=30, _int32_counter=True)
    plain.load_state_dict(env.state_dict())
    _configure(env, PAIRS[0])
    _configure(plain, PAIRS[0])
    got, want = _run_mix(env), _run_mix(plain)
    for k in want:
        assert torch.equal(got[k], want[k]), k


# ---- errors and refusals -------------------------------------------------------------------------------------------
def test_gaussian_failures_from_a_scenario_row_raise_at_the_next_sync():
    env = _env(256)
    bad = Scenarios.distributions("gaussian", [[9.8, 1.0, 1.0, 0.1, 0.01, 0.001, 0.5, 0.05]], "cuda")
    env.set_scenarios(Scenarios.cat(_scenarios(PAIRS[:1]), bad), torch.arange(256) % 2)
    env.reset()
    with pytest.raises(Exception, match="Not all samples"):
        env.check_dr_violations()
    env.check_dr_violations()                       # raised once, then cleared


def test_refusals_while_scenarios_are_set():
    env, a, _ = _pair(n=64)
    with pytest.raises(ValueError, match="set_random_task"):
        env.set_random_task()
    with pytest.raises(ValueError, match="evaluate_population"):
        env.evaluate_population(torch.zeros((2, 5), device="cuda"), 10)
    grid = env.evaluate_grid(torch.zeros((2, 5), device="cuda"), _scenarios(PAIRS[:2]), 10)       # unaffected
    assert tuple(grid.shape) == (2, 2, 6)
    with pytest.raises(ValueError, match="shape"):
        env.set_scenarios(_scenarios(PAIRS), a[:10])
    with pytest.raises(ValueError, match=r"\[0, 7\)"):
        env.set_scenarios(_scenarios(PAIRS), torch.full((64,), 7, device="cuda"))
    env.auto_reset = False
    with pytest.raises(ValueError, match="auto_reset"):
        env.step(env.sample_actions())
    env.auto_reset = True
    env.noisy = True
    with pytest.raises(ValueError, match="observation noise"):
        env.reset()
    env.noisy = False
    # the caller's assignment tensor is copied: editing it afterwards changes nothing
    b = a.clone()
    env.set_scenarios(_scenarios(PAIRS), b)
    b.fill_(99)
    assert torch.equal(env.scenarios[1], a)
