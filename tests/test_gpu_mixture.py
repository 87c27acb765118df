"""Scenario mixtures on the GPU: every reset draws its row from the alias table (purpose 6), and env i then equals a
set_scenarios twin whose assignment is set to the drawn rows before each step, bit for bit; the fused rollouts and
collect equal K steps; per-row statistics equal the episode log attributed on the host; the law of the draw; C = 1 and
C > 64; set_mixture_weights mid-run; shards, checkpoints, clearing and the refusals."""
import numpy as np
import pytest
import torch
from scipy import stats as sps
from torch import nn

import mixture_oracle
import random_envs_b200 as random_envs
from random_envs_b200 import MLPPolicy, Scenarios
from random_envs_b200.vector_env import _mixture_table

pytestmark = pytest.mark.gpu

COV = [[0.30, 0.05, 0.00, 0.02], [0.05, 0.20, 0.03, 0.00], [0.00, 0.03, 0.25, 0.04], [0.02, 0.00, 0.04, 0.30]]
PAIRS = [
    ("uniform", [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]),
    ("truncnorm", [9.8, 1.0, 1.0, 0.2, 0.5, 0.05, 0.5, 0.1]),
    ("gaussian", [9.8, 1.0, 1.0, 0.1, 0.5, 0.05, 0.5, 0.05]),
    ("fullgaussian", {"mean": [2.0, 1.5, 2.5, 2.0], "cov": COV}),
    ("task", [15.5, 0.75, 0.2, 0.25]),
    ("task", [4.0, 2.5, 0.05, 0.9]),
]
WEIGHTS = [3.0, 1.0, 0.0, 2.0, 1.5, 0.5]          # row 2 is never drawn
N = 3000
SEED, ID0 = 11, 5


def _scenarios(pairs=PAIRS):
    return Scenarios.cat(*[Scenarios.tasks([v], "cuda") if k == "task" else Scenarios.distributions(k, [v], "cuda")
                           for k, v in pairs])


def _env(n=N, env_id0=ID0, **kw):
    kw.setdefault("seed", SEED)
    return random_envs.RandomCartPoleVecEnv(n, device="cuda", env_id0=env_id0, **kw)


def _draws(env, tick):
    """The oracle's row of every env for a reset at ``tick``, on the env's device."""
    table = env._scen["table"].cpu().numpy()
    ids = env.env_id0 + np.arange(env.num_envs)
    return torch.from_numpy(mixture_oracle.draw_rows(env._seed, ids, tick, table)).cuda()


def _pair(weights=WEIGHTS, pairs=PAIRS, n=N, **kw):
    env, twin = _env(n, **kw), _env(n, **kw)
    env.set_scenario_mixture(_scenarios(pairs), weights)
    twin.set_scenarios(_scenarios(pairs), torch.zeros(n, dtype=torch.int64))
    return env, twin


def _aim(twin, env):
    """Set the twin's assignment to the rows the mixture env's next reset draws."""
    twin._scen["of_env"][:twin.num_envs].copy_(_draws(env, env._tick).to(torch.int16))


def _snap(env):
    return dict(state=env.state.clone(), xi=env.get_task().clone(), elapsed=env.elapsed.clone(),
                episode=env.episode.clone())


def _assert_same(a, b, what=""):
    for k in a:
        assert torch.equal(a[k], b[k]), (what, k)


def _of_env(env):
    return env.scenarios[1]


# ---- reset and step ------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("layout", ["lean", "int32", "logged"])
@pytest.mark.parametrize("tile_ordering", [False, True])
@pytest.mark.parametrize("integrator", ["euler", "semi-implicit"])
def test_step_loop_equals_a_reassigned_twin(layout, tile_ordering, integrator):
    kw = dict(max_episode_steps=17, tile_ordering=tile_ordering, _int32_counter=layout == "int32",
              kinematics_integrator=integrator)
    env, twin = _pair(**kw)
    logs = [e.start_episode_log(8) for e in (env, twin)] if layout == "logged" else None
    assert torch.equal(_of_env(env), torch.full((N,), len(PAIRS), device="cuda"))
    _aim(twin, env)
    want_rows = _draws(env, env._tick)
    env.reset()
    twin.reset()
    assert torch.equal(_of_env(env), want_rows)
    _assert_same(_snap(env), _snap(twin), "reset")
    for k in range(50):
        draws = _draws(env, env._tick)
        _aim(twin, env)
        before = _of_env(env)
        o = env.step(env.sample_actions())
        w = twin.step(twin.sample_actions())
        assert torch.equal(o[0], w[0]) and torch.equal(o[2], w[2]), k
        assert torch.equal(o[3]["TimeLimit.truncated"], w[3]["TimeLimit.truncated"]), k
        assert torch.equal(_of_env(env), torch.where(o[2], draws, before)), k
    _assert_same(_snap(env), _snap(twin), "steps")
    if logs:
        for name in ("_xi", "_final_state", "_length", "_truncated", "_end_tick", "_count"):
            assert torch.equal(getattr(logs[0], name), getattr(logs[1], name)), name
    assert int(torch.bincount(_of_env(env), minlength=len(PAIRS) + 1)[2]) == 0


def test_step_under_cuda_graph_replay_equals_the_twin():
    env, twin = _pair(max_episode_steps=23)
    _aim(twin, env)
    for e in (env, twin):
        e.reset()
    _aim(twin, env)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for e in (env, twin):
            e.step(e.sample_actions())          # warm up: the step plan and the action buffer
    torch.cuda.current_stream().wait_stream(s)
    captured_tick = env._tick                   # a replay repeats the clock of its capture
    graphs = []
    for e in (env, twin):
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            e.step(e._own_action_view())
        graphs.append(g)
    twin._scen["of_env"][:N].copy_(_draws(env, captured_tick).to(torch.int16))
    for k in range(40):
        for e, g in zip((env, twin), graphs):
            e.sample_actions()
            g.replay()
    torch.cuda.synchronize()
    _assert_same(_snap(env), _snap(twin), "graph replay")


# ---- fused rollouts and collect against K steps --------------------------------------------------------------------
def _net(act, seed):
    torch.manual_seed(seed)
    net = nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2))
    with torch.no_grad():
        net[-1].weight.mul_(3.0)
    return MLPPolicy.from_module(net, "cuda")


TRAJ_FIELDS = ("obs", "actions", "logp", "dones", "truncated")
LINEAR = ((0.1, 0.3, 2.0, 0.4), 0.01)


@pytest.mark.parametrize("policy", ["random", "linear", "tanh", "relu", "collect-greedy", "collect-sample"])
@pytest.mark.parametrize("integrator", ["euler", "semi-implicit"])
def test_rollouts_and_collect_equal_k_steps(policy, integrator):
    """A fused K-step launch under the mixture equals K single steps under it: step() with the random policy's or the
    MLP's actions (policy_actions, sampled with its logp for collect), and for the linear policy K one-step
    rollouts, whose draws and row flushes then happen at launch boundaries instead of inside one launch."""
    kw = dict(max_episode_steps=40, kinematics_integrator=integrator, _int32_counter=True)
    fused, stepped = _env(**kw), _env(**kw)
    mlp = None if policy in ("random", "linear") else _net(nn.Tanh if policy == "tanh" else nn.ReLU, 3)
    collect = policy.startswith("collect")
    logs = []
    for e in (fused, stepped):
        e.reset()
        e.step(e.sample_actions())                  # episodes running at install time: row C
        e.set_scenario_mixture(_scenarios(), WEIGHTS)
        logs.append(e.start_episode_log(64))
    K = 120
    if policy == "random":
        fused.rollout(None, 0.0, K)
    elif policy == "linear":
        fused.rollout(*LINEAR, K)
    elif collect:
        traj = fused.collect(mlp, K, sample=policy == "collect-sample")
    else:
        fused.rollout(mlp, 0.0, K)
    rows = {f: [] for f in TRAJ_FIELDS}
    for k in range(K):
        if policy == "linear":
            stepped.rollout(*LINEAR, 1)
            continue
        if mlp is None:
            a = stepped.sample_actions()
        else:
            a, logp = stepped.policy_actions(mlp, sample=policy == "collect-sample", return_logp=True)
            rows["logp"].append(logp.clone())
        rows["obs"].append(stepped.obs.clone())
        rows["actions"].append(a.clone())
        _, _, done, info = stepped.step(a)
        rows["dones"].append(done.clone())
        rows["truncated"].append(info["TimeLimit.truncated"].clone())
    _assert_same(_snap(fused), _snap(stepped), policy)
    assert torch.equal(_of_env(fused), _of_env(stepped))
    for name in ("_xi", "_final_state", "_length", "_truncated", "_end_tick", "_count"):
        assert torch.equal(getattr(logs[0], name), getattr(logs[1], name)), name
    if collect:
        for f in TRAJ_FIELDS:
            got, want = getattr(traj, f), torch.stack(rows[f])
            assert torch.equal(got, want.to(got.dtype)), f
    if policy == "linear":
        assert torch.equal(fused._scen["stats"], stepped._scen["stats"])
    _check_stats(fused, logs[0], install_tick=fused._tick - K)


def _check_stats(env, log, install_tick):
    """scenario_stats() and stats_tensor against the log's records, each attributed to the oracle's draw at its reset
    tick (end tick - length), or to row C when the episode began before the mixture was installed."""
    C = env._scen["rows"].shape[0]
    table = env._scen["table"].cpu().numpy()
    count = log._count[:env.num_envs].cpu().numpy()
    assert count.max() <= log.capacity
    length = log._length[:, :env.num_envs].cpu().numpy()
    end = log._end_tick[:, :env.num_envs].cpu().numpy()
    want = np.tile(np.array([0.0, 0.0, 0.0, np.inf, -np.inf, 0.0]), (C + 1, 1))
    for i in np.nonzero(count)[0]:
        L, E = length[:count[i], i].astype(np.int64), end[:count[i], i]
        start = E - L
        rows = mixture_oracle.draw_rows(env._seed, env.env_id0 + i, start, table)
        rows = np.where(start < install_tick, C, rows)
        for r, l in zip(rows, L):
            want[r] += [1, l, l * l, 0, 0, l]
            want[r, 3], want[r, 4] = min(want[r, 3], l), max(want[r, 4], l)
    got = env.scenario_stats().cpu().numpy()
    assert np.array_equal(got, want[:C])
    assert np.array_equal(env._scen["stats"].cpu().numpy(), want)
    assert np.array_equal(env.stats_tensor.cpu().numpy(), random_envs.combine_stats(want))


def test_statistics_beyond_64_rows_use_the_global_path():
    rng = np.random.default_rng(1)
    C = 100
    tasks = np.column_stack([rng.uniform(5, 15, C), rng.uniform(0.5, 2, C), rng.uniform(0.05, 0.3, C),
                             rng.uniform(0.2, 1.0, C)])
    env = _env(max_episode_steps=30, _int32_counter=True)
    env.reset()
    env.set_scenario_mixture(Scenarios.tasks(tasks, "cuda"), rng.random(C))
    log = env.start_episode_log(64)
    t0 = env._tick
    env.rollout(_net(nn.ReLU, 2), 0.0, 90)
    env.rollout(None, 0.0, 90)
    env.collect(_net(nn.Tanh, 4), 90)
    _check_stats(env, log, t0)


def test_law_of_the_draw_over_a_million_resets():
    n = 1 << 20
    env = _env(n)
    w = np.array(WEIGHTS)
    env.set_scenario_mixture(_scenarios(), w)
    env.reset()
    rows = _of_env(env)
    assert torch.equal(rows, _draws(env, env._tick - 1))
    counts = torch.bincount(rows, minlength=len(w)).cpu().numpy()
    assert counts[2] == 0
    keep = w > 0
    expected = n * w[keep] / w.sum()
    chi2 = ((counts[keep] - expected) ** 2 / expected).sum()
    assert sps.chi2.sf(chi2, keep.sum() - 1) > 1e-4, (counts, expected)


def test_one_row_equals_set_scenarios_with_a_zero_assignment():
    kw = dict(max_episode_steps=25, _int32_counter=True)
    env, twin = _pair(weights=[1.0], pairs=PAIRS[:1], **kw)
    mlp = _net(nn.Tanh, 5)
    for e in (env, twin):
        e.reset()
        for _ in range(30):
            e.step(e.sample_actions())
        e.rollout(None, 0.0, 60)
        e.rollout(mlp, 0.0, 60)
        e.collect(mlp, 60)
    _assert_same(_snap(env), _snap(twin))
    assert torch.equal(_of_env(env), torch.zeros(N, dtype=torch.int64, device="cuda"))
    assert torch.equal(env.scenario_stats(), twin.scenario_stats())


def test_new_weights_act_at_the_next_resets_only():
    env = _env(max_episode_steps=30, _int32_counter=True)
    env.set_scenario_mixture(_scenarios(), WEIGHTS)
    env.reset()
    env.rollout(None, 0.0, 40)
    stats_before = env._scen["stats"].clone()
    rows_before = _of_env(env)
    w2 = [0.0, 0.0, 1.0, 0.0, 0.0, 1.0]
    env.set_mixture_weights(w2)
    assert np.array_equal(env.scenario_weights, w2)
    assert torch.equal(_of_env(env), rows_before)               # running episodes keep their row
    assert torch.equal(env._scen["stats"], stats_before)        # and the statistics carry over
    draws = _draws(env, env._tick)
    o = env.step(env.sample_actions())
    assert torch.equal(_of_env(env), torch.where(o[2], draws, rows_before))
    assert set(draws[o[2]].unique().tolist()) <= {2, 5}


def _run(env, K=80):
    env.reset()
    for _ in range(20):
        env.step(env.sample_actions())
    env.rollout(None, 0.0, K)
    env.collect(_net(nn.ReLU, 6), K)
    env.check_dr_violations()
    return dict(_snap(env), of_env=_of_env(env)) if env.scenarios is not None else _snap(env)


def test_two_shards_equal_the_whole():
    whole = _env(max_episode_steps=30, _int32_counter=True)
    whole.set_scenario_mixture(_scenarios(), WEIGHTS)
    want = _run(whole)
    half = N // 2 + 7
    parts, stats = [], []
    for lo, hi in ((0, half), (half, N)):
        e = _env(hi - lo, ID0 + lo, max_episode_steps=30, _int32_counter=True)
        e.set_scenario_mixture(_scenarios(), WEIGHTS)
        parts.append(_run(e))
        stats.append(e._scen["stats"])
    for k in want:
        assert torch.equal(torch.cat([p[k] for p in parts]), want[k]), k
    combined = np.stack([random_envs.combine_stats(np.stack([s[c].cpu().numpy() for s in stats]))
                         for c in range(len(PAIRS) + 1)])
    assert np.array_equal(combined, whole._scen["stats"].cpu().numpy())


def test_checkpoint_resume_and_clearing():
    env = _env(max_episode_steps=30, _int32_counter=True)
    env.set_scenario_mixture(_scenarios(), WEIGHTS)
    _run(env)
    sd = env.state_dict()
    assert sd["scenarios"] is None and "mixture" in sd
    other = _env(max_episode_steps=30, _int32_counter=True)
    other.load_state_dict(sd)
    assert np.array_equal(other.scenario_weights, WEIGHTS)
    saved = sd["mixture"]["table"].clone()
    spare = _env(max_episode_steps=30, _int32_counter=True)
    spare.load_state_dict(sd)
    spare.set_mixture_weights([1.0] * len(PAIRS))           # rewrites spare's table, never the checkpoint's
    assert torch.equal(sd["mixture"]["table"], saved) and torch.equal(other._scen["table"], saved)
    _assert_same(_run(env), _run(other), "resumed")
    assert torch.equal(other._scen["stats"], env._scen["stats"])
    plain = _env(max_episode_steps=30, _int32_counter=True)
    assert "mixture" not in plain.state_dict()
    before = env.stats_tensor.clone()
    env.set_scenarios(None)
    assert env.scenarios is None and env.scenario_weights is None
    assert torch.equal(env.stats_tensor, before)
    plain.load_state_dict(env.state_dict())
    _assert_same(_run(env), _run(plain), "cleared")


def test_refusals_while_a_mixture_is_set():
    env = _env(64)
    env.set_scenario_mixture(_scenarios(), WEIGHTS)
    with pytest.raises(ValueError, match="set_random_task.*mixture"):
        env.set_random_task()
    with pytest.raises(ValueError, match="evaluate_population.*mixture"):
        env.evaluate_population(torch.zeros((2, 5), device="cuda"), 10)
    env.auto_reset = False
    with pytest.raises(ValueError, match="mixture.*auto_reset"):
        env.step(env.sample_actions())
    env.auto_reset = True
    env.noisy = True
    with pytest.raises(ValueError, match="mixture.*observation noise"):
        env.reset()
    env.noisy = False
    with pytest.raises(ValueError, match="shape"):
        env.set_mixture_weights([1.0, 2.0])
