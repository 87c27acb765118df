"""Host-side mirror of RandomEnv / RandomCartPoleEnv: everything that needs no GPU.

Mirrors the call sequence of the reference's usage scripts (test.py:9-15, README.md:52-66) and the
error conventions of random_env.py / random_cartpole.py.  Cross-checked live against the real reference
when /root/reference is mounted.
"""
import os

import numpy as np
import pytest

import random_envs_b200 as random_envs
from random_envs_b200 import gym
from oracle import reference_loader as rl

needs_ref = pytest.mark.skipif(not rl.available(), reason=rl.UNAVAILABLE)
SEARCH = [2, 20, 0.5, 3, 0.05, 0.3, 0.1, 1.0]


def test_make_returns_timelimit_500_and_forwards_attributes():
    env = gym.make("RandomCartPole-v0")
    assert type(env).__name__ == "TimeLimit" and env._max_episode_steps == 500
    assert isinstance(env.unwrapped, random_envs.RandomCartPoleEnv)
    assert env.task_dim == 4 and env.reward_threshold == 500 and env.get_reward_threshold() == 500
    assert list(env.get_task()) == [9.8, 1.0, 0.1, 0.5]
    assert env.action_space.n == 2 and env.observation_space.shape == (4,)
    assert env.observation_space.dtype == np.float32
    assert [env.dyn_index_to_name(i) for i in range(4)] == ["gravity", "cart_mass", "pole_mass", "pole_length"]


def test_set_task_keeps_polemass_length_stale():
    env = random_envs.RandomCartPoleEnv()
    env.set_task(5.0, 2.0, 0.2, 0.8)
    assert env.total_mass == 2.2 and env.polemass_length == 0.05
    assert list(env.get_task()) == [5.0, 2.0, 0.2, 0.8]


def test_dr_distribution_semantics():
    env = gym.make("RandomCartPole-v0")
    assert env.get_dr_distribution() is None and env.get_dr_training() is False
    env.set_dr_distribution(dr_type="uniform", distr=SEARCH)
    lo, hi = env.get_dr_distribution()
    assert list(lo) == [2, 0.5, 0.05, 0.1] and list(hi) == [20, 3, 0.3, 1.0] and env.sampling == "uniform"
    env.set_dr_training(True)
    assert env.get_dr_training() is True
    env.set_dr_distribution("truncnorm", [9.8, 1.0, 1.0, 0.1])          # short list sets a prefix
    mu, sd = env.get_dr_distribution()
    assert list(mu) == [9.8, 1.0, 0, 0] and list(sd) == [1.0, 0.1, 0, 0]
    env.set_dr_distribution("gaussian", [9.8, 1.0, 1.0, 0.1, 0.1, 0.01, 0.5, 0.05])
    with pytest.raises(ValueError, match="Not implemented"):
        env.get_dr_distribution()
    with pytest.raises(Exception, match="Unknown dr_type:beta"):
        env.set_dr_distribution("beta", [1, 2])
    with pytest.raises(IndexError):
        env.set_dr_distribution("uniform", list(range(10)))              # 5 pairs into a 4-dim env
    env.set_dr_distribution("fullgaussian", {"mean": [1, 2, 3, 4], "cov": np.eye(4)})
    assert env.sampling == "fullgaussian" and env.cov_task.shape == (4, 4) and list(env.mean_task) == [1, 2, 3, 4]


def test_sampling_unset_and_no_gpu_errors():
    env = random_envs.RandomCartPoleEnv()
    with pytest.raises(ValueError, match="sampling value of random env needs to be set"):
        env.sample_task()
    with pytest.raises(ValueError, match="sampling value of random env needs to be set"):
        env.set_random_task()
    import torch
    if not torch.cuda.is_available():
        env.set_dr_distribution("uniform", SEARCH)
        for call in (env.sample_task, env.reset, lambda: random_envs.RandomCartPoleVecEnv(8).reset()):
            with pytest.raises(RuntimeError, match="no CPU fallback"):
                call()


def test_invalid_actions_are_rejected_before_any_device_work():
    env = random_envs.RandomCartPoleEnv()
    env.state = (0.0, 0.0, 0.0, 0.0)
    for bad in (2, -1, 1.0, np.float32(1.0), "1", np.array([1])):
        with pytest.raises(AssertionError, match="invalid"):
            env.step(bad)


def test_search_bounds_helpers():
    env = random_envs.RandomCartPoleEnv()
    lo, hi = env.get_task_search_bounds()
    assert list(lo) == [2.0, 0.5, 0.05, 0.1] and list(hi) == [20.0, 3.0, 0.3, 1.0]
    env.set_task_search_bounds()
    assert list(env.min_task) == list(lo) and list(env.max_task) == list(hi)
    assert np.allclose(env.denormalize_parameters(np.array([0.0, 4.0, 2.0, 1.0])), [2.0, 3.0, 0.175, 0.325])
    assert [env.get_task_lower_bound(i) for i in range(4)] == [0.1] * 4


def test_load_dr_distribution_from_file(tmp_path):
    env = random_envs.RandomCartPoleEnv()
    f = tmp_path / "dr.csv"
    f.write_text("truncnorm\n9.8,1.0,1.0,0.1,0.1,0.01,0.5,0.05\n")
    env.load_dr_distribution_from_file(str(f))
    assert env.sampling == "truncnorm" and list(env.mean_task) == [9.8, 1.0, 0.1, 0.5]
    f.write_text("uniform\n1,2,3\n")
    with pytest.raises(Exception, match="right number of column values"):
        env.load_dr_distribution_from_file(str(f))
    f.write_text("cauchy\n1,2,3,4,5,6,7,8\n")
    with pytest.raises(Exception, match="Filename is wrongly formatted"):
        env.load_dr_distribution_from_file(str(f))


def test_xi_tables_cover_the_suite():
    T = random_envs.XI_TABLES
    dims = {k: len(v.names) for k, v in T.items()}
    assert dims == {"RandomCartPole-v0": 4, "RandomHopper-v0": 4, "RandomHopperNoisy-v0": 4, "RandomHopperUnmodeled-v0": 3,
                    "RandomHalfCheetah-v0": 8, "RandomHalfCheetahNoisy-v0": 8, "RandomHalfCheetahUnmodeled-v0": 5,
                    "RandomWalker2d-v0": 13, "RandomWalker2dNoisy-v0": 13, "RandomWalker2dUnmodeled-v0": 9,
                    "RandomHumanoid-v0": 30, "RandomHumanoidNoisy-v0": 30, "RandomHumanoidUnmodeled-v0": 23}
    h = T["RandomHumanoid-v0"]
    assert h.lower_bounds == tuple([0.2] * 13 + [0.8] * 6 + [0.15] + [0.8] * 3 + [0.15] * 7)
    assert h.search_bounds[13] == (1.0, 10.0) and h.search_bounds[19] == (0.2, 5.0) and h.names[19] == "damp7"
    assert T["RandomHopperUnmodeled-v0"].lower_bounds == (0.001,) * 3
    assert T["RandomWalker2dUnmodeled-v0"].lower_bounds == (0.1, 0.1, 0.1, 0.1, 0.25, 0.25, 0.12, 0.05, 0.05)
    assert T["RandomHalfCheetah-v0"].search_bounds[7] == (0.1, 2.0) and T["RandomHalfCheetah-v0"].lower_bounds[7] == 0.02
    s = random_envs.TaskSampler("RandomHumanoid-v0")
    assert s.task_dim == 30 and s.dyn_index_to_name(29) == "damp17" and s.preferred_lr == 0.0001
    cfg = s.dr_config()
    assert cfg.dr_type == 0
    s.set_dr_distribution("truncnorm", list(np.stack([random_envs.HUMANOID_NOMINAL, 0.1 * np.array(random_envs.HUMANOID_NOMINAL)], 1).reshape(-1)))
    cfg = s.dr_config()
    assert cfg.dr_type == 2 and cfg.dim == 30 and cfg.lb[29] == 0.15 and cfg.a[0] == 8.322


def test_shard_range_partitions_exactly():
    for total, world in [(1 << 20, 8), (1000003, 8), (7, 8), (64, 1)]:
        spans = [random_envs.shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and spans[-1][1] == total
        assert all(spans[i][1] == spans[i + 1][0] for i in range(world - 1))
        sizes = [b - a for a, b in spans]
        assert max(sizes) - min(sizes) <= 1


def test_stats_combine_and_summary():
    a = [[2, 30, 500, 10, 20, 30], [1, 500, 250000, 500, 500, 500], [0, 0, 0, np.inf, -np.inf, 0]]
    c = random_envs.combine_stats(a)
    assert list(c) == [3, 530, 250500, 10, 500, 530]
    s = random_envs.summarize_stats(c)
    assert s["episodes"] == 3 and abs(s["mean_return"] - 530 / 3) < 1e-12 and s["max_return"] == 500
    assert np.isnan(random_envs.summarize_stats([0, 0, 0, np.inf, -np.inf, 0])["mean_return"])


@needs_ref
def test_attribute_surface_matches_live_reference():
    ref = rl.make_cartpole()
    mine = random_envs.RandomCartPoleEnv()
    for name in ("gravity", "cart_mass", "pole_mass", "total_mass", "pole_length", "polemass_length", "force_mag", "tau",
                 "kinematics_integrator", "theta_threshold_radians", "x_threshold", "task_dim", "reward_threshold",
                 "dyn_ind_to_name", "sampling", "dr_training", "preferred_lr", "steps_beyond_done", "state"):
        assert getattr(ref, name) == getattr(mine, name), name
    for name in ("min_task", "max_task", "mean_task", "stdev_task", "original_task"):
        assert np.array_equal(getattr(ref, name), getattr(mine, name)), name
    public = [m for m in dir(ref) if not m.startswith("_") and callable(getattr(ref, m))]
    missing = [m for m in public if not hasattr(mine, m)]
    assert missing == [], missing
    for i in range(4):
        assert ref.get_search_bounds_mean(i) == mine.get_search_bounds_mean(i)
        assert ref.get_task_lower_bound(i) == mine.get_task_lower_bound(i)
    # same behaviour of the distribution setters on both
    for dr_type, distr in [("uniform", SEARCH), ("truncnorm", [9.8, 1.0, 1.0, 0.1]), ("gaussian", [1, 2, 3, 4, 5, 6, 7, 8])]:
        ref.set_dr_distribution(dr_type, distr); mine.set_dr_distribution(dr_type, distr)
        for name in ("min_task", "max_task", "mean_task", "stdev_task"):
            assert np.array_equal(getattr(ref, name), getattr(mine, name)), (dr_type, name)
        assert ref.sampling == mine.sampling


def test_reference_module_names_resolve_to_this_implementation():
    """`import random_envs` + `import gym` (README.md:52-54) work as a literal drop-in."""
    import importlib
    import sys
    alias = importlib.import_module("random_envs")
    assert alias.RandomCartPoleEnv is random_envs.RandomCartPoleEnv
    from random_envs.random_cartpole import RandomCartPoleEnv as A
    from random_envs.random_env import RandomEnv as B
    assert A is random_envs.RandomCartPoleEnv and B is random_envs.RandomEnv and issubclass(A, B)
    had_gym = "gym" in sys.modules
    g = alias.install_gym()
    try:
        import gym as gym_mod
        env = gym_mod.make("RandomCartPole-v0")
        assert env.unwrapped.__class__ is A and g is gym_mod
    finally:
        if not had_gym and not random_envs.gym_compat.HAVE_REAL_GYM:
            sys.modules.pop("gym", None)
