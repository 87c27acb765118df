"""random_envs_b200 -- B200-native domain-randomised RandomCartPole-v0 hot path.

Drop-in for the CartPole / DR-sampler slice of gabrieletiboni/random-envs::

    import random_envs_b200 as random_envs          # registers RandomCartPole-v0 (as `import random_envs` does)
    from random_envs_b200 import gym                # real gym when installed, else the bundled gym-0.21 subset
    env = gym.make('RandomCartPole-v0')
    env.set_dr_distribution(dr_type='uniform', distr=[2, 20, 0.5, 3, 0.05, 0.3, 0.1, 1.0])
    env.set_dr_training(True)

and the batched variant of the same calls::

    venv = random_envs.RandomCartPoleVecEnv(1 << 20)        # torch CUDA tensors in / out
    obs = venv.reset(); obs, reward, done, info = venv.step(actions)

and offline DR fitting on recorded transitions::

    data = random_envs.TransitionDataset(obs, actions, next_obs, episode_starts=starts)
    ll = data.dr_log_likelihood("truncnorm", candidates, num_samples=1024)     # one log-likelihood per candidate

All compute is in hand-written sm_100a CUDA kernels behind the C ABI of include/renv.h
(librenv_b200.so, loaded with ctypes).  There is no CPU fallback: without the library or without a
GPU the compute entry points raise.
"""
from . import gym_compat as gym
from . import _lib
from .distributed import allgather_stats, combine_stats, make_sharded_env, shard_range, summarize_stats
from .episode_log import EpisodeLog
from .mlp_policy import MLPPolicy, MLPPopulation
from .offline_dr import TransitionDataset
from .random_cartpole import RandomCartPoleEnv
from .random_env import RandomEnv, TaskSampler
from .trajectory import Trajectory
from .vector_env import RandomCartPoleVecEnv
from .gym_vector import RandomCartPoleGymVectorEnv
from .xi_tables import HUMANOID_NOMINAL, XI_TABLES

__all__ = ["gym", "RandomEnv", "TaskSampler", "RandomCartPoleEnv", "RandomCartPoleVecEnv", "RandomCartPoleGymVectorEnv", "EpisodeLog", "MLPPolicy", "MLPPopulation", "Trajectory", "TransitionDataset", "XI_TABLES",
           "HUMANOID_NOMINAL", "shard_range", "combine_stats", "summarize_stats", "allgather_stats",
           "make_sharded_env", "load_library"]

__version__ = "0.1.0"


def load_library():
    """Load librenv_b200.so and verify every symbol of include/renv.h (raises if anything is missing)."""
    return _lib.load()
