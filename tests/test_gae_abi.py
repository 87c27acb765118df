"""Advantage estimation without a GPU: argument validation of renv_cartpole_gae_mlp_f32, the compiled form of its
kernels, the ctypes binding, MLPPolicy.outputs, the Trajectory views and the host-side rejections of gae()."""
import ctypes
import math
import os
import re
import sys

import pytest
import torch
from torch import nn

import random_envs_b200 as random_envs
from abi_support import ROOT, fake_env as _env, fake_policy as _critic, fake_traj as _traj, ptxas_blocks
from random_envs_b200 import MLPPolicy, Trajectory, _device, _lib, build as lib_build


def _rc(env="ok", critic="ok", traj="ok", K=5, gamma=0.99, lam=0.95, values=16384, advantages=20480, returns=24576):
    lib = _lib.load()
    env = _env() if env == "ok" else env
    critic = _critic() if critic == "ok" else critic
    traj = _traj() if traj == "ok" else traj
    ref = lambda s: ctypes.byref(s) if s is not None else None
    return lib.renv_cartpole_gae_mlp_f32(ref(env), ref(critic), ref(traj), K, gamma, lam, values, advantages, returns,
                                         None)


def test_gae_validates_arguments_before_any_cuda_call():
    # every call below fails validation, so none of the fake device pointers is ever touched
    assert _rc(env=None) == -1
    assert _rc(env=_env(state=None)) == -1
    assert _rc(critic=None) == -1
    assert _rc(critic=_critic(params=None)) == -1
    assert _rc(traj=None) == -1
    for f in ("obs", "done", "truncated", "final_obs"):
        assert _rc(traj=_traj(**{f: None})) == -1, f
    for f in ("action", "logp"):                                        # not read: may be NULL
        assert _rc(traj=_traj(**{f: None}), K=9) == -7, f               # (K > capacity: past the NULL checks)
    for f in ("values", "advantages", "returns"):
        assert _rc(**{f: None}) == -1, f
    assert _rc(env=_env(state=4100)) == -2
    assert _rc(env=_env(ld=14)) == -2                                   # ld not a multiple of 4
    assert _rc(critic=_critic(params=4100)) == -2
    for f, v in (("obs", 4104), ("final_obs", 4104), ("done", 4097), ("truncated", 4098)):
        assert _rc(traj=_traj(**{f: v})) == -2, f
    for f in ("values", "advantages", "returns"):
        assert _rc(**{f: 16386}) == -2, f
    for K in (0, -1):
        assert _rc(K=K) == -3, K
    assert _rc(env=_env(n=0)) == -3
    assert _rc(env=_env(n=13)) == -3                                    # ld < n
    assert _rc(K=9) == -7                                               # K > capacity
    assert _rc(traj=_traj(capacity=0), K=1) == -7
    assert _rc(critic=_critic(act=2)) == -7                             # unknown activation
    for bad in (-1e-3, 1.001, math.nan, math.inf, -math.inf):
        assert _rc(gamma=bad) == -7, bad
        assert _rc(lam=bad) == -7, bad


def test_gae_entry_point_is_bound_with_float_gamma_and_lambda():
    restype, argtypes = _lib.SIGNATURES["renv_cartpole_gae_mlp_f32"]
    assert restype is ctypes.c_int and len(argtypes) == 10
    assert argtypes[3] is ctypes.c_int and argtypes[4] is ctypes.c_float and argtypes[5] is ctypes.c_float
    assert argtypes[2] is ctypes.POINTER(_lib.Trajectory)
    assert _lib.load().renv_cartpole_gae_mlp_f32.argtypes == argtypes


def test_gae_kernels_use_the_tensor_cores_without_spills_or_local_memory():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    names = [n for n in sass if "cartpole_gae_mlp_kernel" in n]
    assert len(names) == 2, names                                       # Tanh and ReLU
    blocks = ptxas_blocks()
    for name in names:
        ops = [op for _, op, _ in sass[name]]
        hmma = sum(o.startswith("HMMA.1688.F32.TF32") for o in ops)
        assert hmma > 0 and hmma % 192 == 0, (name, hmma)                # whole copies of mlp_logits
        assert not any(o.startswith("MUFU.TANH") for o in ops), name     # the accurate tanhf, not tanh.approx
        assert not any(o.startswith(("LDL", "STL")) for o in ops), name
        b = blocks[name]
        assert re.search(r"\b0 bytes stack frame, 0 bytes spill stores, 0 bytes spill loads", b), name
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        assert regs <= 168, (name, regs)                                 # 3 CTAs of 128 threads per SM


@pytest.fixture
def cpu_device(monkeypatch):
    """Let the host-side code build policies and env buffers on the CPU: nothing here launches a kernel."""
    monkeypatch.setattr(_device, "require_cuda", lambda device=None: torch.device("cpu"))


def _net(o, act=nn.Tanh, h1=64, h2=64):
    torch.manual_seed(0)
    return nn.Sequential(nn.Linear(4, h1), act(), nn.Linear(h1, h2), act(), nn.Linear(h2, o))


def test_mlp_policy_records_the_width_of_its_head(cpu_device):
    assert MLPPolicy.from_module(_net(1)).outputs == 1
    assert MLPPolicy.from_module(_net(2)).outputs == 2
    assert MLPPolicy.from_module(_net(1, nn.ReLU, 32, 48)).outputs == 1
    params, act = random_envs.mlp_policy.pack(_net(1))
    assert MLPPolicy(params, act, "cpu").outputs == 2                    # the default: a policy head
    with pytest.raises(ValueError):
        MLPPolicy(params, act, "cpu", outputs=3)


def test_gae_views_belong_to_the_collect_they_were_computed_for():
    n, ld, cap = 5, 32, 4
    tr = Trajectory(n, ld, cap, "cpu")
    assert tr.values is None and tr._values is None
    tr.num_steps, tr.tick0 = 3, 17
    assert tr.values is None and tr.advantages is None and tr.returns is None
    storage = tr._gae_storage()
    assert all(s.shape == (cap, ld) and s.dtype == torch.float32 for s in storage)
    tr._gae_done()
    for f in ("values", "advantages", "returns"):
        v = getattr(tr, f)
        assert v.shape == (3, n) and v.stride() == (ld, 1), f
    assert tr.values.data_ptr() == storage[0].data_ptr()
    assert all(a is b for a, b in zip(tr._gae_storage(), storage))      # allocated once, reused
    tr.num_steps, tr.tick0 = 2, 20                                       # the next collect into the same buffer
    assert tr.values is None and tr.advantages is None and tr.returns is None
    tr.tick0 = 20                                                        # even at the same clock (after seed())
    assert tr.values is None


def test_gae_host_side_rejections(cpu_device):
    n, K = 40, 6
    env = random_envs.RandomCartPoleVecEnv(n)
    critic = MLPPolicy.from_module(_net(1))
    traj = env.trajectory_buffer(K)
    env._tick = 10
    traj.tick0, traj.num_steps = 4, K                                    # as collect(K) at clock 4 leaves it
    with pytest.raises(ValueError, match="1-output"):
        env.gae(traj, MLPPolicy.from_module(_net(2)))
    with pytest.raises(ValueError, match="shape"):
        env.gae(random_envs.RandomCartPoleVecEnv(n + 1).trajectory_buffer(K), critic)
    with pytest.raises(ValueError, match="shape"):
        env.gae(object(), critic)
    slim = env.trajectory_buffer(K, final_obs=False)
    slim.tick0, slim.num_steps = 4, K
    with pytest.raises(ValueError, match="final_obs"):
        env.gae(slim, critic)
    with pytest.raises(ValueError, match="no collected steps"):
        env.gae(env.trajectory_buffer(K), critic)
    for g, lam in ((1.01, 0.95), (-0.1, 0.95), (0.99, 1.5), (0.99, -1e-3), (math.nan, 0.95), (0.99, math.inf)):
        with pytest.raises(ValueError, match=r"\[0, 1\]"):
            env.gae(traj, critic, g, lam)
    for tick in (11, 9, 0):                                              # a step / reset / collect since, or seed()
        env._tick = tick
        with pytest.raises(ValueError, match="moved"):
            env.gae(traj, critic)
    with pytest.raises(TypeError):
        env.gae(traj, "critic")
    for kw in (dict(dtype="float64"), dict(noisy=True)):
        other = random_envs.RandomCartPoleVecEnv(n, **kw)
        with pytest.raises(ValueError):
            other.gae(traj, critic)
    assert traj.values is None                                           # nothing ran
