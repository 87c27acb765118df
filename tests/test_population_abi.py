"""Population evaluation without a GPU: argument validation of the two population entry points, MLPPopulation packing,
and the compiled form of the population kernels."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch
from torch import nn

from abi_support import ROOT, fake_env, ptxas_blocks
from random_envs_b200 import _lib, build as lib_build, mlp_policy
from random_envs_b200.mlp_policy import MLPPolicy, MLPPopulation

NULL, ALIGN, SIZE, DIM, DRTYPE, INTEGRATOR, ARG = -1, -2, -3, -4, -5, -6, -7


def _linear(env=None, rows=4096, P=3, K=5, integrator=0, dr=None, stats=8192):
    e = ctypes.byref(env if env is not None else fake_env())
    return _lib.load().renv_cartpole_population_linear_f32(e, rows, P, K, integrator, 500, 0, dr, stats, None, None)


def _mlp(env=None, rows=4096, P=3, K=5, integrator=0, dr=None, stats=8192, activation=0):
    e = ctypes.byref(env if env is not None else fake_env())
    return _lib.load().renv_cartpole_population_mlp_f32(e, rows, activation, P, K, integrator, 500, 0, dr, stats, None,
                                                        None)


def _both(**kw):
    """(linear, MLP) return codes for the same arguments; every call here fails validation, so nothing is launched."""
    return [_linear(**kw), _mlp(**kw)]


def test_population_entry_points_validate_arguments_before_any_cuda_call():
    lib = _lib.load()
    assert lib.renv_cartpole_population_linear_f32(None, 4096, 3, 5, 0, 500, 0, None, 8192, None, None) == NULL
    assert lib.renv_cartpole_population_mlp_f32(None, 4096, 0, 3, 5, 0, 500, 0, None, 8192, None, None) == NULL
    assert _both(rows=None) == [NULL, NULL]
    assert _both(stats=None) == [NULL, NULL]
    assert _both(env=fake_env(xi=None)) == [NULL, NULL]                 # the task table is read without DR
    for P in (0, -1):
        assert _both(P=P) == [SIZE, SIZE]
    for n in (0, -4):
        assert _both(env=fake_env(n=n)) == [SIZE, SIZE]
    for K in (0, -1, (1 << 30) + 1):
        assert _both(K=K) == [SIZE, SIZE]
    assert _both(P=1 << 20, env=fake_env(n=1 << 11)) == [SIZE, SIZE]    # P n = 2^31
    assert _both(P=1, env=fake_env(n=1 << 31)) == [SIZE, SIZE]
    assert _both(P=2, env=fake_env(n=(1 << 30) + 1)) == [SIZE, SIZE]
    assert _both(stats=8196) == [ALIGN, ALIGN]
    assert _both(env=fake_env(xi=4104)) == [ALIGN, ALIGN]
    assert _both(rows=4098) == [ALIGN, ALIGN]                           # linear rows: 4-byte floats
    assert _mlp(rows=4100) == ALIGN                                     # MLP rows: 16 bytes
    assert _both(integrator=2) == [INTEGRATOR, INTEGRATOR]
    assert _mlp(activation=2) == ARG and _mlp(activation=-1) == ARG
    bad_dim = _lib.make_dr_cfg("uniform", [1.0] * 5, [2.0] * 5)
    assert _both(dr=ctypes.byref(bad_dim)) == [DIM, DIM]
    bad_type = _lib.make_dr_cfg("uniform", [1.0] * 4, [2.0] * 4)
    bad_type.dr_type = 9
    assert _both(dr=ctypes.byref(bad_type)) == [DRTYPE, DRTYPE]


def test_an_active_dr_config_does_not_read_the_task_table():
    # NULL xi is no error under DR: the next check, the misaligned policy rows, is what fails
    uniform = ctypes.byref(_lib.make_dr_cfg("uniform", [2.0, 0.5, 0.05, 0.1], [20.0, 3.0, 0.3, 1.0]))
    assert _both(env=fake_env(xi=None), dr=uniform, rows=4098) == [ALIGN, ALIGN]
    assert _both(env=fake_env(xi=4104), dr=uniform, rows=4098) == [ALIGN, ALIGN]
    assert _both(env=fake_env(xi=None), rows=4098) == [NULL, NULL]


def _net(act, h1=64, h2=64, o=2, seed=0):
    torch.manual_seed(seed)
    return nn.Sequential(nn.Linear(4, h1), act(), nn.Linear(h1, h2), act(), nn.Linear(h2, o))


def test_population_rows_equal_the_stacked_policy_params():
    nets = [_net(nn.Tanh, 64, 64, 2, 0), _net(nn.Tanh, 48, 32, 1, 1), _net(nn.Tanh, 17, 64, 2, 2)]
    policies = [MLPPolicy(*mlp_policy.pack(n), device="cpu") for n in nets]
    pop = MLPPopulation.from_policies(policies)
    assert len(pop) == 3 and pop.activation == mlp_policy.TANH
    assert pop.params.dtype == torch.float32 and tuple(pop.params.shape) == (3, mlp_policy.PARAM_FLOATS)
    assert torch.equal(pop.params, torch.stack([p.params for p in policies]))
    for p, policy in enumerate(policies):
        m = pop.member(p)
        assert m.activation == pop.activation and torch.equal(m.params, policy.params)
        assert m.params.data_ptr() == pop.params.data_ptr() + p * mlp_policy.PARAM_FLOATS * 4     # a view of row p
        assert m.params.data_ptr() % 16 == 0
    pop.params[1, 0] += 1.0                                              # in-place edits show through the view
    assert torch.equal(pop.member(1).params, pop.params[1])


def test_population_rejects_mixed_activations_and_bad_shapes():
    with pytest.raises(ValueError):
        MLPPopulation.from_modules([_net(nn.Tanh), _net(nn.ReLU)])
    with pytest.raises(ValueError):
        MLPPopulation.from_modules([])
    with pytest.raises(ValueError):
        MLPPopulation.from_policies([MLPPolicy(*mlp_policy.pack(_net(nn.Tanh)), device="cpu"),
                                     MLPPolicy(*mlp_policy.pack(_net(nn.ReLU)), device="cpu")])
    with pytest.raises(ValueError):
        MLPPopulation.from_policies([])
    with pytest.raises(ValueError):
        MLPPopulation(np.zeros((0, mlp_policy.PARAM_FLOATS), np.float32), mlp_policy.TANH, "cpu")
    with pytest.raises(ValueError):
        MLPPopulation(np.zeros((2, mlp_policy.PARAM_FLOATS - 4), np.float32), mlp_policy.TANH, "cpu")
    with pytest.raises(ValueError):
        MLPPopulation(np.zeros((2, mlp_policy.PARAM_FLOATS), np.float32), 2, "cpu")


def test_population_kernels_compile_as_the_rollouts_do():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    mlp = [n for n in sass if "cartpole_population_mlp_kernel" in n]
    linear = [n for n in sass if "cartpole_population_linear_kernel" in n]
    rollout = [n for n in sass if "cartpole_rollout_mlp_kernel" in n]
    assert len(mlp) == 4 and len(linear) == 2, (mlp, linear)        # {tanh, relu} x {euler, semi}; {euler, semi}
    hmma = lambda name: sum(op.startswith("HMMA.1688.F32.TF32") for _, op, _ in sass[name])
    assert {hmma(n) for n in rollout} == {192}
    for name in mlp:
        assert hmma(name) == 192, name
    blocks = ptxas_blocks()
    frame = lambda name: int(re.search(r"(\d+) bytes stack frame", blocks[name]).group(1))
    rollout_frame = max(frame(n) for n in rollout)
    for name in mlp + linear:
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", blocks[name]), name
        assert frame(name) <= rollout_frame, (name, frame(name), rollout_frame)
