"""MLP policy without a GPU: the C struct layout seen from Python, argument validation of the three MLP entry points,
rejection of unsupported networks, exactness of the 64-unit padding, and the compiled form of the new kernels."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch
from torch import nn

from abi_support import ROOT, fake_env as _env, fake_log, fake_policy as _policy, gcc_layout, ptxas_blocks
from random_envs_b200 import _lib, build as lib_build, mlp_policy


def test_mlp_policy_struct_offsets_in_python_match_the_header(tmp_path):
    got = gcc_layout(tmp_path, "renv_mlp_policy", ["params", "activation"],
                     [("floats", "%d", "RENV_MLP_PARAM_FLOATS"), ("hidden", "%d", "RENV_MLP_HIDDEN"),
                      ("tanh", "%d", "RENV_MLP_TANH"), ("relu", "%d", "RENV_MLP_RELU")])
    want = dict(params=_lib.MlpPolicy.params.offset, activation=_lib.MlpPolicy.activation.offset,
                sizeof=ctypes.sizeof(_lib.MlpPolicy), floats=mlp_policy.PARAM_FLOATS, hidden=mlp_policy.HIDDEN,
                tanh=mlp_policy.TANH, relu=mlp_policy.RELU)
    assert {k: int(v) for k, v in got.items()} == want
    assert mlp_policy.PARAM_FLOATS == 4612 and (64 * 4 + 64 + 64 * 64 + 64 + 2 * 64 + 2 + 3) // 4 * 4 == 4612


def _rcs(env, pol, K=5, integrator=0, dr=None, stats=4096):
    lib = _lib.load()
    log = fake_log()
    pp = ctypes.byref(pol) if pol is not None else None
    e = ctypes.byref(env)
    return [lib.renv_cartpole_rollout_mlp_f32(e, pp, K, integrator, 500, 0, dr, stats, None, None),
            lib.renv_cartpole_rollout_mlp_logged_f32(e, ctypes.byref(log), pp, K, integrator, 500, 0, dr, stats, None, None)]


def test_mlp_entry_points_validate_arguments_before_any_cuda_call():
    lib = _lib.load()
    env = _env()
    assert _rcs(env, None) == [-1, -1]                              # NULL policy
    assert _rcs(env, _policy(params=None)) == [-1, -1]              # NULL params
    assert _rcs(env, _policy(params=4100)) == [-2, -2]              # params not 16-byte aligned
    assert _rcs(env, _policy(act=2)) == [-7, -7]                    # unknown activation
    assert _rcs(env, _policy(act=-1)) == [-7, -7]
    for K in (0, -1, (1 << 30) + 1):                                # the linear rollout's K range
        assert _rcs(env, _policy(), K=K) == [-3, -3]
    assert _rcs(env, _policy(), integrator=5) == [-6, -6]
    assert _rcs(env, _policy(), stats=None) == [-1, -1]
    bad_dim = _lib.make_dr_cfg("uniform", [1.0] * 5, [2.0] * 5)
    assert _rcs(env, _policy(), dr=ctypes.byref(bad_dim)) == [-4, -4]
    bad_env = _env(); bad_env.n = 0
    assert _rcs(bad_env, _policy()) == [-3, -3]
    # policy_actions
    e = ctypes.byref(env)
    assert lib.renv_cartpole_policy_actions_mlp_f32(None, ctypes.byref(_policy()), 4096, None, None) == -1
    assert lib.renv_cartpole_policy_actions_mlp_f32(e, None, 4096, None, None) == -1
    assert lib.renv_cartpole_policy_actions_mlp_f32(e, ctypes.byref(_policy()), None, None, None) == -1
    assert lib.renv_cartpole_policy_actions_mlp_f32(e, ctypes.byref(_policy(params=4104)), 4096, None, None) == -2
    assert lib.renv_cartpole_policy_actions_mlp_f32(e, ctypes.byref(_policy(act=3)), 4096, None, None) == -7
    assert lib.renv_cartpole_policy_actions_mlp_f32(e, ctypes.byref(_policy()), 4097, None, None) == -2
    assert lib.renv_cartpole_policy_actions_mlp_f32(e, ctypes.byref(_policy()), 4096, 4100, None) == -2
    assert lib.renv_cartpole_policy_actions_mlp_f32(ctypes.byref(bad_env), ctypes.byref(_policy()), 4096, None, None) == -3


def _net(h1=64, h2=64, o=2, act=nn.Tanh, bias=True):
    return nn.Sequential(nn.Linear(4, h1, bias=bias), act(), nn.Linear(h1, h2), act(), nn.Linear(h2, o))


@pytest.mark.parametrize("net", [
    nn.Sequential(nn.Linear(4, 64), nn.Tanh(), nn.Linear(64, 2)),                                       # depth
    nn.Sequential(nn.Linear(4, 8), nn.Tanh(), nn.Linear(8, 8), nn.Tanh(), nn.Linear(8, 8), nn.Tanh(), nn.Linear(8, 2)),
    _net(h1=65), _net(h2=128),                                                                          # width
    _net(o=3),                                                                                          # outputs
    nn.Sequential(nn.Linear(5, 64), nn.Tanh(), nn.Linear(64, 64), nn.Tanh(), nn.Linear(64, 2)),         # input size
    nn.Sequential(nn.Linear(4, 64), nn.Sigmoid(), nn.Linear(64, 64), nn.Sigmoid(), nn.Linear(64, 2)),   # activation
    nn.Sequential(nn.Linear(4, 64), nn.Tanh(), nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 2)),         # mixed
    nn.Sequential(nn.Linear(4, 64), nn.Tanh(), nn.Linear(32, 64), nn.Tanh(), nn.Linear(64, 2)),         # no chain
    nn.Linear(4, 2),
])
def test_from_module_rejects_unsupported_networks(net):
    with pytest.raises(ValueError):
        mlp_policy.pack(net)


def _dyadic_(net, seed):
    """Weights k / 64 with small integers k: every float64 sum and product of a ReLU net on dyadic inputs is exact."""
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for p in net.parameters():
            p.copy_(torch.randint(-64, 65, p.shape, generator=g).float() / 64)
    return net


@pytest.mark.parametrize("h1,h2,o", [(64, 64, 2), (48, 32, 2), (48, 32, 1), (64, 17, 1)])
def test_padding_is_exact(h1, h2, o):
    torch.manual_seed(h1 + h2 + o)
    obs = torch.randint(-256, 257, (4096, 4)).double() / 128
    # ReLU with dyadic weights: the padded float64 evaluation equals the module's bit for bit
    net = _dyadic_(_net(h1, h2, o, nn.ReLU), h1 * h2 + o)
    params, act = mlp_policy.pack(net)
    assert act == mlp_policy.RELU and params.dtype == np.float32 and params.shape == (mlp_policy.PARAM_FLOATS,)
    got = mlp_policy.reference_logits(params, act, obs)
    want = net.double()(obs)
    if o == 1:
        assert torch.equal(got[:, 0], torch.zeros(len(obs), dtype=torch.float64))
        assert torch.equal(got[:, 1], want[:, 0])
    else:
        assert torch.equal(got, want)
    # Tanh, default init: the zero-padded units add exact zeros
    net = _net(h1, h2, o, nn.Tanh)
    params, act = mlp_policy.pack(net)
    got = mlp_policy.reference_logits(params, act, obs)
    want = net.double()(obs)
    torch.testing.assert_close(got[:, 2 - o:], want, rtol=0, atol=1e-15)
    assert act == mlp_policy.TANH


def test_pack_layout_matches_the_header():
    net = _net(48, 32, 2, nn.Tanh)
    params, _ = mlp_policy.pack(net)
    w1 = params[0:256].reshape(64, 4); b1 = params[256:320]
    w2 = params[320:4416].reshape(64, 64); b2 = params[4416:4480]
    w3 = params[4480:4608].reshape(2, 64); b3 = params[4608:4610]
    assert np.array_equal(w1[:48], net[0].weight.detach().numpy()) and not w1[48:].any() and not b1[48:].any()
    assert np.array_equal(w2[:32, :48], net[2].weight.detach().numpy()) and not w2[32:].any() and not w2[:, 48:].any()
    assert np.array_equal(b2[:32], net[2].bias.detach().numpy()) and not b2[32:].any()
    assert np.array_equal(w3[:, :32], net[4].weight.detach().numpy()) and not w3[:, 32:].any()
    assert np.array_equal(b3, net[4].bias.detach().numpy()) and not params[4610:].any()


def test_mlp_kernels_run_layer_2_on_the_tensor_cores_without_spills():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    rollout = [n for n in sass if "cartpole_rollout_mlp_kernel" in n]
    actions = [n for n in sass if "cartpole_policy_actions_mlp_kernel" in n]
    assert len(rollout) == 8 and len(actions) == 2, (rollout, actions)     # {tanh, relu} x {euler, semi} x {plain, logged}
    for name in rollout + actions:
        ops = [op for _, op, _ in sass[name]]
        # 2 row tiles x 8 N-tiles x 8 K-steps x 3 (head / tail split), emitted once: the row-tile loop is rolled
        assert sum(o.startswith("HMMA.1688.F32.TF32") for o in ops) == 192, name
        assert not any(o.startswith("MUFU.TANH") for o in ops), name        # the accurate tanh, not tanh.approx
    for name in actions:                                                     # no local memory at all
        assert not any(op.startswith(("LDL", "STL")) for _, op, _ in sass[name]), name
    blocks = ptxas_blocks()
    for name in rollout + actions:
        b = blocks[name]
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", b), name
        # the rollout's only stack frame is the full-range sincosf of its first step (an injected state may hold any
        # angle), which the plain rollouts carry as well
        frame = int(re.search(r"(\d+) bytes stack frame", b).group(1))
        assert frame <= (32 if name in rollout else 0), (name, frame)
