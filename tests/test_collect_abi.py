"""Trajectory collection without a GPU: the renv_trajectory layout seen from Python, argument validation of the
collect and policy_logp entry points, the compiled form of the new kernels, and the Trajectory views."""
import ctypes
import os
import re
import sys

import pytest
import torch

from abi_support import ROOT, fake_env as _env, fake_log, fake_policy as _policy, fake_traj as _traj, gcc_layout, \
    ptxas_blocks
from random_envs_b200 import Trajectory, _lib, build as lib_build

FIELDS = ["obs", "action", "done", "logp", "truncated", "final_obs", "capacity"]


def test_trajectory_struct_offsets_in_python_match_the_header(tmp_path):
    got = gcc_layout(tmp_path, "renv_trajectory", FIELDS)
    want = {f: getattr(_lib.Trajectory, f).offset for f in FIELDS}
    want["sizeof"] = ctypes.sizeof(_lib.Trajectory)
    assert {k: int(v) for k, v in got.items()} == want


def _rcs(env=None, pol="ok", traj="ok", sample=1, K=5, integrator=0, dr=None, stats=4096):
    """Status of the plain and the logged collect entry point for the same arguments."""
    lib = _lib.load()
    log = fake_log()
    env = _env() if env is None else env
    pol = _policy() if pol == "ok" else pol
    traj = _traj() if traj == "ok" else traj
    pp = ctypes.byref(pol) if pol is not None else None
    tp = ctypes.byref(traj) if traj is not None else None
    e = ctypes.byref(env)
    return [lib.renv_cartpole_collect_mlp_f32(e, pp, tp, sample, K, integrator, 500, 0, dr, stats, None, None),
            lib.renv_cartpole_collect_mlp_logged_f32(e, ctypes.byref(log), pp, tp, sample, K, integrator, 500, 0, dr,
                                                     stats, None, None)]


def test_collect_validates_arguments_before_any_cuda_call():
    lib = _lib.load()
    null_env = _lib.CartpoleEnv()
    assert lib.renv_cartpole_collect_mlp_f32(None, ctypes.byref(_policy()), ctypes.byref(_traj()), 1, 5, 0, 500, 0, None,
                                             4096, None, None) == -1
    assert _rcs(env=null_env) == [-1, -1]                               # NULL state / xi / elapsed
    assert _rcs(pol=None) == [-1, -1]
    assert _rcs(pol=_policy(params=None)) == [-1, -1]
    assert _rcs(traj=None) == [-1, -1]
    for f in ("obs", "action", "done"):
        assert _rcs(traj=_traj(**{f: None})) == [-1, -1], f
    for f in ("logp", "truncated", "final_obs"):                          # optional
        assert _rcs(traj=_traj(**{f: None}), K=9) == [-7, -7], f        # (K > capacity: past the NULL checks)
    for f, v in (("obs", 4104), ("final_obs", 4104), ("logp", 4098), ("action", 4097), ("done", 4098), ("truncated", 4099)):
        assert _rcs(traj=_traj(**{f: v})) == [-2, -2], f
    assert _rcs(pol=_policy(params=4100)) == [-2, -2]
    for K in (0, -1, (1 << 30) + 1):                                      # the rollout's K range and code
        assert _rcs(K=K) == [-3, -3], K
    assert _rcs(K=9) == [-7, -7]                                          # K > capacity
    assert _rcs(traj=_traj(capacity=0), K=1) == [-7, -7]
    assert _rcs(pol=_policy(act=2)) == [-7, -7]                           # unknown activation
    for sample in (-1, 2):
        assert _rcs(sample=sample) == [-7, -7], sample
    assert _rcs(integrator=5) == [-6, -6]
    assert _rcs(stats=None) == [-1, -1]
    bad_dim = _lib.make_dr_cfg("uniform", [1.0] * 5, [2.0] * 5)
    assert _rcs(dr=ctypes.byref(bad_dim)) == [-4, -4]
    bad_env = _env(); bad_env.n = 0
    assert _rcs(env=bad_env) == [-3, -3]


def test_policy_logp_validates_arguments_before_any_cuda_call():
    lib = _lib.load()
    e, p = ctypes.byref(_env()), ctypes.byref(_policy())
    f = lib.renv_cartpole_policy_logp_mlp_f32
    assert f(None, p, 1, 0, 4096, None, None, None) == -1
    assert f(e, None, 1, 0, 4096, None, None, None) == -1
    assert f(e, ctypes.byref(_policy(params=None)), 1, 0, 4096, None, None, None) == -1
    assert f(e, p, 1, 0, None, 4096, None, None) == -1                   # NULL action
    assert f(e, ctypes.byref(_policy(params=4104)), 1, 0, 4096, None, None, None) == -2
    assert f(e, p, 1, 0, 4097, None, None, None) == -2                   # action
    assert f(e, p, 1, 0, 4096, 4098, None, None) == -2                   # logp
    assert f(e, p, 1, 0, 4096, None, 4100, None) == -2                   # logits
    assert f(e, ctypes.byref(_policy(act=3)), 1, 0, 4096, None, None, None) == -7
    for sample in (-1, 2, 255):
        assert f(e, p, sample, 0, 4096, 4096, None, None) == -7
    bad_env = _env(); bad_env.n = 0
    assert f(ctypes.byref(bad_env), p, 0, 0, 4096, None, None, None) == -3


def test_collect_and_policy_logp_kernels_keep_the_mlp_budgets():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    collect = [n for n in sass if "cartpole_collect_mlp_kernel" in n]
    logp = [n for n in sass if "cartpole_policy_logp_mlp_kernel" in n]
    assert len(collect) == 8 and len(logp) == 2, (collect, logp)     # {tanh, relu} x {euler, semi} x {plain, logged}
    for name in collect + logp:
        ops = [op for _, op, _ in sass[name]]
        assert sum(o.startswith("HMMA.1688.F32.TF32") for o in ops) == 192, name     # mlp_logits, emitted once
        assert not any(o.startswith("MUFU.TANH") for o in ops), name
    for name in logp:                                                    # no local memory at all
        assert not any(op.startswith(("LDL", "STL")) for _, op, _ in sass[name]), name
    blocks = ptxas_blocks()
    for name in collect + logp:
        b = blocks[name]
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", b), name
        frame = int(re.search(r"(\d+) bytes stack frame", b).group(1))
        assert frame <= (32 if name in collect else 0), (name, frame)   # the rollout's first-step sincosf frame
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        assert regs <= 168, (name, regs)                                 # 3 CTAs of 128 threads per SM


def test_trajectory_fields_are_views_of_the_capacity_storage():
    n, ld, cap = 5, 32, 4
    tr = Trajectory(n, ld, cap, "cpu")
    assert tr.num_steps == 0 and tr.tick0 is None and tr.obs.shape == (0, n, 4)
    tr.num_steps, tr.tick0 = 3, 17
    assert tr.obs.shape == (3, n, 4) and tr.obs.dtype == torch.float32
    assert tr.final_obs.shape == (3, n, 4)
    for f in ("actions", "logp", "dones", "truncated", "rewards"):
        assert getattr(tr, f).shape == (3, n), f
    assert tr.actions.dtype == torch.uint8 and tr.logp.dtype == torch.float32
    assert tr.dones.dtype == torch.bool and tr.truncated.dtype == torch.bool
    assert tr.rewards.dtype == torch.float32 and bool((tr.rewards == 1).all()) and tr.rewards.stride() == (0, 0)
    # views over [:num_steps, :N] of (capacity, ld, ...) storage: row k of env i is element k * ld + i
    tr._obs.view(-1, 4)[:, 0] = torch.arange(cap * ld, dtype=torch.float32)
    tr._done.view(-1)[:] = (torch.arange(cap * ld) % 3 == 0).to(torch.uint8)
    k, i = 2, 4
    assert float(tr.obs[k, i, 0]) == k * ld + i
    assert bool(tr.dones[k, i]) == ((k * ld + i) % 3 == 0)
    assert tr.obs.data_ptr() == tr._obs.data_ptr() and tr.obs.stride() == (ld * 4, 4, 1)
    s = tr.struct
    assert (s.obs, s.action, s.done, s.logp, s.truncated, s.final_obs, s.capacity) == (
        tr._obs.data_ptr(), tr._action.data_ptr(), tr._done.data_ptr(), tr._logp.data_ptr(), tr._truncated.data_ptr(),
        tr._final_obs.data_ptr(), cap)
    lean = Trajectory(n, ld, cap, "cpu", logp=False, final_obs=False)
    lean.num_steps = 2
    assert lean.logp is None and lean.final_obs is None and lean.struct.logp is None and lean.struct.final_obs is None
    with pytest.raises(ValueError):
        Trajectory(n, ld, 0, "cpu")
