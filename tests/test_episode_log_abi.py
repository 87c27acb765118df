"""Episode log without a GPU: the C struct layout seen from Python, argument validation of the four logged entry
points, the Python-side rejection of unsupported env variants, and the compiled form of the logged kernels."""
import ctypes
import os
import re
import sys

import pytest

from abi_support import ROOT, fake_env as _env, fake_log as _log, gcc_layout, ptxas_blocks
from random_envs_b200 import _lib, build as lib_build
import random_envs_b200 as random_envs

FIELDS = ["xi", "final_state", "length", "truncated", "end_tick", "count", "capacity"]


def test_episode_log_struct_offsets_in_python_match_the_header(tmp_path):
    got = gcc_layout(tmp_path, "renv_episode_log", FIELDS)
    want = {f: getattr(_lib.EpisodeLog, f).offset for f in FIELDS}
    want["sizeof"] = ctypes.sizeof(_lib.EpisodeLog)
    assert {k: int(v) for k, v in got.items()} == want


def _calls(env, log):
    """rc of each logged entry point for (env, log) with otherwise valid host arguments (nothing reaches CUDA when
    validation fails)."""
    lib = _lib.load()
    w = (ctypes.c_double * 4)(0, 0, 1, 0)
    lp = ctypes.byref(log) if log is not None else None
    return [lib.renv_cartpole_step_logged_f32(ctypes.byref(env), lp, 4096, 4096, 4096, None, 0, 500, 0, None, None, None),
            lib.renv_cartpole_step_logged_f64(ctypes.byref(env), lp, 4096, 4096, 4096, None, 0, 500, 0, None, None, None),
            lib.renv_cartpole_rollout_logged_f32(ctypes.byref(env), lp, w, 0.0, 5, 0, 500, 0, None, 4096, None, None),
            lib.renv_cartpole_rollout_logged_f64(ctypes.byref(env), lp, None, 0.0, 5, 0, 500, 0, None, 4096, None, None)]


def test_logged_entry_points_validate_the_log_before_any_cuda_call():
    env = _env()
    assert _calls(env, None) == [-1] * 4                        # NULL log
    for f in FIELDS[:-1]:                                       # any NULL field
        log = _log(); setattr(log, f, None)
        assert _calls(env, log) == [-1] * 4, f
    for cap in (0, -1, 1 << 31):
        log = _log(); log.capacity = cap
        assert _calls(env, log) == [-3] * 4, cap
    for f, bad in (("xi", 8200), ("final_state", 12296), ("length", 16386), ("end_tick", 24580), ("count", 28674)):
        log = _log(); setattr(log, f, bad)
        assert _calls(env, log) == [-2] * 4, f
    log = _log(); log.truncated = 20481                          # a byte array needs no alignment: passes validation
    env_bad = _env(); env_bad.n = 0                             # ... and the env's own checks still apply first
    assert _calls(env_bad, log) == [-3] * 4
    # the plain arguments keep their checks
    lib = _lib.load()
    assert lib.renv_cartpole_step_logged_f32(ctypes.byref(env), ctypes.byref(_log()), 4096, 4096, 4096, None, 7, 500, 0,
                                             None, None, None) == -6
    assert lib.renv_cartpole_rollout_logged_f32(ctypes.byref(env), ctypes.byref(_log()), None, 0.0, 0, 0, 500, 0, None,
                                                4096, None, None) == -3


@pytest.mark.parametrize("kw", [dict(lean=True), dict(noisy=True), dict(auto_reset=False)])
def test_start_episode_log_rejects_unsupported_envs_before_touching_cuda(kw):
    env = random_envs.RandomCartPoleVecEnv(64, **kw)
    with pytest.raises(ValueError, match="episode log"):
        env.start_episode_log(4)
    with pytest.raises(ValueError, match="episode log"):
        env.stop_episode_log()
    assert env._buffers is None


def test_logged_kernels_have_no_spills_and_keep_their_occupancy():
    logged = {name: b for name, b in ptxas_blocks().items() if "logged_kernel" in name}
    assert len(logged) == 10, sorted(logged)      # step f32/f64, pair x2, generic (fp64 x2 policies, fp32 random) x2
    for name, b in logged.items():
        for st, ld in re.findall(r"(\d+) bytes spill stores, (\d+) bytes spill loads", b):
            assert st == "0" and ld == "0", (name, st, ld)
        regs = int(re.search(r"Used (\d+) registers", b).group(1))
        if "cartpole_step_logged_kernelIf" in name:
            assert regs <= 64, (name, regs)           # 4 CTAs of 256 threads per SM, like the plain step
        if "rollout_pair" in name or re.search(r"rollout_logged_kernelIdLb[01]ELb0E", name):
            assert regs <= 80, (name, regs)           # 3 CTAs of 256 threads per SM, like the plain rollouts


def test_logged_pair_rollout_stays_on_the_packed_fp32_pipe():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    pair = [name for name in sass if "cartpole_rollout_pair_logged_kernelILb1" in name]
    assert len(pair) == 1, pair
    ops = [op for _, op, _ in sass[pair[0]]]
    assert sum(o.startswith("FFMA2") for o in ops) >= 100 and sum(o.startswith("FMUL2") for o in ops) >= 50
