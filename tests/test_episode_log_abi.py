"""Episode log without a GPU: the C struct layout seen from Python, argument validation of the four logged entry
points, the Python-side rejection of unsupported env variants, and the compiled form of the logged kernels."""
import ctypes
import os
import re
import shutil
import subprocess
import sys

import pytest

from random_envs_b200 import _lib, build as lib_build
import random_envs_b200 as random_envs

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "renv.h")
FIELDS = ["xi", "final_state", "length", "truncated", "end_tick", "count", "capacity"]


def test_episode_log_struct_offsets_in_python_match_the_header(tmp_path):
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    src = tmp_path / "offsets.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "renv.h"\nint main(void) {\n' +
                   "".join('  printf("%s %%zu\\n", offsetof(renv_episode_log, %s));\n' % (f, f) for f in FIELDS) +
                   '  printf("sizeof %zu\\n", sizeof(renv_episode_log));\n  return 0;\n}\n')
    exe = tmp_path / "offsets"
    subprocess.run([gcc, "-I", os.path.dirname(HEADER), "-o", str(exe), str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())
    want = {f: getattr(_lib.EpisodeLog, f).offset for f in FIELDS}
    want["sizeof"] = ctypes.sizeof(_lib.EpisodeLog)
    assert {k: int(v) for k, v in got.items()} == want


def _env():
    env = _lib.CartpoleEnv()
    env.state = env.xi = env.elapsed = env.episode = 4096
    env.n, env.ld = 10, 12
    return env


def _log():
    log = _lib.EpisodeLog()
    log.xi, log.final_state, log.length, log.truncated, log.end_tick, log.count = 8192, 12288, 16384, 20480, 24576, 28672
    log.capacity = 2
    return log


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


def _ptxas_blocks():
    path = os.path.join(ROOT, "random_envs_b200", "librenv_b200.ptxas.log")
    if lib_build.is_stale() or not os.path.isfile(path):
        lib_build.build(force=True)
    blocks = {}
    for b in re.split(r"ptxas info\s+: Compiling entry function '", open(path).read())[1:]:
        blocks[b.split("'")[0]] = b
    return blocks


def test_logged_kernels_have_no_spills_and_keep_their_occupancy():
    logged = {name: b for name, b in _ptxas_blocks().items() if "logged_kernel" in name}
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
