"""Helpers of the no-GPU ABI tests: fake argument structs, struct layouts as gcc sees include/renv.h, and the per-kernel
blocks of the build's ptxas log.

The fake structs hold small aligned integers in place of device pointers.  The tests pass them only to calls that fail
validation, so no pointer is ever dereferenced and nothing reaches CUDA."""
import os
import re
import shutil
import subprocess

import pytest

from random_envs_b200 import _lib, build as lib_build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "renv.h")
PTXAS_LOG = os.path.join(ROOT, "random_envs_b200", "librenv_b200.ptxas.log")


def _fill(s, kw):
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def fake_env(**kw):
    """10 envs, ld 12, with state, xi, elapsed and episode set."""
    env = _lib.CartpoleEnv()
    env.state = env.xi = env.elapsed = env.episode = 4096
    env.n, env.ld = 10, 12
    return _fill(env, kw)


def fake_log(**kw):
    log = _lib.EpisodeLog()
    log.xi, log.final_state, log.length, log.truncated, log.end_tick, log.count = 8192, 12288, 16384, 20480, 24576, 28672
    log.capacity = 2
    return _fill(log, kw)


def fake_policy(params=4096, act=0):
    p = _lib.MlpPolicy()
    p.params, p.activation = params, act
    return p


def fake_traj(**kw):
    t = _lib.Trajectory()
    t.obs, t.action, t.done, t.logp, t.truncated, t.final_obs, t.capacity = 4096, 8192, 8448, 8704, 8960, 12288, 8
    return _fill(t, kw)


def gcc_layout(tmp_path, struct, fields, extra=()):
    """{name: printed value} from a C program compiled with gcc against include/renv.h: offsetof(struct, f) for each
    field, "sizeof", and one entry per (name, printf format, C expression) in ``extra``.  Skips the test without gcc."""
    gcc = shutil.which("gcc")
    if gcc is None:
        pytest.skip("no gcc")
    lines = [("%s %%zu" % f, "offsetof(%s, %s)" % (struct, f)) for f in fields] + [("sizeof %zu", "sizeof(%s)" % struct)]
    lines += [("%s %s" % (name, fmt), expr) for name, fmt, expr in extra]
    src = tmp_path / "offsets.c"
    src.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "renv.h"\nint main(void) {\n' +
                   "".join('  printf("%s\\n", %s);\n' % line for line in lines) + "  return 0;\n}\n")
    exe = tmp_path / "offsets"
    subprocess.run([gcc, "-I", os.path.dirname(HEADER), "-o", str(exe), str(src)], check=True)
    return dict(line.split() for line in subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.splitlines())


def ptxas_blocks():
    """{kernel: its block of the ptxas -v log} of the current build (the log is written by the build, not tracked)."""
    lib_build.build(force=not os.path.isfile(PTXAS_LOG))
    return {b.split("'")[0]: b for b in re.split(r"ptxas info\s+: Compiling entry function '", open(PTXAS_LOG).read())[1:]}
