"""The uint16 TimeLimit counter without a GPU: which entry points take an env whose `elapsed` is NULL, the 65535 bound
they check before any CUDA call, and the compiled form of the step the default env takes."""
import ctypes
import os
import sys

from random_envs_b200 import _lib, build as lib_build

from abi_support import ROOT, fake_env, fake_log, fake_policy, fake_traj

E_NULL, E_SIZE = -1, -3
W = (ctypes.c_double * 4)(0.0, 0.0, 1.0, 0.0)


def _calls(env, max_steps):
    """Every fp32 entry point that takes either counter, with arguments that pass all other checks."""
    lib = _lib.load()
    e, log, p, t = ctypes.byref(env), ctypes.byref(fake_log()), ctypes.byref(fake_policy()), ctypes.byref(fake_traj())
    return [lib.renv_cartpole_rollout_f32(e, W, 0.0, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_rollout_f32(e, None, 0.0, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_rollout_logged_f32(e, log, W, 0.0, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_rollout_mlp_f32(e, p, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_rollout_mlp_logged_f32(e, log, p, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_collect_mlp_f32(e, p, t, 1, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_collect_mlp_logged_f32(e, log, p, t, 1, 5, 0, max_steps, 0, None, 4096, None, None),
            lib.renv_cartpole_step_logged_f32(e, log, 4096, None, 4096, None, 0, max_steps, 0, None, None, None)]


def test_a_uint16_counter_alone_is_bounded_by_65535():
    assert _calls(fake_env(elapsed=None, elapsed16=8192), 65536) == [E_SIZE] * 8
    assert _calls(fake_env(elapsed=None, elapsed16=8192), 70000) == [E_SIZE] * 8


def test_an_env_needs_one_of_the_two_counters():
    assert _calls(fake_env(elapsed=None), 500) == [E_NULL] * 8
    lib = _lib.load()
    # fp64 has no uint16 counter: its rollout and logged step still need `elapsed`
    e = ctypes.byref(fake_env(elapsed=None, elapsed16=8192))
    assert lib.renv_cartpole_rollout_f64(e, W, 0.0, 5, 0, 500, 0, None, 4096, None, None) == E_NULL
    assert lib.renv_cartpole_step_logged_f64(e, ctypes.byref(fake_log()), 4096, None, 4096, None, 0, 500, 0, None, None,
                                             None) == E_NULL


def test_the_default_fp32_step_moves_its_counter_in_64_bit_accesses():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    lean = [n for n in sass if "cartpole_step_kernelIfLb1ELb0ELb1" in n]
    plain = [n for n in sass if "cartpole_step_kernelIfLb1ELb0ELb0" in n]
    assert len(lean) == 1 and len(plain) == 1, (lean, plain)
    ops = [op for _, op, _ in sass[lean[0]]]
    ops32 = [op for _, op, _ in sass[plain[0]]]
    # four uint16 counters per thread: one 64-bit load and one 64-bit store, where the int32 step moves 128 bits
    assert sum(o.startswith("LDG.E.64") for o in ops) >= 1 and sum(o.startswith("STG.E.64") for o in ops) >= 1
    assert sum(o.startswith("LDG.E.128") for o in ops) < sum(o.startswith("LDG.E.128") for o in ops32)
