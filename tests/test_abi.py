"""The C-ABI library loads on a CPU-only machine and exports exactly what include/renv.h declares."""
import ctypes
import os
import re

import pytest

from abi_support import fake_env, gcc_layout
from random_envs_b200 import _lib, build

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "renv.h")


def _declared():
    text = open(HEADER).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(renv_[a-z0-9_]+)\s*\(", text)))


def test_library_is_built_and_fresh():
    assert os.path.isfile(build.LIB_PATH), "run python -m random_envs_b200.build"
    assert not build.is_stale(), "librenv_b200.so is older than its sources"


def test_every_declared_symbol_is_exported_and_bound():
    names = _declared()
    assert len(names) >= 13
    lib = ctypes.CDLL(_lib.LIB_PATH)
    for n in names:
        assert hasattr(lib, n), "%s declared in renv.h but not exported" % n
    assert sorted(_lib.SIGNATURES) == names, "ctypes binding and header disagree"
    header_version = int(re.search(r"#define RENV_ABI_VERSION (\d+)", open(HEADER).read()).group(1))
    assert _lib.load().renv_abi_version() == _lib.ABI_VERSION == header_version == 6


def test_header_constants_match_binding():
    text = open(HEADER).read()
    assert int(re.search(r"#define RENV_MAX_DIM (\d+)", text).group(1)) == _lib.MAX_DIM
    assert int(re.search(r"#define RENV_NUM_STATS (\d+)", text).group(1)) == _lib.NUM_STATS
    assert int(re.search(r"#define RENV_TILE_ENVS_F32 (\d+)", text).group(1)) == _lib.TILE_ENVS["float32"]
    assert int(re.search(r"#define RENV_TILE_ENVS_F64 (\d+)", text).group(1)) == _lib.TILE_ENVS["float64"]
    assert ctypes.sizeof(_lib.DrCfg) == 8 + 3 * 8 * _lib.MAX_DIM + 8 * _lib.MAX_DIM ** 2
    assert ctypes.sizeof(_lib.CartpoleEnv) == 7 * 8 + 4 * 8


def test_strerror_and_argument_validation_without_a_gpu():
    """Negative status codes come from host-side validation, before any CUDA call."""
    lib = _lib.load()
    assert _lib.strerror(0) == "ok"
    assert "NULL" in _lib.strerror(-1) and "Unknown dr_type" in _lib.strerror(-5)
    cfg = _lib.make_dr_cfg("uniform", [0.0] * 4, [1.0] * 4)
    assert lib.renv_dr_sample_f32(None, 10, ctypes.byref(cfg), 0, 0, 0, None, None) == -1          # NULL out
    assert lib.renv_dr_sample_f32(ctypes.c_void_p(256), 0, ctypes.byref(cfg), 0, 0, 0, None, None) == -3   # n <= 0
    assert lib.renv_dr_sample_f32(ctypes.c_void_p(260), 8, ctypes.byref(cfg), 0, 0, 0, None, None) == -2   # misaligned
    cfg.dim = 33
    assert lib.renv_dr_sample_f32(ctypes.c_void_p(256), 8, ctypes.byref(cfg), 0, 0, 0, None, None) == -4
    cfg.dim, cfg.dr_type = 4, 9
    assert lib.renv_dr_sample_f32(ctypes.c_void_p(256), 8, ctypes.byref(cfg), 0, 0, 0, None, None) == -5
    assert lib.renv_cartpole_reset_f32(ctypes.byref(_lib.CartpoleEnv()), None, 0, None, None, None) == -1
    env = fake_env(ld=8)
    assert lib.renv_cartpole_reset_f32(ctypes.byref(env), None, 0, None, None, None) == -3             # ld < n
    env.ld = 10
    assert lib.renv_cartpole_reset_f32(ctypes.byref(env), None, 0, None, None, None) == -2             # ld % 4
    env.ld = 11
    assert lib.renv_cartpole_reset_f64(ctypes.byref(env), None, 0, None, None, None) == -2             # ld % 2 for f64
    env.ld = 12
    assert lib.renv_cartpole_step_f32(ctypes.byref(env), 4096, 4096, 4096, None, 7, 500, 1, 0, None, None, None) == -6
    assert lib.renv_cartpole_step_f32(ctypes.byref(env), 4096, 4096, 4096, None, 0, 500, 0, 0, None, None, None) == -1  # beyond
    w = (ctypes.c_double * 4)(0, 0, 1, 0)
    assert lib.renv_cartpole_rollout_f32(ctypes.byref(env), w, 0.0, 0, 0, 500, 0, None, 4096, None, None) == -3
    with pytest.raises(_lib.RenvError, match="alignment"):
        _lib.call("renv_random_actions_u8", ctypes.c_void_p(4101), 16, 0, 0, 0, None)


def test_unknown_dr_type_raises_reference_message():
    with pytest.raises(Exception, match="Unknown dr_type:beta"):
        _lib.make_dr_cfg("beta", [0.0], [1.0])


def test_noisy_and_rollout_argument_validation_without_a_gpu():
    lib = _lib.load()
    env = fake_env(beyond=4096)
    w = (ctypes.c_double * 4)(0, 0, 1, 0)
    noise = _lib.ObsNoise()
    assert lib.renv_cartpole_step_noisy_f32(ctypes.byref(env), None, 4096, 4096, 4096, None, 0, 500, 1, 0, None, None, None) == -1
    assert lib.renv_cartpole_reset_noisy_f64(ctypes.byref(env), ctypes.byref(noise), None, 0, None, None, None) == -1   # obs NULL
    noise.obs, noise.std = 4100, 0.1
    assert lib.renv_cartpole_reset_noisy_f32(ctypes.byref(env), ctypes.byref(noise), None, 0, None, None, None) == -2   # obs alignment
    noise.obs, noise.std = 4096, -1.0
    assert lib.renv_cartpole_step_noisy_f32(ctypes.byref(env), ctypes.byref(noise), 4096, 4096, 4096, None, 0, 500, 1, 0, None,
                                            None, None) == -7                                                           # std < 0
    noise.std = float("nan")
    assert lib.renv_cartpole_rollout_noisy_f32(ctypes.byref(env), ctypes.byref(noise), w, 0.0, 5, 0, 500, 0, None, 4096, None,
                                               None) == -7
    noise.std = 0.1
    assert lib.renv_cartpole_rollout_noisy_f64(ctypes.byref(env), ctypes.byref(noise), None, 0.0, 5, 0, 500, 0, None, 4096, None,
                                               None) == -7                      # the random policy ignores observations
    assert lib.renv_cartpole_rollout_f32(ctypes.byref(env), w, 0.0, (1 << 30) + 1, 0, 500, 0, None, 4096, None, None) == -3
    assert lib.renv_cartpole_rollout_f32(ctypes.byref(env), w, 0.0, 5, 0, 500, 0, None, None, None, None) == -1            # stats NULL
    assert lib.renv_cartpole_rollout_f32(ctypes.byref(env), w, 0.0, 5, 0, 500, 0, None, 4100, None, None) == -2            # stats alignment
    cfg = _lib.make_dr_cfg("uniform", [0.0] * 5, [1.0] * 5)
    assert lib.renv_cartpole_rollout_f32(ctypes.byref(env), w, 0.0, 5, 0, 500, 0, ctypes.byref(cfg), 4096, None, None) == -4   # dim != 4


def test_scalar_ctrl_offsets_in_python_match_the_header(tmp_path):
    """random_cartpole._ResidentScalarCore addresses struct renv_scalar_ctrl by byte offset (the block is shared with a
    running kernel through pinned host memory): the offsets must be the C compiler's."""
    fields = ["request", "arg", "arg_u64", "state", "obs", "xi", "reward", "done", "beyond", "violations", "ack",
              "exited", "next", "next_seq"]
    got = gcc_layout(tmp_path, "renv_scalar_ctrl", fields,
                     [("stride", "%zu", "sizeof(struct renv_scalar_outcome)"),
                      ("outcome_reward", "%zu", "offsetof(struct renv_scalar_outcome, reward)")])
    from random_envs_b200.random_cartpole import _ResidentScalarCore as C
    want = dict(request=C.OFF_REQUEST, arg=C.OFF_ARG, arg_u64=C.OFF_ARG_U64, state=C.OFF_STATE, obs=C.OFF_OBS, xi=C.OFF_XI,
                reward=C.OFF_REWARD, done=C.OFF_DONE, beyond=C.OFF_BEYOND, violations=C.OFF_VIOL, ack=C.OFF_ACK,
                exited=C.OFF_EXITED, next=C.OFF_NEXT, next_seq=C.OFF_NEXT_SEQ, sizeof=C.SIZE, stride=C.NEXT_STRIDE,
                outcome_reward=64)
    assert {k: int(v) for k, v in got.items()} == want
