"""Evaluation grids without a GPU: argument validation of the two grid entry points, the scenario packer for a fixed
task and each of the four laws, the Python Scenarios rows, and the compiled form of the grid kernels."""
import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest
import torch

from abi_support import ROOT, fake_env, ptxas_blocks
from random_envs_b200 import Scenarios, TaskSampler, _lib, build as lib_build
from random_envs_b200.random_env import covariance_factor

NULL, ALIGN, SIZE, DIM, DRTYPE, INTEGRATOR, ARG = -1, -2, -3, -4, -5, -6, -7
F = _lib.SCENARIO_FLOATS


def _linear(env=None, rows=4096, P=3, scen=8192, C=5, K=5, integrator=0, stats=16384):
    e = ctypes.byref(env if env is not None else fake_env())
    return _lib.load().renv_cartpole_grid_linear_f32(e, rows, P, scen, C, K, integrator, 500, 0, stats, None, None)


def _mlp(env=None, rows=4096, P=3, scen=8192, C=5, K=5, integrator=0, stats=16384, activation=0):
    e = ctypes.byref(env if env is not None else fake_env())
    return _lib.load().renv_cartpole_grid_mlp_f32(e, rows, activation, P, scen, C, K, integrator, 500, 0, stats, None,
                                                  None)


def _both(**kw):
    """(linear, MLP) return codes for the same arguments; every call here fails validation, so nothing is launched."""
    return [_linear(**kw), _mlp(**kw)]


def test_grid_entry_points_validate_arguments_before_any_cuda_call():
    lib = _lib.load()
    assert lib.renv_cartpole_grid_linear_f32(None, 4096, 3, 8192, 5, 5, 0, 500, 0, 16384, None, None) == NULL
    assert lib.renv_cartpole_grid_mlp_f32(None, 4096, 0, 3, 8192, 5, 5, 0, 500, 0, 16384, None, None) == NULL
    assert _both(rows=None) == [NULL, NULL]
    assert _both(scen=None) == [NULL, NULL]
    assert _both(stats=None) == [NULL, NULL]
    for P in (0, -1):
        assert _both(P=P) == [SIZE, SIZE]
    for C in (0, -1):
        assert _both(C=C) == [SIZE, SIZE]
    for n in (0, -4):
        assert _both(env=fake_env(n=n)) == [SIZE, SIZE]
    for K in (0, -1, (1 << 30) + 1):
        assert _both(K=K) == [SIZE, SIZE]
    assert _both(P=1 << 10, C=1 << 10, env=fake_env(n=1 << 11)) == [SIZE, SIZE]    # P C n = 2^31
    assert _both(P=1 << 10, C=(1 << 10) - 1, env=fake_env(n=(1 << 11) + 3)) == [SIZE, SIZE]
    assert _both(P=(1 << 31) - 1, C=(1 << 31) - 1, env=fake_env(n=(1 << 31) - 1)) == [SIZE, SIZE]   # no overflow
    assert _both(P=1 << 16, C=1 << 15, env=fake_env(n=1)) == [SIZE, SIZE]
    assert _both(P=1, C=1, env=fake_env(n=1 << 31)) == [SIZE, SIZE]
    assert _both(stats=16388) == [ALIGN, ALIGN]
    assert _both(scen=8200) == [ALIGN, ALIGN]                           # scenario rows: 16 bytes
    assert _both(rows=4098) == [ALIGN, ALIGN]                           # linear rows: 4-byte floats
    assert _mlp(rows=4100) == ALIGN and _linear(rows=4100) != ALIGN     # MLP rows: 16 bytes
    assert _both(integrator=2) == [INTEGRATOR, INTEGRATOR]
    assert _mlp(activation=2) == ARG and _mlp(activation=-1) == ARG


def test_the_grid_does_not_read_the_task_table():
    # NULL or misaligned xi is no error: the next check, the misaligned scenario rows, is what fails
    assert _both(env=fake_env(xi=None), scen=8200) == [ALIGN, ALIGN]
    assert _both(env=fake_env(xi=4104), scen=8200) == [ALIGN, ALIGN]
    assert _both(env=fake_env(xi=None, state=None, elapsed=None), scen=8200) == [ALIGN, ALIGN]


def _pack(cfg, task):
    out = np.full(F, np.nan, dtype=np.float32)          # every slot must be written
    arg = (ctypes.c_double * 4)(*task) if task is not None else None
    rc = _lib.load().renv_scenario_pack_f32(ctypes.byref(cfg) if cfg is not None else None, arg,
                                            ctypes.c_void_p(out.ctypes.data))
    return rc, out


def _ints(row):
    return row[:2].view(np.int32).tolist()


def test_packer_fixed_task_row():
    task = [9.81, 1.1, 0.123456789, 0.7]
    for cfg in (None, _lib.make_dr_cfg(None, None, None)):
        rc, row = _pack(cfg, task)
        assert rc == 0
        assert _ints(row) == [_lib.DR_NONE, 4]
        assert np.array_equal(row[2:6], np.array(task, dtype=np.float32))
        assert not row[6:].any()


def test_packer_uniform_row():
    lo, hi = [2.0, 0.5, 0.05, 0.1], [20.0, 3.0, 0.3, 1.0 / 3.0]
    rc, row = _pack(_lib.make_dr_cfg("uniform", lo, hi), None)
    assert rc == 0 and _ints(row) == [_lib.DR_UNIFORM, 4]
    lo32, hi32 = np.array(lo, np.float32), np.array(hi, np.float32)
    assert np.array_equal(row[2:6], lo32)
    assert np.array_equal(row[6:10], (hi32 - lo32) * np.float32(2.0 ** -24))
    assert not row[10:].any()


def test_packer_truncnorm_and_gaussian_rows_carry_their_floors():
    mean, std, lb = [9.8, 1.0, 0.1, 0.5], [1.0, 0.2, 0.03, 0.1], [0.5, 0.05, 0.01, 0.02]
    rc, row = _pack(_lib.make_dr_cfg("truncnorm", mean, std, lb), None)
    assert rc == 0 and _ints(row) == [_lib.DR_TRUNCNORM, 4]
    assert np.array_equal(row[2:6], np.array(mean, np.float32))
    assert np.array_equal(row[6:10], np.array(std, np.float32))
    assert np.array_equal(row[10:14], np.array(lb, np.float32))
    assert not row[14:].any()
    rc, row = _pack(_lib.make_dr_cfg("gaussian", mean, std), None)
    assert rc == 0 and _ints(row) == [_lib.DR_GAUSSIAN, 4]
    assert np.array_equal(row[10:14], np.full(4, 0.1, np.float32))


def test_packer_fullgaussian_row_carries_its_factor():
    mean = [2.0, 1.5, 2.5, 2.0]
    cov = np.array([[0.30, 0.05, 0.00, 0.02], [0.05, 0.20, 0.03, 0.00],
                    [0.00, 0.03, 0.25, 0.04], [0.02, 0.00, 0.04, 0.30]])
    lo, hi = [2.0, 0.5, 0.05, 0.1], [20.0, 3.0, 0.3, 1.0]
    factor = covariance_factor(cov)
    rc, row = _pack(_lib.make_dr_cfg("fullgaussian", mean, lo, hi, factor), None)
    assert rc == 0 and _ints(row) == [_lib.DR_FULLGAUSSIAN, 4]
    assert np.array_equal(row[2:6], np.array(mean, np.float32))
    assert np.array_equal(row[6:10], np.array(lo, np.float32))
    assert np.array_equal(row[10:14], np.array(hi, np.float32))
    assert np.array_equal(row[14:30], factor.astype(np.float32).ravel())
    assert not row[30:].any()


def test_packer_errors():
    lib = _lib.load()
    task = (ctypes.c_double * 4)(9.8, 1.0, 0.1, 0.5)
    assert lib.renv_scenario_pack_f32(None, task, None) == NULL
    assert _pack(None, None)[0] == NULL
    assert _pack(_lib.make_dr_cfg(None, None, None), None)[0] == NULL
    for bad in (math.nan, math.inf, -math.inf):
        assert _pack(None, [9.8, 1.0, bad, 0.5])[0] == ARG
    assert _pack(_lib.make_dr_cfg("uniform", [1.0] * 5, [2.0] * 5), None)[0] == DIM
    for t in (9, -1):
        cfg = _lib.make_dr_cfg("uniform", [1.0] * 4, [2.0] * 4)
        cfg.dr_type = t
        assert _pack(cfg, None)[0] == DRTYPE
    # a distribution row ignores the task
    cfg = _lib.make_dr_cfg("uniform", [1.0] * 4, [2.0] * 4)
    assert np.array_equal(_pack(cfg, None)[1], _pack(cfg, [math.nan] * 4)[1])


def test_scenarios_rows_equal_the_packers():
    tasks = np.array([[9.8, 1.0, 0.1, 0.5], [2.0, 3.0, 0.3, 1.0], [15.5, 0.75, 0.2, 0.25]])
    s = Scenarios.tasks(tasks, device="cpu")
    assert len(s) == 3 and s.rows.dtype == torch.float32 and tuple(s.rows.shape) == (3, F) and s.device.type == "cpu"
    for c in range(3):
        assert np.array_equal(s.rows[c].numpy(), _pack(None, tasks[c].tolist())[1])
    assert torch.equal(Scenarios.tasks(torch.tensor(tasks), device="cpu").rows, s.rows)
    distrs = {
        "uniform": [[2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0], [9.8, 9.8, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]],
        "truncnorm": [[9.8, 1.0, 1.0, 0.2, 0.1, 0.03, 0.5, 0.1]],
        "gaussian": [[9.8, 1.0, 1.0, 0.2, 0.3, 0.03, 0.5, 0.1]],
        "fullgaussian": [{"mean": [2.0, 1.5, 2.5, 2.0], "cov": np.eye(4) * 0.2}],
    }
    parts = []
    for dr_type, ds in distrs.items():
        part = Scenarios.distributions(dr_type, ds, device="cpu")
        for c, d in enumerate(ds):
            twin = TaskSampler("RandomCartPole-v0")
            twin.set_dr_distribution(dr_type, d)
            assert np.array_equal(part.rows[c].numpy(), _pack(twin.dr_config(), None)[1]), (dr_type, c)
        parts.append(part)
    everything = Scenarios.cat(s, *parts)
    assert len(everything) == 3 + 5
    assert torch.equal(everything.rows, torch.cat([s.rows] + [p.rows for p in parts]))
    # an ADR boundary: lo = hi on one dim pins it (width 0)
    row = Scenarios.distributions("uniform", [distrs["uniform"][1]], device="cpu").rows[0].numpy()
    assert row[2] == np.float32(9.8) and row[6] == 0.0


def test_scenarios_reject_bad_input():
    with pytest.raises(ValueError):
        Scenarios.tasks(np.zeros((0, 4)), device="cpu")
    with pytest.raises(ValueError):
        Scenarios.tasks(np.zeros((2, 3)), device="cpu")
    with pytest.raises(ValueError):
        Scenarios.tasks([[9.8, 1.0, math.nan, 0.5]], device="cpu")
    with pytest.raises(ValueError):
        Scenarios.distributions("uniform", [], device="cpu")
    with pytest.raises(Exception, match="Unknown dr_type"):
        Scenarios.distributions("beta", [[1.0] * 8], device="cpu")
    with pytest.raises(TypeError):
        Scenarios.cat()
    with pytest.raises(ValueError):
        Scenarios(torch.zeros((2, F - 1)))


def test_grid_kernels_compile_as_the_population_kernels_do():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    mlp = [n for n in sass if "cartpole_grid_mlp_kernel" in n]
    linear = [n for n in sass if "cartpole_grid_linear_kernel" in n]
    population = [n for n in sass if "cartpole_population_" in n]
    assert len(mlp) == 4 and len(linear) == 2 and len(population) == 6, (mlp, linear, population)
    for name in mlp:
        ops = [op for _, op, _ in sass[name]]
        assert sum(op.startswith("HMMA.1688.F32.TF32") for op in ops) == 192, name
        assert not any(op.startswith("MUFU.TANH") for op in ops), name
    blocks = ptxas_blocks()
    frame = lambda name: int(re.search(r"(\d+) bytes stack frame", blocks[name]).group(1))
    regs = lambda name: int(re.search(r"Used (\d+) registers", blocks[name]).group(1))
    population_frame = max(frame(n) for n in population)
    assert population_frame == 16
    for name in mlp + linear:
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", blocks[name]), name
        assert frame(name) <= population_frame, (name, frame(name), population_frame)
    # the population kernels' launch bounds: 256 threads x 3 CTAs (linear), 128 x 3 (MLP) per SM
    for name in linear:
        assert regs(name) <= 65536 // (256 * 3), (name, regs(name))
    for name in mlp:
        assert regs(name) <= 65536 // (128 * 3), (name, regs(name))
