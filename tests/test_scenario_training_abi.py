"""Per-env task scenarios without a GPU: argument validation of the five scenario entry points, the Python checks of
set_scenarios, the ADR boundary rows, and the compiled form of the scenario kernels."""
import ctypes
import os
import re
import sys

import numpy as np
import pytest
import torch

from abi_support import ROOT, fake_env, fake_log, fake_policy, fake_traj, gcc_layout, ptxas_blocks
from random_envs_b200 import RandomCartPoleVecEnv, Scenarios, _lib, build as lib_build

NULL, ALIGN, SIZE, DIM, DRTYPE, INTEGRATOR, ARG = -1, -2, -3, -4, -5, -6, -7
ENTRIES = ("reset", "step", "rollout", "rollout_mlp", "collect_mlp")


def fake_scen(**kw):
    s = _lib.EnvScenarios()
    s.rows, s.of_env, s.C = 32768, 36864, 5
    for k, v in kw.items():
        setattr(s, k, v)
    return s


def _call(entry, env=None, scen="default", log=None, **kw):
    """Return code of the scenario entry point ``entry`` on fake arguments that fail validation somewhere."""
    lib = _lib.load()
    e = ctypes.byref(env if env is not None else fake_env())
    s = ctypes.byref(fake_scen()) if isinstance(scen, str) else (ctypes.byref(scen) if scen is not None else None)
    lg = ctypes.byref(log) if log is not None else None
    K, integ, max_steps = kw.get("K", 5), kw.get("integrator", 0), kw.get("max_steps", 500)
    stats, viol = kw.get("stats", 16384), None
    if entry == "reset":
        return lib.renv_cartpole_reset_scen_f32(e, s, kw.get("mask"), 0, viol, None)
    if entry == "step":
        return lib.renv_cartpole_step_scen_f32(e, s, lg, kw.get("action", 40960), kw.get("reward", 45056),
                                               kw.get("done", 49152), kw.get("truncated", 53248), integ, max_steps, 0,
                                               kw.get("counters"), None)
    if entry == "rollout":
        w = (ctypes.c_double * 4)(0.0, 0.0, 1.0, 0.0) if kw.get("w", True) else None
        return lib.renv_cartpole_rollout_scen_f32(e, s, lg, w, 0.0, K, integ, max_steps, 0, stats, viol, None)
    p = ctypes.byref(kw.get("policy", fake_policy()))
    if entry == "rollout_mlp":
        return lib.renv_cartpole_rollout_mlp_scen_f32(e, s, lg, p, K, integ, max_steps, 0, stats, viol, None)
    t = ctypes.byref(kw.get("traj", fake_traj()))
    return lib.renv_cartpole_collect_mlp_scen_f32(e, s, lg, p, t, kw.get("sample", 1), K, integ, max_steps, 0, stats,
                                                  viol, None)


def test_env_scenarios_struct_offsets_in_python_match_the_header(tmp_path):
    fields = [f for f, _ in _lib.EnvScenarios._fields_]
    got = gcc_layout(tmp_path, "renv_env_scenarios", fields)
    for f in fields:
        assert int(got[f]) == getattr(_lib.EnvScenarios, f).offset, f
    assert int(got["sizeof"]) == ctypes.sizeof(_lib.EnvScenarios)


@pytest.mark.parametrize("entry", ENTRIES)
def test_scenario_errors_before_any_cuda_call(entry):
    assert _call(entry, scen=None) == NULL
    assert _call(entry, scen=fake_scen(rows=None)) == NULL
    assert _call(entry, scen=fake_scen(of_env=None)) == NULL
    for C in (0, -1, 65536, 1 << 30):
        assert _call(entry, scen=fake_scen(C=C)) == SIZE, C
    assert _call(entry, scen=fake_scen(rows=32776)) == ALIGN          # 16 bytes
    assert _call(entry, scen=fake_scen(of_env=36866)) == ALIGN        # 4 bytes
    for C in (1, 65535):                                              # in range: the alignment check comes next
        assert _call(entry, scen=fake_scen(C=C, rows=32776)) == ALIGN


@pytest.mark.parametrize("entry", ENTRIES)
def test_plain_checks_come_first_with_their_codes(entry):
    bad = fake_scen(C=0)                                              # would be RENV_E_SIZE
    assert _call(entry, env=fake_env(state=None), scen=bad) == NULL
    assert _call(entry, env=fake_env(n=0), scen=bad) == SIZE
    assert _call(entry, env=fake_env(state=4100), scen=bad) == ALIGN
    assert _call(entry, env=fake_env(elapsed=None), scen=bad) == NULL      # neither counter layout
    if entry == "reset":
        return
    assert _call(entry, log=fake_log(capacity=0), scen=bad) == SIZE
    assert _call(entry, log=fake_log(count=None), scen=bad) == NULL
    assert _call(entry, integrator=2, scen=bad) == INTEGRATOR
    # the uint16 counter holds at most 65535 steps
    assert _call(entry, env=fake_env(elapsed=None, elapsed16=4096), max_steps=65536, scen=bad) == SIZE
    if entry == "step":
        assert _call(entry, action=None, scen=bad) == NULL
        assert _call(entry, done=None, scen=bad) == NULL
        assert _call(entry, reward=45060, scen=bad) == ALIGN
        assert _call(entry, counters=49156, scen=bad) == ALIGN
        return
    assert _call(entry, stats=None, scen=bad) == NULL
    assert _call(entry, stats=16388, scen=bad) == ALIGN
    for K in (0, -1, (1 << 30) + 1):
        assert _call(entry, K=K, scen=bad) == SIZE
    if entry in ("rollout_mlp", "collect_mlp"):
        assert _call(entry, policy=fake_policy(act=2), scen=bad) == ARG
        assert _call(entry, policy=fake_policy(params=4100), scen=bad) == ALIGN
    if entry == "collect_mlp":
        assert _call(entry, traj=fake_traj(capacity=4), scen=bad) == ARG
        assert _call(entry, sample=2, scen=bad) == ARG
        assert _call(entry, traj=fake_traj(obs=None), scen=bad) == NULL


def test_random_policy_rollout_checks_the_same_way():
    assert _call("rollout", w=False, scen=None) == NULL
    assert _call("rollout", w=False, stats=None, scen=fake_scen(C=0)) == NULL


# ---- Python checks (none of them reaches CUDA) ----------------------------------------------------------------------
def _rows(C=3, device="cpu"):
    return Scenarios.tasks(np.tile([[9.8, 1.0, 0.1, 0.5]], (C, 1)), device=device)


class _CudaRows(Scenarios):
    """Scenarios that claim a CUDA device, so that set_scenarios gets past its device check on a CPU-only machine."""

    def __init__(self, C):
        Scenarios.__init__(self, _rows(C).rows)
        self.device = torch.device("cuda", 0)


@pytest.mark.parametrize("kw", [dict(dtype="float64"), dict(noisy=True)])
def test_set_scenarios_refuses_fp64_and_noisy_envs(kw):
    env = RandomCartPoleVecEnv(8, **kw)
    with pytest.raises(ValueError, match="float32 env without observation noise"):
        env.set_scenarios(_CudaRows(3), [0] * 8)
    assert env._buffers is None                       # nothing was allocated


def test_set_scenarios_validates_the_assignment_on_the_host():
    env = RandomCartPoleVecEnv(8)
    s = _CudaRows(3)
    with pytest.raises(TypeError):
        env.set_scenarios(_rows(3).rows, [0] * 8)               # a tensor, not a Scenarios
    with pytest.raises(ValueError, match="CUDA device|env's device"):
        env.set_scenarios(_rows(3), [0] * 8)                    # scenarios on the CPU
    with pytest.raises(ValueError, match="needs an assignment"):
        env.set_scenarios(s)
    with pytest.raises(ValueError, match="shape"):
        env.set_scenarios(s, [0] * 7)
    with pytest.raises(ValueError, match="shape"):
        env.set_scenarios(s, np.zeros((8, 1), np.int64))
    for bad in (np.zeros(8, np.float32), np.zeros(8, bool), torch.zeros(8, dtype=torch.float64)):
        with pytest.raises(ValueError, match="integer"):
            env.set_scenarios(s, bad)
    for bad in ([0, 1, 2, 3, 0, 1, 2, -1], [0] * 7 + [3], torch.full((8,), 70000)):
        with pytest.raises(ValueError, match=r"\[0, 3\)"):
            env.set_scenarios(s, bad)
    with pytest.raises(ValueError, match="no assignment"):
        env.set_scenarios(None, [0] * 8)
    env.set_scenarios(None)                                     # nothing set: a no-op
    assert env.scenarios is None and env._buffers is None
    with pytest.raises(ValueError, match="no scenarios"):
        env.scenario_stats()


def test_set_scenarios_refuses_too_many_rows():
    env = RandomCartPoleVecEnv(8)

    class Many(_CudaRows):
        def __len__(self):
            return 65536
    with pytest.raises(ValueError, match="65535"):
        env.set_scenarios(Many(1), [0] * 8)


# ---- ADR boundary rows ----------------------------------------------------------------------------------------------
def test_adr_boundaries_rows_are_the_pinned_boxes():
    lo, hi = [2.0, 0.5, 0.05, 0.1], [20.0, 3.0, 0.3, 1.0 / 3.0]
    s = Scenarios.adr_boundaries(lo, hi, device="cpu")
    assert len(s) == 9
    boxes = [[lo, hi]]
    for k in range(4):
        for v in (lo[k], hi[k]):
            pl, ph = list(lo), list(hi)
            pl[k] = ph[k] = v
            boxes.append([pl, ph])
    for c, (pl, ph) in enumerate(boxes):
        distr = [x for pair in zip(pl, ph) for x in pair]
        ref = Scenarios.distributions("uniform", [distr], device="cpu").rows[0]
        assert s.rows[c].numpy().tobytes() == ref.numpy().tobytes(), c
    # a pinned dim has width 0 (the draw is lo exactly); the others keep the box
    r = s.rows.numpy()
    assert _lib.DR_UNIFORM == r[0, :1].view(np.int32)[0]
    for k in range(4):
        for j, v in enumerate((lo[k], hi[k])):
            row = r[1 + 2 * k + j]
            assert row[2 + k] == np.float32(v) and row[6 + k] == 0.0
            others = [d for d in range(4) if d != k]
            assert np.array_equal(row[[2 + d for d in others]], r[0, [2 + d for d in others]])
            assert np.array_equal(row[[6 + d for d in others]], r[0, [6 + d for d in others]])


def test_adr_boundaries_reject_bad_boxes():
    with pytest.raises(ValueError):
        Scenarios.adr_boundaries([1.0] * 3, [2.0] * 3, device="cpu")
    with pytest.raises(ValueError):
        Scenarios.adr_boundaries([[1.0] * 4], [[2.0] * 4], device="cpu")


# ---- compiled form --------------------------------------------------------------------------------------------------
def test_scenario_kernels_compile_without_spills_and_keep_the_hot_paths():
    sys.path.insert(0, os.path.join(ROOT, "profiles"))
    import sass_stats
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    kinds = {k: [n for n in sass if "cartpole_scen_%s_kernel" % k in n]
             for k in ("reset", "step", "rollout", "rollout_mlp", "collect_mlp")}
    assert [len(kinds[k]) for k in ("reset", "step", "rollout", "rollout_mlp", "collect_mlp")] == [1, 4, 8, 8, 8], kinds
    # the pre-existing kernels keep their names and counts (the new ones match none of their substrings)
    for needle, count in (("logged_kernel", 10), ("cartpole_step_kernel", 10), ("cartpole_rollout_kernelId", 6),
                          ("cartpole_rollout_mlp_kernel", 8), ("cartpole_collect_mlp_kernel", 8),
                          ("cartpole_population_", 6), ("cartpole_grid_", 6), ("rollout_pair", 4)):
        assert sum(needle in n for n in sass) == count, needle
    for name in kinds["rollout_mlp"] + kinds["collect_mlp"]:
        ops = [op for _, op, _ in sass[name]]
        assert sum(op.startswith("HMMA.1688.F32.TF32") for op in ops) == 192, name
    for name in kinds["step"]:
        ops = [op for _, op, _ in sass[name]]
        assert sum(op.startswith("LDG.E.128") for op in ops) >= 9, name      # the plain step's 128-bit tile loads
        assert "ACQBULK" in ops and "PREEXIT" in ops, name
    blocks = ptxas_blocks()
    regs = lambda name: int(re.search(r"Used (\d+) registers", blocks[name]).group(1))
    for name in sum(kinds.values(), []):
        assert re.search(r"\b0 bytes spill stores, 0 bytes spill loads", blocks[name]), name
    for name in kinds["step"]:
        assert regs(name) <= 64, (name, regs(name))                           # 4 CTAs of 256 threads per SM
    for name in kinds["rollout"]:
        assert regs(name) <= 80, (name, regs(name))                           # 3 CTAs of 256 threads per SM
    for name in kinds["rollout_mlp"] + kinds["collect_mlp"]:
        assert regs(name) <= 65536 // (128 * 3), (name, regs(name))
