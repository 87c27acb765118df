"""Scenario mixtures without a GPU: argument validation of the five mixture entry points, the struct layout, the
alias-table builder against exact probabilities, the host draw against the C oracle's Philox words, and the Python
checks of set_scenario_mixture."""
import ctypes

import numpy as np
import pytest
import torch

import mixture_oracle
from abi_support import HEADER, fake_env, fake_log, fake_policy, fake_traj, gcc_layout
from oracle import c_oracle
from random_envs_b200 import RandomCartPoleVecEnv, Scenarios, _lib
from random_envs_b200.vector_env import _mixture_table

NULL, ALIGN, SIZE, INTEGRATOR, ARG = -1, -2, -3, -6, -7
ENTRIES = ("reset", "step", "rollout", "rollout_mlp", "collect_mlp")


def fake_mix(**kw):
    m = _lib.EnvMixture()
    m.rows, m.table, m.of_env, m.C = 32768, 34816, 36864, 5
    for k, v in kw.items():
        setattr(m, k, v)
    return m


def _call(entry, env=None, mix="default", log=None, **kw):
    lib = _lib.load()
    e = ctypes.byref(env if env is not None else fake_env())
    m = ctypes.byref(fake_mix()) if isinstance(mix, str) else (ctypes.byref(mix) if mix is not None else None)
    lg = ctypes.byref(log) if log is not None else None
    K, integ, max_steps = kw.get("K", 5), kw.get("integrator", 0), kw.get("max_steps", 500)
    stats = kw.get("stats", 16384)
    if entry == "reset":
        return lib.renv_cartpole_reset_mix_f32(e, m, kw.get("mask"), 0, None, None)
    if entry == "step":
        return lib.renv_cartpole_step_mix_f32(e, m, lg, kw.get("action", 40960), kw.get("reward", 45056),
                                              kw.get("done", 49152), kw.get("truncated", 53248), integ, max_steps, 0,
                                              kw.get("counters"), None)
    if entry == "rollout":
        w = (ctypes.c_double * 4)(0.0, 0.0, 1.0, 0.0) if kw.get("w", True) else None
        return lib.renv_cartpole_rollout_mix_f32(e, m, lg, w, 0.0, K, integ, max_steps, 0, stats, None, None)
    p = ctypes.byref(kw.get("policy", fake_policy()))
    if entry == "rollout_mlp":
        return lib.renv_cartpole_rollout_mlp_mix_f32(e, m, lg, p, K, integ, max_steps, 0, stats, None, None)
    t = ctypes.byref(kw.get("traj", fake_traj()))
    return lib.renv_cartpole_collect_mlp_mix_f32(e, m, lg, p, t, kw.get("sample", 1), K, integ, max_steps, 0, stats,
                                                 None, None)


# ---- C ABI ----------------------------------------------------------------------------------------------------------
def test_mixture_structs_in_python_match_the_header(tmp_path):
    fields = [f for f, _ in _lib.EnvMixture._fields_]
    got = gcc_layout(tmp_path, "renv_env_mixture", fields)
    for f in fields:
        assert int(got[f]) == getattr(_lib.EnvMixture, f).offset, f
    assert int(got["sizeof"]) == ctypes.sizeof(_lib.EnvMixture)
    entry = gcc_layout(tmp_path, "renv_alias_entry", ["q", "alias", "pad"])
    assert (int(entry["q"]), int(entry["alias"]), int(entry["sizeof"])) == (0, 4, 8)


def test_symbols_are_exported_and_declared():
    lib = _lib.load()
    header = open(HEADER).read()
    for entry in ENTRIES:
        name = "renv_cartpole_%s_mix_f32" % entry
        assert hasattr(lib, name) and name in _lib.SIGNATURES
        assert name + "(" in header
    assert "purpose 6" in header


@pytest.mark.parametrize("entry", ENTRIES)
def test_mixture_errors_before_any_cuda_call(entry):
    assert _call(entry, mix=None) == NULL
    for f in ("rows", "table", "of_env"):
        assert _call(entry, mix=fake_mix(**{f: None})) == NULL, f
    for C in (0, -1, 65536, 1 << 30):
        assert _call(entry, mix=fake_mix(C=C)) == SIZE, C
    assert _call(entry, mix=fake_mix(rows=32776)) == ALIGN           # 16 bytes
    assert _call(entry, mix=fake_mix(table=34820)) == ALIGN          # 8 bytes
    assert _call(entry, mix=fake_mix(of_env=36866)) == ALIGN         # 4 bytes
    for C in (1, 65535):
        assert _call(entry, mix=fake_mix(C=C, table=34820)) == ALIGN


@pytest.mark.parametrize("entry", ENTRIES)
def test_plain_checks_come_first_with_their_codes(entry):
    bad = fake_mix(C=0)
    assert _call(entry, env=fake_env(state=None), mix=bad) == NULL
    assert _call(entry, env=fake_env(n=0), mix=bad) == SIZE
    assert _call(entry, env=fake_env(state=4100), mix=bad) == ALIGN
    assert _call(entry, env=fake_env(elapsed=None), mix=bad) == NULL
    if entry == "reset":
        return
    assert _call(entry, log=fake_log(capacity=0), mix=bad) == SIZE
    assert _call(entry, integrator=2, mix=bad) == INTEGRATOR
    assert _call(entry, env=fake_env(elapsed=None, elapsed16=4096), max_steps=65536, mix=bad) == SIZE
    if entry == "step":
        assert _call(entry, action=None, mix=bad) == NULL
        assert _call(entry, reward=45060, mix=bad) == ALIGN
        return
    assert _call(entry, stats=None, mix=bad) == NULL
    assert _call(entry, K=0, mix=bad) == SIZE
    if entry in ("rollout_mlp", "collect_mlp"):
        assert _call(entry, policy=fake_policy(act=2), mix=bad) == ARG
    if entry == "collect_mlp":
        assert _call(entry, sample=2, mix=bad) == ARG


# ---- the alias table ------------------------------------------------------------------------------------------------
def _weights(kind, C, rng):
    if kind == "random":
        return rng.random(C)
    if kind == "onehot":
        w = np.zeros(C)
        w[C // 2] = 3.0
        return w
    if kind == "zeros":
        w = rng.random(C)
        w[::3] = 0.0
        if not w.any():
            w[-1] = 1.0
        return w
    w = np.full(C, 1e-9)                 # very skewed
    w[0] = 1e6
    return w


@pytest.mark.parametrize("C", [1, 2, 9, 1000, 65535])
@pytest.mark.parametrize("kind", ["random", "onehot", "zeros", "skewed"])
def test_table_probabilities_are_the_weights(C, kind):
    rng = np.random.default_rng(C)
    w = _weights(kind, C, rng)
    _, table = _mixture_table(w, C)
    counts = np.array(mixture_oracle.exact_counts(table), dtype=object)
    assert sum(counts) == 1 << 64
    prob = np.array([float(c) for c in counts]) / 2.0 ** 64
    assert np.all(np.abs(prob - w / w.sum()) <= C * 2.0 ** -31)
    assert all(counts[j] == 0 for j in np.nonzero(w == 0)[0])           # weight 0: never drawn, exactly
    q, alias = mixture_oracle.split(table)
    full = q == 2 ** 32 - 1
    assert np.array_equal(alias[full], np.nonzero(full)[0])             # a column keeping all its mass aliases itself
    assert np.all(alias < C)


def test_host_draw_uses_the_c_oracle_philox_words():
    C, seed = 9, 0x1234_5678_9ABC
    _, table = _mixture_table(np.arange(1.0, C + 1), C)
    q, alias = mixture_oracle.split(table)
    ids, ticks = np.array([0, 5, 77, (1 << 40) + 3]), np.array([1, 2, 1 << 33, 9])
    got = mixture_oracle.draw_rows(seed, ids, ticks, table)
    for k in range(len(ids)):
        i, t = int(ids[k]), int(ticks[k])
        ctr = (i & 0xFFFFFFFF, ((i >> 32) & 0xFFFF) | (((t >> 32) & 0xFFFF) << 16), t & 0xFFFFFFFF, 6 << 24)
        x, y = c_oracle.philox(ctr, (seed & 0xFFFFFFFF, seed >> 32))[:2]
        j = (x * C) >> 32
        assert got[k] == (j if y < q[j] else alias[j])


def test_host_draw_frequencies_follow_the_weights():
    w = np.array([0.5, 0.0, 0.25, 0.125, 0.125])
    _, table = _mixture_table(w, len(w))
    rows = mixture_oracle.draw_rows(7, np.arange(200000), 3, table)
    freq = np.bincount(rows, minlength=len(w)) / len(rows)
    assert freq[1] == 0.0
    assert np.all(np.abs(freq - w) < 0.005)


# ---- Python checks --------------------------------------------------------------------------------------------------
class _CudaRows(Scenarios):
    def __init__(self, C):
        Scenarios.__init__(self, Scenarios.tasks(np.tile([[9.8, 1.0, 0.1, 0.5]], (C, 1)), device="cpu").rows)
        self.device = torch.device("cuda", 0)


@pytest.mark.parametrize("kw", [dict(dtype="float64"), dict(noisy=True)])
def test_set_scenario_mixture_refuses_fp64_and_noisy_envs(kw):
    env = RandomCartPoleVecEnv(8, **kw)
    with pytest.raises(ValueError, match="mixture needs a float32 env without observation noise"):
        env.set_scenario_mixture(_CudaRows(3), [1, 1, 1])
    assert env._buffers is None


@pytest.mark.parametrize("weights, match", [
    ([1.0, 1.0], "shape"), ([[1.0, 1.0, 1.0]], "shape"), ([1.0, -1.0, 1.0], ">= 0"), ([1.0, np.nan, 1.0], "finite"),
    ([1.0, np.inf, 1.0], "finite"), ([0.0, 0.0, 0.0], "positive sum"), (torch.tensor([1.0, -2.0, 0.0]), ">= 0"),
])
def test_set_scenario_mixture_validates_the_weights(weights, match):
    env = RandomCartPoleVecEnv(8)
    with pytest.raises(ValueError, match=match):
        env.set_scenario_mixture(_CudaRows(3), weights)
    assert env._buffers is None


def test_set_scenario_mixture_validates_rows_and_device():
    env = RandomCartPoleVecEnv(8)
    with pytest.raises(TypeError):
        env.set_scenario_mixture(_CudaRows(3).rows, [1, 1, 1])
    with pytest.raises(ValueError, match="env's device"):
        env.set_scenario_mixture(Scenarios.tasks([[9.8, 1.0, 0.1, 0.5]], device="cpu"), [1.0])
    big = _CudaRows(1)
    big.rows = big.rows.expand(65536, -1)
    with pytest.raises(ValueError, match="65535"):
        env.set_scenario_mixture(big, np.ones(65536))
    with pytest.raises(ValueError, match="no scenario mixture"):
        env.set_mixture_weights([1.0])
    assert env.scenario_weights is None
