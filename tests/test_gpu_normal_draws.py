"""Every fp32 normal, truncated-normal, full-Gaussian and observation-noise draw, value for value, against the float64
restatement of the fp32 draw contract (oracle/f32_draws.py): each output element must lie within the bound derived
from the transform errors stated in renv_dr.cuh.  Draws whose accept / reject decision falls within that bound of a
floor are ambiguous and may take either branch; every other value must match.

Covers the sampler (packed attempt 0, the two-sample loop and the one-sample tail, sampler_redo_block with attempts 1
and 2, give-ups), the env-reset xi of reset(), step() and rollout(), the observation noise of the Noisy envs, and both
fullgaussian kernels (FMA chain at D = 4, 8, 16; tcgen05 at 23 and 30 dims, up to ~14 tiles per CTA).
"""
import numpy as np
import pytest
import torch

import random_envs_b200 as random_envs
from random_envs_b200.random_env import covariance_factor
from oracle import f32_draws as F

pytestmark = pytest.mark.gpu

ENV_BY_DIM = {3: "RandomHopperUnmodeled-v0", 4: "RandomCartPole-v0", 5: "RandomHalfCheetahUnmodeled-v0",
              8: "RandomHalfCheetah-v0", 9: "RandomWalker2dUnmodeled-v0", 13: "RandomWalker2d-v0",
              23: "RandomHumanoidUnmodeled-v0", 30: "RandomHumanoid-v0"}
SEED = (3 << 32) | 41
CART_SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]


def _np(t):
    return t.detach().double().cpu().numpy()


def _interleave(a, b):
    return list(np.stack([a, b], 1).reshape(-1))


def _dr_params(law, lb, dim, rs):
    """mean = floor + c std with c in [-0.6, 2.5]: a large share of blocks retry, some dims give up."""
    std = rs.uniform(0.05, 2.0, dim)
    floor = np.asarray(lb, float) if law == "truncnorm" else np.full(dim, F.GAUSSIAN_FLOOR)
    c = rs.uniform(-0.6, 2.5, dim)
    c[0] = -0.6
    return floor + c * std, std, floor


def _check_sampler_call(s, law, mean, std, floor, n, tick, id0):
    x = s.sample_tasks_tensor(n, dtype=torch.float32, sample_id0=id0)
    viol = int(s._dr_violations[0].item())
    s._dr_violations.zero_()
    ids = np.uint64(id0) + np.arange(n, dtype=np.uint64)
    ref = F.sample_dr(law, SEED, ids, tick, F.PURPOSE_TASKS, mean, std, floor)
    F.check_dr(_np(x), ref)
    if law == "gaussian":
        sure = ref["gave_up"] & ~ref["ambiguous"]
        assert int(sure.sum()) <= viol <= int((ref["gave_up"] | ref["ambiguous"]).sum())
    else:
        assert viol == 0
    redone = (ref["candidates"][:, :, 0] < F.f32(floor)).reshape(n, -1)
    return redone, ref


@pytest.mark.parametrize("law", ["gaussian", "truncnorm"])
@pytest.mark.parametrize("dim", sorted(ENV_BY_DIM))
def test_sampler_values_follow_the_fp32_contract(law, dim):
    env_id = ENV_BY_DIM[dim]
    rs = np.random.RandomState(dim)
    lb = random_envs.XI_TABLES[env_id].lower_bounds
    mean, std, floor = _dr_params(law, lb, dim, rs)
    s = random_envs.TaskSampler(env_id); s.seed_dr(SEED)
    s.set_dr_distribution(law, _interleave(mean, std))
    s._violation_counter(torch.device("cuda", torch.cuda.current_device())).zero_()
    # call 0: 4099 samples (per thread: the two-sample loop, then a one-sample tail); call 1 across sample id 2^32
    redone0, ref0 = _check_sampler_call(s, law, mean, std, floor, 4099, 0, 0)
    redone1, ref1 = _check_sampler_call(s, law, mean, std, floor, 1501, 1, (1 << 32) - 700)
    blocks = np.concatenate([redone0, redone1]).reshape(-1)
    assert blocks.mean() > 0.01                                  # sampler_redo_block runs for > 1 % of the dims
    for ref in (ref0, ref1):
        cand = ref["candidates"]
        f32floor = F.f32(floor)
        assert ((cand[:, :, 0] < f32floor) & (cand[:, :, 1] < f32floor) & (cand[:, :, 2] >= f32floor)).any()  # attempt 2
        assert ref["gave_up"].any()                              # give-up: lb (truncnorm) / a violation (gaussian)


def test_gaussian_violations_raise_exactly_when_the_contract_gives_up():
    """check_dr_violations raises after a call in which the contract gives up on some dim, and only then."""
    s = random_envs.TaskSampler("RandomCartPole-v0"); s.seed_dr(SEED)
    mean, std = np.array([9.8, 1.0, 0.3, 0.5]), np.array([1.0, 0.1, 0.5, 0.05])   # pole mass: 4 % give up
    s.set_dr_distribution("gaussian", _interleave(mean, std))
    seen = set()
    for call in range(40):
        x = s.sample_tasks_tensor(10, dtype=torch.float32)
        ref = F.sample_dr("gaussian", SEED, np.arange(10, dtype=np.uint64), call, F.PURPOSE_TASKS, mean, std,
                          np.full(4, 0.1))
        F.check_dr(_np(x), ref)
        if ref["ambiguous"].any():
            s._dr_violations.zero_()
            continue
        gave_up = bool(ref["gave_up"].any())
        seen.add(gave_up)
        if gave_up:
            with pytest.raises(Exception, match="Not all samples were above"):
                s.check_dr_violations()
        else:
            s.check_dr_violations()
    assert seen == {False, True}


# ----------------------------------------------------------------------------- env-reset xi
def _env(law, n, seed, env_id0, **kw):
    env = random_envs.RandomCartPoleVecEnv(n, dtype="float32", seed=seed, env_id0=env_id0, **kw)
    rs = np.random.RandomState(5)
    if law == "fullgaussian":
        a = 0.3 * rs.randn(4, 4) + 0.6 * np.eye(4)
        mean, cov = np.array([1.5, 2.0, 2.5, 1.0]), a @ a.T
        env.set_dr_distribution("fullgaussian", {"mean": mean, "cov": cov})
        lo, hi = env.get_task_search_bounds()
        ref = lambda ids, tick: F.fullgaussian_sample(seed, ids, tick, F.PURPOSE_XI, mean, covariance_factor(cov), lo, hi)
    else:
        lb = random_envs.XI_TABLES["RandomCartPole-v0"].lower_bounds
        mean, std, floor = _dr_params(law, lb, 4, rs)
        env.set_dr_distribution(law, _interleave(mean, std))
        ref = lambda ids, tick: F.sample_dr(law, seed, ids, tick, F.PURPOSE_XI, mean, std, floor)
    env.set_dr_training(True)
    return env, ref


def _check_xi(got, ref):
    if isinstance(ref, tuple):
        value, bound = ref
        err = np.abs(got - value) - bound
        assert np.all(err <= 0), (np.max(err), np.argwhere(err > 0)[0])
    else:
        F.check_dr(got, ref)


def _matches(got, ref):
    if isinstance(ref, tuple):
        return np.all(np.abs(got - ref[0]) <= ref[1], axis=1)
    ok = np.abs(got - ref["value"]) <= ref["bound"]
    amb = ref["ambiguous"]
    near = (np.abs(got[..., None] - ref["candidates"]) <= ref["cand_bound"]).any(-1)
    return np.all(np.where(amb, near, ok), axis=1)


@pytest.mark.parametrize("law", ["gaussian", "truncnorm", "fullgaussian"])
def test_env_reset_xi_follows_the_fp32_contract(law):
    n, seed, id0 = 3001, 77, (1 << 32) - 1000
    env, ref = _env(law, n, seed, id0, max_episode_steps=7)
    ids = np.uint64(id0) + np.arange(n, dtype=np.uint64)
    env.reset()                                                   # tick 0
    _check_xi(_np(env.get_task()), ref(ids, 0))
    for tick in range(1, 16):                                     # auto-resets inside step() at the step's tick
        before = _np(env.get_task())
        _, _, done, _ = env.step(env.sample_actions())
        d = done.cpu().numpy()
        after = _np(env.get_task())
        assert np.array_equal(after[~d], before[~d])
        if d.any():
            _check_xi(after[d], ref(ids[d], tick))
    assert env._tick == 16
    before = _np(env.get_task())
    K = 20
    env.rollout((0.0, 0.0, 1.0, 0.3), 0.0, K)                     # steps at ticks 16 .. 35
    after = _np(env.get_task())
    changed = np.any(after != before, axis=1)
    assert changed.mean() > 0.5
    found = np.zeros(int(changed.sum()), bool)
    for tick in range(16, 16 + K):                                # the last reset of an env happened at one of them
        found |= _matches(after[changed], ref(ids[changed], tick))
    assert found.all(), np.argwhere(~found)[:5]


# ----------------------------------------------------------------------------- observation noise
@pytest.mark.parametrize("n", [1, 1027])
def test_observation_noise_follows_the_fp32_contract(n):
    level = 2e-3
    env = random_envs.RandomCartPoleVecEnv(n, dtype="float32", seed=SEED, noisy=True, noise_level=level, max_episode_steps=5)
    env.set_dr_distribution("uniform", CART_SEARCH); env.set_dr_training(True)
    ids = np.arange(n, dtype=np.uint64)
    std = np.sqrt(level)
    o = _np(env.reset())
    value, bound = F.obs_noise(SEED, ids, 0, 1, _np(env.state), std)      # the reset's observation: which = 1
    assert np.all(np.abs(o - value) <= bound)
    for tick in range(1, 12):
        o, _, done, _ = env.step(env.sample_actions())
        o, d, s = _np(o), done.cpu().numpy(), _np(env.state)
        which = d.astype(int)
        for w in (0, 1):
            sel = which == w
            if sel.any():
                value, bound = F.obs_noise(SEED, ids[sel], tick, w, s[sel], std)
                err = np.abs(o[sel] - value) - bound
                assert np.all(err <= 0), (tick, w, np.max(err))
    assert env._tick == 12
    # rollout() leaves the observation of its last step (tick 12 + K - 1): which = 1 for an env that reset there
    K = 9
    env.rollout((0.0, 0.0, 1.0, 0.3), 0.0, K)
    o, s = _np(env.obs), _np(env.state)
    ok = np.zeros(n, bool)
    for w in (0, 1):
        value, bound = F.obs_noise(SEED, ids, 12 + K - 1, w, s, std)
        ok |= np.all(np.abs(o - value) <= bound, axis=1)
    assert ok.all(), np.argwhere(~ok)[:5]


# ----------------------------------------------------------------------------- fullgaussian sampler
def _fullgaussian_sampler(env_id, dim, tensor, seed=21):
    rs = np.random.RandomState(dim)
    a = 0.2 * rs.randn(dim, dim) + 0.5 * np.eye(dim)
    cov, mean = a @ a.T, rs.uniform(1.0, 3.0, dim)
    s = random_envs.TaskSampler(env_id); s.seed_dr(seed)
    s.set_dr_distribution("fullgaussian", {"mean": mean, "cov": cov})
    lo, hi = s.get_task_search_bounds()
    return s, mean, covariance_factor(cov), lo, hi


def _check_fullgaussian(x, seed, id0, tick, mean, f, lo, hi, tensor_core, chunk=1 << 17):
    n = x.shape[0]
    for start in range(0, n, chunk):
        stop = min(n, start + chunk)
        ids = np.uint64(id0) + np.arange(start, stop, dtype=np.uint64)
        value, bound = F.fullgaussian_sample(seed, ids, tick, F.PURPOSE_TASKS, mean, f, lo, hi, tensor_core)
        got = _np(x[start:stop])
        err = np.abs(got - value) - bound
        assert np.all(err <= 0), (start, np.max(err), np.argwhere(err > 0)[0])


@pytest.mark.parametrize("dim", [3, 4, 5, 8, 9, 13])
def test_fullgaussian_fma_chain_kernel_follows_the_fp32_contract(dim):
    s, mean, f, lo, hi = _fullgaussian_sampler(ENV_BY_DIM[dim], dim, False)
    x = s.sample_tasks_tensor(1000 + dim, dtype=torch.float32)
    _check_fullgaussian(x, 21, 0, 0, mean, f, lo, hi, False)
    y = s.sample_tasks_tensor(300, dtype=torch.float32, sample_id0=(1 << 32) - 100)
    _check_fullgaussian(y, 21, (1 << 32) - 100, 1, mean, f, lo, hi, False)


@pytest.mark.parametrize("dim", [23, 30])
@pytest.mark.parametrize("n", [37, 128 * 5, (1 << 20) + 77])
def test_fullgaussian_tensor_core_kernel_follows_the_fp32_contract(dim, n):
    """(1 << 20) + 77 samples are 8193 tiles: about 14 per CTA, so every CTA cycles its two accumulators and the
    mbarrier parity many times."""
    s, mean, f, lo, hi = _fullgaussian_sampler(ENV_BY_DIM[dim], dim, True)
    x = s.sample_tasks_tensor(n, dtype=torch.float32)
    y = s.sample_tasks_tensor(n, dtype=torch.float32, sample_id0=5)
    s.check_dr_violations()                 # raises if a CTA's wait for its MMAs timed out
    _check_fullgaussian(x, 21, 0, 0, mean, f, lo, hi, True)
    _check_fullgaussian(y, 21, 5, 1, mean, f, lo, hi, True)
