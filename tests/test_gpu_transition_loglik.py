"""Offline DR log-likelihood on the GPU: the kernel against the float64 oracle over both integrators, window lengths,
sample counts, DR laws and eps forms; the compensated totals; bitwise reproducibility across batch composition and
repeated calls; the -inf and NaN edge cases; common random numbers across candidates; and recovery of the task that
generated the data."""
import ctypes
import math

import numpy as np
import pytest
import torch

import random_envs_b200 as random_envs
from oracle import transition_loglik as oracle
from random_envs_b200 import _device, _lib
from random_envs_b200.random_env import GAUSSIAN_FAIL_MSG

pytestmark = pytest.mark.gpu

XI_TRUE = (12.0, 1.5, 0.2, 0.7)
SIGMA = 1e-2                                  # noise_level 1e-4
EPS = 2 * SIGMA ** 2
EPS_VEC = [1e-4, 3e-4, 2e-4, 4e-4]
LOWER = np.array([2.0, 0.5, 0.05, 0.1])      # cart-pole search bounds (the fullgaussian normalisation)
UPPER = np.array([20.0, 3.0, 0.3, 1.0])


def _tol(ref):
    return 1e-9 * np.maximum(1.0, np.abs(ref))


def _record(n, K, euler=True, seed=0, xi=XI_TRUE):
    """Noisy fp64 transitions under sample_actions() at a fixed task.  The transition of a `done` step ends in the
    reset observation, not in the dynamics' successor: it is dropped and the next transition starts an episode."""
    env = random_envs.RandomCartPoleVecEnv(n, dtype="float64", seed=seed, noisy=True, noise_level=SIGMA ** 2,
                                           kinematics_integrator="euler" if euler else "semi-implicit")
    env.set_task(*xi)
    env.reset()
    obs, act, nxt, done = [], [], [], []
    for _ in range(K):
        o = env.obs.clone()
        a = env.sample_actions().clone()
        o2, _, d, _ = env.step(a)
        obs.append(o); act.append(a); nxt.append(o2.clone()); done.append(d.clone())
    # env-major order: transition k of env i at i * K + k
    obs, nxt = (torch.stack(v, 1).reshape(-1, 4).cpu().numpy() for v in (obs, nxt))
    act, done = (torch.stack(v, 1).reshape(-1).cpu().numpy() for v in (act, done))
    done = done.astype(bool)
    start = np.zeros(n * K, bool)
    start[::K] = True
    start[1:] |= done[:-1]
    keep = ~done
    return obs[keep], act[keep], nxt[keep], np.flatnonzero(start[keep])


@pytest.fixture(scope="module")
def recorded():
    return {euler: _record(4, 48, euler, seed=3 + euler) for euler in (True, False)}


def _distrs(kind):
    mean = np.array(XI_TRUE)
    if kind == "uniform":
        return [list(np.stack([0.8 * mean, 1.2 * mean], 1).reshape(-1)), list(np.stack([0.9 * mean, 1.3 * mean], 1).reshape(-1))]
    if kind == "truncnorm":
        return [list(np.stack([mean, 0.1 * mean], 1).reshape(-1)), list(np.stack([1.1 * mean, 0.05 * mean], 1).reshape(-1))]
    assert kind == "fullgaussian"
    mu = 4 * (mean - LOWER) / (UPPER - LOWER)
    cov = 0.02 * (np.eye(4) + 0.3 * (np.ones((4, 4)) - np.eye(4)))
    return [{"mean": mu, "cov": cov}, {"mean": mu * 0.95, "cov": 0.5 * cov}]


CASES = [  # (euler, lam, M, DR law, eps)
    (True, 1, 2, "uniform", EPS),
    (False, 1, 33, "truncnorm", EPS_VEC),
    (True, 3, 256, "fullgaussian", EPS_VEC),
    (False, 3, 33, "fullgaussian", EPS),
    (False, 8, 256, "uniform", EPS),
    (True, 8, 33, "truncnorm", EPS_VEC),
]


@pytest.mark.parametrize("euler,lam,M,kind,eps", CASES)
def test_loglik_matches_the_oracle(recorded, euler, lam, M, kind, eps):
    obs, act, nxt, starts = recorded[euler]
    data = random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    xi = data.sample_candidates(kind, _distrs(kind), num_samples=M, seed=11)
    integ = "euler" if euler else "semi-implicit"
    total, ll = data.log_likelihood(xi, lam=lam, epsilon=eps, kinematics_integrator=integ, per_window=True)
    windows = data.window_starts(lam)
    assert np.array_equal(windows, oracle.window_starts(len(obs), lam, starts)) and len(windows) >= 40
    ref, ref_total = oracle.loglik(obs, act, nxt, windows, xi.cpu().numpy(), lam, eps, euler)
    got = ll.cpu().numpy()
    assert np.all(np.isfinite(ref)) and got.shape == ref.shape
    err = np.abs(got - ref)
    assert np.all(err <= _tol(ref)), (float(err.max()), float(np.max(err / _tol(ref))))
    # the totals: a compensated fixed-order sum, against math.fsum of the kernel's own values
    for c in range(len(got)):
        assert abs(float(total[c]) - math.fsum(got[c])) <= 1e-12 * abs(math.fsum(got[c])), c
        assert abs(float(total[c]) - ref_total[c]) <= 1e-9 * abs(ref_total[c])
    # the same through dr_log_likelihood (same sampler, same seed => the same xi and bits)
    t2, l2 = data.dr_log_likelihood(kind, _distrs(kind), num_samples=M, seed=11, lam=lam, epsilon=eps,
                                    kinematics_integrator=integ, per_window=True)
    assert torch.equal(t2, total) and torch.equal(l2, ll)


def test_results_do_not_depend_on_the_batch_or_on_repetition(recorded):
    obs, act, nxt, starts = recorded[False]
    data = random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    mean = np.array(XI_TRUE)
    distrs = [list(np.stack([mean * (0.8 + 0.01 * c), 0.05 * mean], 1).reshape(-1)) for c in range(37)]
    xi = data.sample_candidates("truncnorm", distrs, num_samples=301, seed=2)   # 301: two xi chunks, not a multiple of 4
    for lam in (1, 5):
        total, ll = data.log_likelihood(xi, lam=lam, epsilon=EPS_VEC, kinematics_integrator="semi", per_window=True)
        again = data.log_likelihood(xi, lam=lam, epsilon=EPS_VEC, kinematics_integrator="semi", per_window=True)
        assert torch.equal(again[0], total) and torch.equal(again[1], ll)
        for c in (0, 20, 36):
            alone_t, alone_l = data.log_likelihood(xi[c], lam=lam, epsilon=EPS_VEC, kinematics_integrator="semi",
                                                   per_window=True)
            assert torch.equal(alone_t, total[c]) and torch.equal(alone_l, ll[c])
            pair = data.log_likelihood(torch.stack([xi[(c + 1) % 37], xi[c]]), lam=lam, epsilon=EPS_VEC,
                                       kinematics_integrator="semi", per_window=True)
            assert torch.equal(pair[0][1], total[c]) and torch.equal(pair[1][1], ll[c])
        # permuting the samples reorders the sums: equal within the tolerance, not bit for bit
        perm = torch.randperm(301, generator=torch.Generator().manual_seed(0)).to(xi.device)
        pt, pl = data.log_likelihood(xi[:, perm].contiguous(), lam=lam, epsilon=EPS_VEC, kinematics_integrator="semi",
                                     per_window=True)
        ref = ll.cpu().numpy()
        assert np.all(np.abs(pl.cpu().numpy() - ref) <= _tol(ref))


def test_degenerate_covariance_gives_minus_inf_and_bad_windows_nan(recorded):
    obs, act, nxt, starts = recorded[True]
    data = random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    same = torch.tensor(XI_TRUE, dtype=torch.float64, device="cuda").repeat(2, 8, 1)
    for integ in ("euler", "semi-implicit"):
        total, ll = data.log_likelihood(same, lam=2, epsilon=0.0, kinematics_integrator=integ, per_window=True)
        assert torch.all(ll == -math.inf) and torch.all(total == -math.inf)
        assert torch.all(torch.isfinite(data.log_likelihood(same, lam=2, epsilon=EPS, kinematics_integrator=integ)))
    # Euler, lam = 1: x and theta rows of Sigma vanish, so eps on x or theta alone is not enough
    xi = data.sample_candidates("uniform", _distrs("uniform"), num_samples=64)
    assert torch.all(data.log_likelihood(xi, epsilon=[0.0, 1e-4, 1e-4, 1e-4]) == -math.inf)
    assert torch.all(torch.isfinite(data.log_likelihood(xi, epsilon=[1e-4, 0.0, 1e-4, 0.0])))

    # out-of-range windows through the raw ABI: NaN for them and for the totals, every other value unchanged
    lam, T = 3, data.num_transitions
    good = torch.as_tensor(data.window_starts(lam)[:50], device="cuda")
    bad = good.clone()
    bad[7], bad[31] = T - 2, -1                                          # t + lam > T, t < 0
    out = {}
    for name, win in (("good", good), ("bad", bad)):
        d = _lib.Transitions()
        d.obs, d.next_obs, d.action, d.window = (data.obs.data_ptr(), data.next_obs.data_ptr(), data.actions.data_ptr(),
                                                 win.data_ptr())
        d.T, d.W = T, win.numel()
        ll = torch.empty((2, d.W), dtype=torch.float64, device="cuda")
        total = torch.empty(2, dtype=torch.float64, device="cuda")
        _lib.call("renv_cartpole_transition_loglik_f64", ctypes.byref(d), lam, _lib.EULER, _device.ptr(xi), 2, 64,
                  (ctypes.c_double * 4)(*[EPS] * 4), _device.ptr(ll), _device.ptr(total), _device.stream_ptr(ll.device))
        out[name] = (total.clone(), ll.clone())
    keep = torch.ones(50, dtype=torch.bool)
    keep[[7, 31]] = False
    assert torch.all(torch.isnan(out["bad"][1][:, ~keep])) and torch.all(torch.isnan(out["bad"][0]))
    assert torch.equal(out["bad"][1][:, keep], out["good"][1][:, keep])
    assert torch.all(torch.isfinite(out["good"][0]))


def test_candidates_share_their_random_numbers(recorded):
    obs, act, nxt, starts = recorded[True]
    data = random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    lo0, hi0 = np.array([5.0, 0.5, 0.05, 0.2]), np.array([15.0, 2.5, 0.25, 0.9])
    lo1, hi1 = np.array([10.0, 1.0, 0.1, 0.6]), np.array([11.0, 1.2, 0.3, 0.8])
    distrs = [list(np.stack([lo, hi], 1).reshape(-1)) for lo, hi in ((lo0, hi0), (lo1, hi1))]
    xi = data.sample_candidates("uniform", distrs, num_samples=512, seed=9).cpu().numpy()
    u = (xi[0] - lo0) / (hi0 - lo0)
    assert 0.0 <= u.min() and u.max() < 1.0 and 0.4 < u.mean() < 0.6
    assert np.allclose(xi[1], lo1 + (hi1 - lo1) * u, rtol=1e-12, atol=0)
    sampler = random_envs.TaskSampler("RandomCartPole-v0")                 # = what sample_tasks would draw
    sampler.set_dr_distribution("uniform", distrs[1])
    sampler.seed_dr(9)
    assert np.array_equal(sampler.sample_tasks(512), xi[1])
    with pytest.raises(Exception, match=GAUSSIAN_FAIL_MSG):                # every draw of dim 0 below 0.1
        data.dr_log_likelihood("gaussian", [[9.8, 1.0, 1.0, 0.1, 0.2, 0.02, 0.5, 0.05],
                                            [-5.0, 0.1, 1.0, 0.1, 0.2, 0.02, 0.5, 0.05]], num_samples=64)


def test_the_generating_task_scores_highest():
    obs, act, nxt, starts = _record(64, 140, True, seed=21)
    assert 7000 <= len(obs) <= 9000
    data = random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    mean = np.array(XI_TRUE)
    centres = [mean]
    for d in range(4):
        for f in (0.8, 1.2):
            m = mean.copy(); m[d] *= f
            centres.append(m)
    distrs = [list(np.stack([m, 0.02 * m], 1).reshape(-1)) for m in centres]
    total = data.dr_log_likelihood("truncnorm", distrs, num_samples=256, seed=4, epsilon=EPS).cpu().numpy()
    assert np.all(np.isfinite(total))
    margins = total[0] - total[1:]
    assert np.all(margins > 0), margins
