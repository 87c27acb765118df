"""Offline DR log-likelihood at the kernel's edges, against the exact-moment reference (oracle.transition_loglik with
exact=True): windows past the 64-step action mask, large angles at lam = 1 (both sides of the small-angle branch and
the full-range sincos), sample counts around the 256-sample xi chunks with an outlying shift sample, bitwise
independence of window placement and W, far-off states (the shifted sums), the compensated totals against the Sum2
error bound, non-physical samples, and the same bits on a second GPU."""
import ctypes
import math

import numpy as np
import pytest
import torch

import random_envs_b200 as random_envs
from oracle import cartpole_port as port, transition_loglik as oracle
from random_envs_b200 import _device, _lib

pytestmark = pytest.mark.gpu

XI_TRUE = (12.0, 1.5, 0.2, 0.7)
XI_BENIGN = (2.5, 1.0, 0.1, 1.0)              # slow unstable mode (~e^{1.3 t}): ulp differences stay ulp-sized
LOWER = np.array([2.0, 0.5, 0.05, 0.1])      # cart-pole search box (tests/test_gpu_transition_loglik.py)
UPPER = np.array([20.0, 3.0, 0.3, 1.0])
U = 2.0 ** -53


def _check(got, ref, what=""):
    """|l_kernel - l_ref| <= 1e-9 max(1, |l_ref|) per window (the suite's tolerance)."""
    got, ref = np.asarray(got), np.asarray(ref)
    assert np.all(np.isfinite(ref)) and got.shape == ref.shape, what
    tol = 1e-9 * np.maximum(1.0, np.abs(ref))
    err = np.abs(got - ref)
    assert np.all(err <= tol), (what, float(err.max()), float(np.max(err / tol)))


def _episode(T, xi, euler, seed, sigma):
    """T transitions of one episode under a linear balancing controller (bang-bang on theta + 0.5 theta_dot +
    0.05 x + 0.1 x_dot), simulated with cartpole_port.dynamics_step; obs[t + 1] = next_obs[t] = true state + noise."""
    rs = np.random.RandomState(seed)
    s = (0.02, -0.05, 0.03, 0.01)
    states, act = [s], []
    for _ in range(T):
        x, xd, th, thd = s
        a = int(th + 0.5 * thd + 0.05 * x + 0.1 * xd > 0)
        s, _ = port.dynamics_step(s, xi, a, euler)
        states.append(s)
        act.append(a)
    noisy = np.array(states) + rs.normal(0.0, sigma, (T + 1, 4))
    return noisy[:-1].copy(), np.array(act, np.uint8), noisy[1:].copy()


def _candidates(centres, M, spread, seed):
    """(C, M, 4) samples uniform in centre * (1 +- spread); common random numbers across the candidates."""
    u = np.random.RandomState(seed).uniform(-1.0, 1.0, (M, 4))
    return np.stack([np.asarray(c, np.float64) * (1.0 + spread * u) for c in centres])


def _cuda(a, dtype=torch.float64, device="cuda"):
    return torch.as_tensor(np.ascontiguousarray(a), dtype=dtype).to(device)


def _raw(obs, act, nxt, windows, xi, lam, euler, eps):
    """renv_cartpole_transition_loglik_f64 on arbitrary int32 window starts (device tensors): (total, ll) on the host."""
    win = _cuda(np.asarray(windows, np.int32), torch.int32, obs.device)
    xi = xi.contiguous()
    C, M = xi.shape[0], xi.shape[1]
    d = _lib.Transitions()
    d.obs, d.next_obs, d.action, d.window = obs.data_ptr(), nxt.data_ptr(), act.data_ptr(), win.data_ptr()
    d.T, d.W = obs.shape[0], win.numel()
    ll = torch.empty((C, d.W), dtype=torch.float64, device=obs.device)
    total = torch.empty(C, dtype=torch.float64, device=obs.device)
    with torch.cuda.device(obs.device):
        rc = _lib.load().renv_cartpole_transition_loglik_f64(
            ctypes.byref(d), lam, _lib.EULER if euler else _lib.SEMI_IMPLICIT, _device.ptr(xi), C, M,
            (ctypes.c_double * 4)(*np.broadcast_to(np.asarray(eps, np.float64), (4,))), _device.ptr(ll),
            _device.ptr(total), _device.stream_ptr(obs.device))
        assert rc == 0, rc
        torch.cuda.synchronize()
    return total.cpu().numpy(), ll.cpu().numpy()


def _subset(n, k):
    """At most k indices spread evenly over range(n), first and last included."""
    return np.unique(np.linspace(0, n - 1, min(n, k)).round().astype(int))


# ---------------------------------------------------------------- 1. windows past the 64-step action mask
@pytest.fixture(scope="module")
def long_episode():
    return {euler: _episode(200, XI_BENIGN, euler, seed=5 + euler, sigma=1e-3) for euler in (True, False)}


@pytest.mark.parametrize("euler", [True, False])
@pytest.mark.parametrize("lam", [63, 64, 65, 130])
def test_windows_past_the_action_mask(long_episode, euler, lam):
    obs, act, nxt = long_episode[euler]
    assert 40 <= act.sum() <= 160 and np.count_nonzero(np.diff(act.astype(int))) >= 20     # the actions vary
    data = random_envs.TransitionDataset(obs, act, nxt)
    xi = _candidates([XI_BENIGN, 0.93 * np.array(XI_BENIGN), 1.07 * np.array(XI_BENIGN)], 32, 0.1, seed=1)
    total, ll = data.log_likelihood(_cuda(xi), lam=lam, epsilon=2e-6, kinematics_integrator="euler" if euler else
                                    "semi-implicit", per_window=True)
    windows = data.window_starts(lam)
    assert len(windows) == 201 - lam
    pick = _subset(len(windows), 12)
    # A 1-ulp difference of sin / cos (the kernel's polynomial or CUDA's sincos against glibc) grows with the
    # unstable mode, about e^{1.3 * 0.02 * 130} ~ 30x at lam = 130 -- still ~1e-14 relative to a state whose spread
    # over the +-10 % candidates is many orders larger, so the shared tolerance holds as is.
    ref, _ = oracle.loglik(obs, act, nxt, windows[pick], xi, lam, 2e-6, euler, exact=True)
    _check(ll.cpu().numpy()[:, pick], ref, (euler, lam))


# ---------------------------------------------------------------- 2. large angles at lam = 1
LARGE_THETA = [0.25, float(np.nextafter(0.25, 1.0)), -0.25, 0.3, 3.0, -3.0, 1e3, 2e5, 1e9]


@pytest.mark.parametrize("euler", [True, False])
def test_large_angles_at_lam_1(euler):
    # windows alternate large / small start angles, so the 8 lane groups of a warp take both branches
    rows = []
    for k, th in enumerate(LARGE_THETA):
        rows.append((0.1, -0.2, th, 0.3))
        rows.append((-0.05, 0.1, 0.01 * (k + 1) * (-1) ** k, -0.2))
    obs = np.array(rows)
    rs = np.random.RandomState(2)
    act = rs.randint(0, 2, len(obs)).astype(np.uint8)
    nxt = np.array([port.dynamics_step(tuple(o), XI_TRUE, int(a), euler)[0] for o, a in zip(obs, act)])
    nxt += rs.normal(0.0, 1e-3, nxt.shape)
    xi = _candidates([XI_TRUE, 1.1 * np.array(XI_TRUE)], 64, 0.05, seed=3)
    data = random_envs.TransitionDataset(obs, act, nxt)
    total, ll = data.log_likelihood(_cuda(xi), lam=1, epsilon=1e-6,
                                    kinematics_integrator="euler" if euler else "semi-implicit", per_window=True)
    ref, _ = oracle.loglik(obs, act, nxt, np.arange(len(obs)), xi, 1, 1e-6, euler, exact=True)
    _check(ll.cpu().numpy(), ref, euler)


# ---------------------------------------------------------------- 3. sample counts around the xi chunks
@pytest.fixture(scope="module")
def short_episode():
    return {euler: _episode(60, XI_TRUE, euler, seed=7 + euler, sigma=1e-2) for euler in (True, False)}


@pytest.mark.parametrize("M", [2, 3, 255, 256, 257, 511, 513, 1000])
def test_sample_counts_around_the_chunks(short_episode, M):
    euler = M % 2 == 1
    obs, act, nxt = short_episode[euler]
    data = random_envs.TransitionDataset(obs, act, nxt)
    xi = _candidates([XI_TRUE, XI_TRUE], M, 0.05, seed=M)
    xi[1, 0] = UPPER if M % 3 else LOWER      # candidate 1: sample 0 (the shift) at a corner of the search box
    lam, eps = 2, [1e-4, 3e-4, 2e-4, 4e-4]
    total, ll = data.log_likelihood(_cuda(xi), lam=lam, epsilon=eps,
                                    kinematics_integrator="euler" if euler else "semi-implicit", per_window=True)
    windows = data.window_starts(lam)
    pick = _subset(len(windows), 10)
    ref, _ = oracle.loglik(obs, act, nxt, windows[pick], xi, lam, eps, euler, exact=True)
    _check(ll.cpu().numpy()[:, pick], ref, M)


# ---------------------------------------------------------------- 4. window placement and W
def test_window_placement_and_count_do_not_change_the_bits(long_episode):
    obs, act, nxt = long_episode[True]
    lam, eps, T = 3, 2e-6, len(obs)
    dev = [_cuda(obs), _cuda(act, torch.uint8), _cuda(nxt)]
    xi = _candidates([XI_BENIGN, 0.9 * np.array(XI_BENIGN)], 40, 0.1, seed=4)
    xt = _cuda(xi)
    rs = np.random.RandomState(8)
    valid = np.arange(T - lam + 1)
    big = rs.permutation(np.tile(valid, 12289 // len(valid) + 1))[:12289]        # >= 10^4, every start repeated
    assert set(big) == set(valid)
    calls = [big, rs.permutation(valid)] + [rs.choice(valid, W) for W in (63, 64, 65, 257)]  # duplicates
    calls.append(np.concatenate([big[:64], big[:64][::-1]]))
    seen = {}
    for windows in calls:
        _, ll = _raw(*dev, windows, xt, lam, True, eps)
        for pos, t in enumerate(windows):
            v = ll[:, pos]
            if t in seen:
                assert np.array_equal(v.view(np.int64), seen[t].view(np.int64)), (len(windows), pos, t)
            else:
                seen[t] = v.copy()
    for t in valid[::17]:                                                           # alone: W = 1
        _, ll = _raw(*dev, [t], xt, lam, True, eps)
        assert np.array_equal(ll[:, 0].view(np.int64), seen[t].view(np.int64)), t
    pick = big[_subset(len(big), 16)]
    ref, _ = oracle.loglik(obs, act, nxt, pick, xi, lam, eps, True, exact=True)
    _check(np.stack([seen[t] for t in pick], 1), ref)


# ---------------------------------------------------------------- 5. far-off states
def _offset_data(comp, offset, lam, seed):
    """A small-angle episode with state component comp moved by offset.  x does not enter the dynamics, so for
    comp = 0 the recorded data are translated as a whole; theta_dot does, so for comp = 3 next_obs[u] is the
    prediction from obs[u - lam + 1] at the true task plus noise of the size of the candidates' spread."""
    obs, act, nxt = _episode(40, XI_TRUE, False, seed=seed, sigma=1e-5)
    obs[:, comp] += offset
    if comp == 0:
        nxt[:, 0] += offset
    else:
        rs = np.random.RandomState(seed)
        for u in range(lam - 1, len(obs)):
            p = oracle.predict(obs, act, u - lam + 1, lam, np.array([XI_TRUE]), False)[0]
            nxt[u] = p * (1.0 + 1e-3 * rs.normal(size=4))
    return obs, act, nxt


@pytest.mark.parametrize("lam", [2, 5])
@pytest.mark.parametrize("offset", [1e2, 1e4, 1e6])
def test_far_off_x(lam, offset):
    # The spread of x comes from x_dot (~1e-4 here) while x sits at 1e6: the float64 two-pass covariance of the
    # oracle loses ~3e-8 relative at 1e6, a naive E[ss'] - E[s]E[s]' far more; the kernel's sums shifted by the
    # prediction under sample 0 must meet the tolerance against the exact moments.
    obs, act, nxt = _offset_data(0, offset, lam, seed=11)
    data = random_envs.TransitionDataset(obs, act, nxt)
    xi = _candidates([XI_TRUE, 1.05 * np.array(XI_TRUE)], 300, 0.05, seed=12)
    total, ll = data.log_likelihood(_cuda(xi), lam=lam, epsilon=1e-8, kinematics_integrator="semi-implicit",
                                    per_window=True)
    windows = data.window_starts(lam)
    pick = _subset(len(windows), 8)
    ref, _ = oracle.loglik(obs, act, nxt, windows[pick], xi, lam, 1e-8, False, exact=True)
    _check(ll.cpu().numpy()[:, pick], ref, (lam, offset))
    print("x offset %g, lam %d: max relative error %.2g"
          % (offset, lam, np.max(np.abs(ll.cpu().numpy()[:, pick] - ref) / np.maximum(1.0, np.abs(ref)))))


@pytest.mark.parametrize("lam", [2, 5])
@pytest.mark.parametrize("offset", [1e2, 1e4, 1e6])
def test_far_off_theta_dot(lam, offset):
    # theta_dot enters the dynamics squared, so the spread grows with the offset and the predicted covariance becomes
    # nearly rank one: kappa(S) ~ 1e6 at 1e2, 1e9 - 1e11 at 1e4, > 1e14 at 1e6.  A float64 Cholesky factorisation --
    # the kernel's and the reference's alike -- and the 1-ulp differences of sin / cos then move l by about
    # kappa(S) u relative (1-ulp sin / cos perturbations of the oracle move the exact reference by 1e-5 at 1e4,
    # lam = 5, and 8e-5 at 1e6, lam = 2).  First order, a relative perturbation e of S (<= M u for sums of M terms)
    # changes l by <= kappa(S) e (r'S^-1 r / 2 + 2); that bound is asserted per window on top of the shared
    # tolerance.  It vanishes at 1e2 (B200 error 8e-13 relative; 1e-6 and 2e-5 at 1e4, 9e-9 at 1e6 with lam = 2).
    # Where S is numerically singular (kappa u > 1e-3) the float64 reference may itself fail the factorisation; the
    # kernel must then still give -inf or a number, never NaN.
    M, eps = 300, 1e-8
    obs, act, nxt = _offset_data(3, offset, lam, seed=13)
    data = random_envs.TransitionDataset(obs, act, nxt)
    xi = _candidates([XI_TRUE, 1.05 * np.array(XI_TRUE)], M, 0.05, seed=14)
    total, ll = data.log_likelihood(_cuda(xi), lam=lam, epsilon=eps, kinematics_integrator="semi-implicit",
                                    per_window=True)
    windows = data.window_starts(lam)
    pick = _subset(len(windows), 8)
    ref, _ = oracle.loglik(obs, act, nxt, windows[pick], xi, lam, eps, False, exact=True)
    got = ll.cpu().numpy()[:, pick]
    worst = 0.0
    for c in range(2):
        for k, t in enumerate(windows[pick]):
            _, Sigma, r = oracle.exact_fit(nxt[t + lam - 1], oracle.predict(obs, act, int(t), lam, xi[c], False))
            S = Sigma + eps * np.eye(4)
            kappa = np.linalg.cond(S)
            if kappa * U > 1e-3:
                assert not math.isnan(got[c, k]), (c, t)
                continue
            quad = float(r @ np.linalg.solve(S, r))
            tol = 1e-9 * max(1.0, abs(ref[c, k])) + kappa * M * U * (quad / 2 + 2)
            assert abs(got[c, k] - ref[c, k]) <= tol, (c, t, got[c, k], ref[c, k], kappa, tol)
            worst = max(worst, abs(got[c, k] - ref[c, k]) / max(1.0, abs(ref[c, k])))
    if offset == 1e2:
        assert worst <= 1e-9, worst
    print("theta_dot offset %g, lam %d: max relative error %.2g" % (offset, lam, worst))


# ---------------------------------------------------------------- 6. compensated totals
def _plain_sum_in_kernel_order(v, threads=256):
    """loglik_total_kernel's order without compensation: thread i sums w = i, i + 256, ... then the fixed tree."""
    part = np.zeros(threads)
    for k in range(0, len(v), threads):
        chunk = v[k:k + threads]
        part[:len(chunk)] += chunk
    half = threads // 2
    while half:
        part[:half] += part[half:2 * half]
        half //= 2
    return float(part[0])


def test_compensated_totals_meet_the_sum2_bound():
    rs = np.random.RandomState(21)
    n_near, far = 60, [(1.0, 0.0, 0.0, 0.0), (0.0, 0.0, 1.2, 0.0), (0.8, 0.0, 0.5, 0.0), (1.1, 0.0, 0.0, 0.2)]
    obs = np.column_stack([rs.uniform(-0.5, 0.5, n_near + len(far) + 1), rs.uniform(-0.5, 0.5, n_near + len(far) + 1),
                           rs.uniform(-0.1, 0.1, n_near + len(far) + 1), rs.uniform(-0.5, 0.5, n_near + len(far) + 1)])
    act = rs.randint(0, 2, len(obs)).astype(np.uint8)
    nxt = np.array([port.dynamics_step(tuple(o), XI_TRUE, int(a), True)[0] for o, a in zip(obs, act)])
    nxt[:n_near] += rs.normal(0.0, 3e-4, (n_near, 4))
    nxt[n_near:n_near + len(far)] += np.array(far)                   # ~1 from the prediction: l ~ -1e6 at eps 1e-6
    t_nan = len(obs) - 1
    obs[t_nan, 1] = math.nan                                         # its window gives -inf (raw ABI only)
    dev = [_cuda(obs), _cuda(act, torch.uint8), _cuda(nxt)]
    xi = _cuda(_candidates([XI_TRUE], 16, 0.05, seed=22))
    eps = 1e-6
    _, base = _raw(*dev, np.arange(len(obs)), xi, 1, True, eps)
    base = base[0]
    assert np.all((base[:n_near] > 10) & (base[:n_near] < 40)), base[:n_near]
    assert np.all(base[n_near:t_nan] < -3e5) and base[t_nan] == -math.inf

    # every far window once, then near windows until the running sum comes back to ~0
    windows, s = list(range(n_near, n_near + len(far))), math.fsum(base[n_near:n_near + len(far)])
    near = rs.permutation(np.tile(np.arange(n_near), 5000))
    for t in near:
        if s + base[t] > 0:
            break
        windows.append(int(t)); s += base[t]
    best = min(range(n_near), key=lambda t: abs(s + base[t]))        # the last window: the smallest residual
    windows.append(best)
    windows = rs.permutation(np.array(windows, np.int32))
    W = len(windows)
    assert 80000 <= W <= 150000, W

    total, ll = _raw(*dev, windows, xi, 1, True, eps)
    v = ll[0]
    assert np.array_equal(v, base[windows])
    exact = math.fsum(v)
    mag = math.fsum(np.abs(v))
    assert mag / abs(exact) >= 1e5, (mag, exact)
    # Sum2 (Ogita, Rump, Oishi 2005): |res - s| <= u |s| + gamma_{n-1}^2 sum |p_i|, gamma_n = n u / (1 - n u)
    bound = 2 * math.ulp(exact) + (W * U) ** 2 * mag
    assert abs(total[0] - exact) <= bound, (total[0], exact, bound)
    plain = _plain_sum_in_kernel_order(v)
    assert abs(plain - exact) > bound, (plain, exact, bound)        # the test is sharp: a plain sum fails it

    # non-finite values pass through the totals at any thread position: -inf alone -> -inf, with NaN -> NaN
    for p in (0, 255, 256, W - 1):
        win = windows.copy()
        win[p] = t_nan
        total, _ = _raw(*dev, win, xi, 1, True, eps)
        assert total[0] == -math.inf, p
        for q in (0, 255, 256, W - 1):
            if q != p:
                win2 = win.copy()
                win2[q] = -1                                         # out of range: NaN
                total, ll = _raw(*dev, win2, xi, 1, True, eps)
                assert ll[0, p] == -math.inf and math.isnan(ll[0, q]) and math.isnan(total[0]), (p, q)


# ---------------------------------------------------------------- 7. non-physical samples
@pytest.mark.parametrize("euler", [True, False])
@pytest.mark.parametrize("lam", [1, 3])
def test_non_physical_samples_give_minus_inf(short_episode, euler, lam):
    obs, act, nxt = short_episode[euler]
    data = random_envs.TransitionDataset(obs, act, nxt)
    M = 64
    xi = np.repeat(_candidates([XI_TRUE], M, 0.05, seed=31), 7, axis=0)
    xi[1, 0, 3] = 0.0                                    # pole_length = 0 at the shift sample
    xi[2, M - 1, 3] = 0.0                                # ... at the last sample
    xi[3, 17, 1] = -xi[3, 17, 2]                         # cart_mass = -pole_mass: zero total mass
    xi[4, 0, 1] = -xi[4, 0, 2]
    xi[5, 40, 0] = math.nan                              # a NaN field
    xi[6, 0, 2] = math.nan
    integ = "euler" if euler else "semi-implicit"
    total, ll = data.log_likelihood(_cuda(xi), lam=lam, epsilon=1e-4, kinematics_integrator=integ, per_window=True)
    total, ll = total.cpu().numpy(), ll.cpu().numpy()
    assert np.all(ll[1:] == -math.inf), [(c, ll[c][~(ll[c] == -math.inf)][:4]) for c in range(1, 7)]
    assert np.all(total[1:] == -math.inf), total
    t0, l0 = data.log_likelihood(_cuda(xi[:1]), lam=lam, epsilon=1e-4, kinematics_integrator=integ, per_window=True)
    assert np.all(np.isfinite(l0.cpu().numpy()))
    assert np.array_equal(ll[0], l0.cpu().numpy()[0]) and total[0] == t0.cpu().numpy()[0]


# ---------------------------------------------------------------- 8. a second GPU
def test_a_second_gpu_gives_the_same_bits(long_episode):
    if torch.cuda.device_count() < 2:
        pytest.skip("one CUDA device visible: no second GPU to compare with")
    obs, act, nxt = long_episode[False]
    xi = _candidates([XI_BENIGN, 0.9 * np.array(XI_BENIGN)], 300, 0.1, seed=41)
    out = []
    for dev in ("cuda:0", "cuda:1"):
        data = random_envs.TransitionDataset(obs, act, nxt, device=dev)
        for lam in (1, 70):
            t, l = data.log_likelihood(_cuda(xi, device=dev), lam=lam, epsilon=2e-6, kinematics_integrator="semi",
                                       per_window=True)
            out.append((t.cpu().numpy(), l.cpu().numpy()))
    for a, b in zip(out[:2], out[2:]):
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])
