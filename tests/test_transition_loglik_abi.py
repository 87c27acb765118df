"""Offline DR log-likelihood without a GPU: argument validation of renv_cartpole_transition_loglik_f64, the ctypes struct
against the C compiler's layout, the compiled form of its kernels, the host-side rejections and window construction of
TransitionDataset, and the float64 oracle against scipy (and, where the reference is mounted, against it)."""
import ctypes
import math
import os
import re
import sys

import numpy as np
import pytest
import torch

import random_envs_b200 as random_envs
from abi_support import ROOT, gcc_layout, ptxas_blocks
from oracle import cartpole_port as port, reference_loader as rl, transition_loglik as oracle
from random_envs_b200 import _device, _lib, build as lib_build

sys.path.insert(0, os.path.join(ROOT, "profiles"))
import sass_stats  # noqa: E402


def _data(**kw):
    d = _lib.Transitions()
    d.obs, d.next_obs, d.action, d.window, d.T, d.W = 4096, 8192, 12288, 16384, 100, 10
    for k, v in kw.items():
        setattr(d, k, v)
    return d


def _rc(data="ok", lam=1, integrator=0, xi=20480, C=3, M=16, eps=(1e-4, 1e-4, 1e-4, 1e-4), loglik=24576, total=28672):
    lib = _lib.load()
    data = _data() if data == "ok" else data
    e = (ctypes.c_double * 4)(*eps) if eps is not None else None
    return lib.renv_cartpole_transition_loglik_f64(ctypes.byref(data) if data is not None else None, lam, integrator, xi,
                                                   C, M, e, loglik, total, None)


def test_transition_loglik_validates_arguments_before_any_cuda_call():
    # every call below fails validation, so none of the fake device pointers is ever touched
    assert _rc(data=None) == -1
    for f in ("obs", "next_obs", "action", "window"):
        assert _rc(data=_data(**{f: None})) == -1, f
    for k in ("xi", "eps", "loglik", "total"):
        assert _rc(**{k: None}) == -1, k
    for f, v in (("obs", 4104), ("next_obs", 8200), ("window", 16386)):
        assert _rc(data=_data(**{f: v})) == -2, f
    assert _rc(data=_data(action=12289), lam=0) == -3                   # actions are bytes: any address is aligned
    assert _rc(xi=20488) == -2
    assert _rc(loglik=24580) == -2 and _rc(total=28676) == -2
    for bad in (dict(data=_data(T=0)), dict(data=_data(W=0)), dict(data=_data(W=-1)), dict(C=0), dict(M=1), dict(M=0),
                dict(lam=0), dict(lam=101)):
        assert _rc(**bad) == -3, bad
    assert _rc(lam=100, integrator=2) == -6                             # lam == T is allowed
    assert _rc(integrator=-1) == -6
    for e in ((-1e-9, 0, 0, 0), (0, 0, 0, math.nan), (0, math.inf, 0, 0), (0, 0, -math.inf, 0)):
        assert _rc(eps=e) == -7, e
    assert _rc(eps=(0, 0, 0, 0), integrator=3) == -6                    # eps = 0 is valid


def test_transitions_struct_matches_the_header(tmp_path):
    fields = [f for f, _ in _lib.Transitions._fields_]
    got = gcc_layout(tmp_path, "renv_transitions", fields)
    for f in fields:
        assert int(got[f]) == getattr(_lib.Transitions, f).offset, f
    assert int(got["sizeof"]) == ctypes.sizeof(_lib.Transitions)
    restype, argtypes = _lib.SIGNATURES["renv_cartpole_transition_loglik_f64"]
    assert restype is ctypes.c_int and len(argtypes) == 10
    assert argtypes[0] is ctypes.POINTER(_lib.Transitions) and argtypes[6] is ctypes.POINTER(ctypes.c_double)
    assert _lib.load().renv_cartpole_transition_loglik_f64.argtypes == argtypes


def test_loglik_kernel_runs_dynamics_on_dfma_without_philox_spills_or_local_memory():
    lib_build.build()
    sass = sass_stats.functions(lib_build.LIB_PATH)
    names = [n for n in sass if "cartpole_transition_loglik_kernel" in n]
    assert len(names) == 2, names                                      # Euler and semi-implicit
    philox = ("-0x2daee0ad", "-0x326172a9")                             # the Philox4x32 multipliers as SASS immediates
    assert any(p in o.lower() for n in sass if "dr_sample_kernel" in n for _, _, o in sass[n] for p in philox)
    blocks = ptxas_blocks()
    for name in names + [n for n in sass if "loglik_total_kernel" in n]:
        rows = sass[name]
        assert not any(p in o.lower() for _, _, o in rows for p in philox), name     # no xi is drawn here
        b = blocks[name]
        assert re.search(r"0 bytes spill stores, 0 bytes spill loads", b), name
        # local memory only in the out-of-line frame of the full-range sincos (|theta| > 0.25), after the last EXIT
        last_exit = max(a for a, op, _ in rows if op == "EXIT")
        assert all(a > last_exit for a, op, _ in rows if op.startswith(("LDL", "STL"))), name
        assert int(re.search(r"(\d+) bytes stack frame", b).group(1)) <= 40, name
    for name in names:
        ops = [op for _, op, _ in sass[name]]
        assert sum(o.startswith("DFMA") for o in ops) > 200, name
        assert any(o.startswith("MUFU.RCP64H") for o in ops), name    # the correctly rounded 1 / total_mass


# ---------------------------------------------------------------- host side
@pytest.fixture
def cpu_device(monkeypatch):
    """Let TransitionDataset keep its tensors on the CPU: nothing here launches a kernel."""
    monkeypatch.setattr(_device, "require_cuda", lambda device=None: torch.device("cpu"))


def _arrays(T=12, seed=0):
    rs = np.random.RandomState(seed)
    return rs.uniform(-0.05, 0.05, (T, 4)), rs.randint(0, 2, T).astype(np.uint8), rs.uniform(-0.05, 0.05, (T, 4))


def test_transition_dataset_host_side_rejections(cpu_device):
    obs, act, nxt = _arrays()
    with pytest.raises(ValueError, match="shape"):
        random_envs.TransitionDataset(obs[:, :3], act, nxt[:, :3])
    with pytest.raises(ValueError, match="shape"):
        random_envs.TransitionDataset(obs, act, nxt[:-1])
    with pytest.raises(ValueError, match="shape"):
        random_envs.TransitionDataset(obs, act[:-1], nxt)
    with pytest.raises(ValueError, match="shape"):
        random_envs.TransitionDataset(obs[:0], act[:0], nxt[:0])
    for bad in (math.nan, math.inf):
        o = obs.copy(); o[3, 1] = bad
        with pytest.raises(ValueError, match="finite"):
            random_envs.TransitionDataset(o, act, nxt)
        with pytest.raises(ValueError, match="finite"):
            random_envs.TransitionDataset(obs, act, o)
    a = act.astype(np.int64); a[5] = 2
    with pytest.raises(AssertionError, match=r"^2 \(<class 'int'>\) invalid$"):
        random_envs.TransitionDataset(obs, a, nxt)
    with pytest.raises(AssertionError, match="invalid"):
        random_envs.TransitionDataset(obs, np.full(12, 0.5), nxt)
    for starts in ([12], [-1], [1.5]):
        with pytest.raises(ValueError, match="episode_starts"):
            random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    with pytest.raises(ValueError, match="mask"):
        random_envs.TransitionDataset(obs, act, nxt, episode_starts=np.zeros(5, bool))
    data = random_envs.TransitionDataset(torch.as_tensor(obs), torch.as_tensor(act), torch.as_tensor(nxt))
    assert data.obs.dtype == torch.float64 and data.actions.dtype == torch.uint8 and data.num_transitions == 12
    xi = torch.tensor(port.NOMINAL_TASK, dtype=torch.float64).repeat(4, 1)
    for kw, match in ((dict(xi=xi.float()), "float64"), (dict(xi=xi[:1]), "M >= 2"), (dict(xi=xi[:, :3]), "shape"),
                      (dict(xi=xi.reshape(1, 1, 4, 4)), "shape"), (dict(xi=xi, lam=0), "lam"), (dict(xi=xi, lam=13), "lam"),
                      (dict(xi=xi, epsilon=-1e-3), "epsilon"), (dict(xi=xi, epsilon=[1e-4] * 3), "epsilon"),
                      (dict(xi=xi, epsilon=[0, 0, math.nan, 0]), "epsilon")):
        with pytest.raises(ValueError, match=match):
            data.log_likelihood(**kw)
    split = random_envs.TransitionDataset(obs, act, nxt, episode_starts=list(range(12)))
    with pytest.raises(ValueError, match="no window"):
        split.log_likelihood(xi, lam=2)
    with pytest.raises(ValueError, match="at least one"):
        data.sample_candidates("uniform", [])
    with pytest.raises(ValueError, match="num_samples"):
        data.sample_candidates("uniform", [[1, 2] * 4], num_samples=1)


@pytest.mark.parametrize("lam", [1, 3])
def test_windows_stay_inside_episodes(cpu_device, lam):
    obs, act, nxt = _arrays(20)
    starts = [0, 4, 5, 11, 18]
    data = random_envs.TransitionDataset(obs, act, nxt, episode_starts=starts)
    expect = oracle.window_starts(20, lam, starts)
    assert np.array_equal(data.window_starts(lam), expect) and data.num_windows(lam) == len(expect)
    if lam == 1:
        assert np.array_equal(expect, np.arange(20))                    # one transition never crosses a start
    else:                                                                # episodes [0,4) [4,5) [5,11) [11,18) [18,20)
        assert expect.tolist() == [0, 1, 5, 6, 7, 8, 11, 12, 13, 14, 15]
    mask = np.zeros(20, bool); mask[starts] = True
    assert np.array_equal(random_envs.TransitionDataset(obs, act, nxt, episode_starts=mask).window_starts(lam), expect)
    assert np.array_equal(random_envs.TransitionDataset(obs, act, nxt).window_starts(lam), np.arange(20 - lam + 1))


# ---------------------------------------------------------------- the oracle
def test_oracle_matches_scipy_multivariate_normal():
    stats = pytest.importorskip("scipy.stats")
    rs = np.random.RandomState(3)
    obs = rs.uniform(-0.1, 0.1, (30, 4))
    act = rs.randint(0, 2, 30)
    nxt = obs + rs.normal(0, 0.01, (30, 4))
    lo, hi = np.array([5.0, 0.5, 0.05, 0.3]), np.array([15.0, 2.0, 0.3, 1.0])
    xi = lo + (hi - lo) * rs.uniform(size=(2, 40, 4))
    eps = np.array([1e-4, 2e-4, 3e-4, 4e-4])
    for euler, lam in ((True, 1), (False, 1), (True, 3), (False, 4)):
        windows = oracle.window_starts(30, lam)
        ll, total = oracle.loglik(obs, act, nxt, windows, xi, lam, eps, euler)
        for c in range(2):
            for w, t in enumerate(windows[:6]):
                pred = oracle.predict(obs, act, int(t), lam, xi[c], euler)
                ref = stats.multivariate_normal.logpdf(nxt[t + lam - 1], pred.mean(0), np.cov(pred.T) + np.diag(eps))
                assert abs(ll[c, w] - ref) <= 1e-10 * max(1.0, abs(ref)), (euler, lam, c, w)
            assert total[c] == math.fsum(ll[c])
    # Euler, lam = 1: x and theta of the prediction do not depend on xi -- singular without eps
    ll, _ = oracle.loglik(obs, act, nxt, [0, 1], xi, 1, 0.0, True)
    assert np.all(ll == -np.inf)
    ll, total = oracle.loglik(obs, act, nxt, [0, 29, 30, -1], xi[:1], 1, eps, True)
    assert np.isfinite(ll[0, :2]).all() and np.isnan(ll[0, 2:]).all() and np.isnan(total[0])


def _fraction_logpdf(y, pred, eps):
    """The whole objective in rational arithmetic from the float64 predictions: mu, Sigma, S = Sigma + diag(eps),
    r' S^-1 r and det S exact (Gaussian elimination); only the final quad form and log det are rounded."""
    from fractions import Fraction
    M = len(pred)
    P = [[Fraction(float(v)) for v in row] for row in pred]
    mu = [sum(row[i] for row in P) / M for i in range(4)]
    A = [[sum((row[i] - mu[i]) * (row[j] - mu[j]) for row in P) / (M - 1) + (Fraction(float(eps[i])) if i == j else 0)
          for j in range(4)] + [Fraction(float(y[i])) - mu[i]] for i in range(4)]
    r = [A[i][4] for i in range(4)]
    det = Fraction(1)
    for k in range(4):
        det *= A[k][k]
        for i in range(k + 1, 4):
            f = A[i][k] / A[k][k]
            for j in range(k, 5):
                A[i][j] -= f * A[k][j]
    z = [Fraction(0)] * 4
    for i in reversed(range(4)):
        z[i] = (A[i][4] - sum(A[i][j] * z[j] for j in range(i + 1, 4))) / A[i][i]
    quad = sum(r[i] * z[i] for i in range(4))
    return -0.5 * float(quad) - 0.5 * (math.log(det.numerator) - math.log(det.denominator)) - 2.0 * oracle.LOG_2PI


def test_exact_oracle_matches_scipy_and_keeps_its_accuracy_far_from_the_origin():
    stats = pytest.importorskip("scipy.stats")
    rs = np.random.RandomState(4)
    obs = rs.uniform(-0.1, 0.1, (20, 4))
    act = rs.randint(0, 2, 20)
    nxt = obs + rs.normal(0, 0.01, (20, 4))
    xi = np.array([5.0, 0.5, 0.05, 0.3]) + np.array([10.0, 1.5, 0.25, 0.7]) * rs.uniform(size=(2, 40, 4))
    eps = np.array([1e-4, 2e-4, 3e-4, 4e-4])
    for euler, lam in ((True, 1), (False, 1), (True, 3), (False, 4)):
        windows = oracle.window_starts(20, lam)[:6]
        ll, total = oracle.loglik(obs, act, nxt, windows, xi, lam, eps, euler, exact=True)
        for c in range(2):
            for w, t in enumerate(windows):
                pred = oracle.predict(obs, act, int(t), lam, xi[c], euler)
                ref = stats.multivariate_normal.logpdf(nxt[t + lam - 1], pred.mean(0), np.cov(pred.T) + np.diag(eps))
                assert abs(ll[c, w] - ref) <= 1e-12 * max(1.0, abs(ref)), (euler, lam, c, w)
            assert total[c] == math.fsum(ll[c])
    assert np.all(oracle.loglik(obs, act, nxt, [0, 1], xi, 1, 0.0, True, exact=True)[0] == -np.inf)

    # x = 1e6 with a spread of ~1e-4 (x does not enter the dynamics; the spread comes from x_dot): the exact moments
    # keep l within 1e-13 of the rational value, np.cov's float64 moments do not
    xi = np.array([12.0, 1.5, 0.2, 0.7]) * (1.0 + 0.05 * rs.uniform(-1.0, 1.0, (300, 4)))
    start = np.array([[1e6 + 0.01, 0.05, 0.02, -0.1]] * 2)
    pred = oracle.predict(start, [1, 0], 0, 2, xi, False)
    y = pred.mean(0) + pred.std(0) * np.array([0.5, -0.3, 0.8, 0.1])
    eps = np.full(4, 1e-8)
    ref = _fraction_logpdf(y, pred, eps)
    assert 10.0 < ref < 50.0
    assert abs(oracle.gauss_logpdf_exact(y, pred, eps) - ref) <= 1e-13 * abs(ref)
    assert abs(oracle.gauss_logpdf(y, pred, eps) - ref) > 1e-10 * abs(ref)


@pytest.mark.reference
@pytest.mark.skipif(not rl.available(), reason=rl.UNAVAILABLE)
def test_oracle_predictions_against_the_live_reference():
    rs = np.random.RandomState(5)
    obs = rs.uniform(-0.2, 0.2, (12, 4))
    act = rs.randint(0, 2, 12)
    lo, hi = np.array(port.SEARCH_BOUNDS)[:, 0], np.array(port.SEARCH_BOUNDS)[:, 1]
    xi = lo + (hi - lo) * rs.uniform(size=(6, 4))
    for euler in (True, False):
        for lam, t in ((1, 0), (3, 4), (8, 2)):
            pred = oracle.predict(obs, act, t, lam, xi, euler)
            for m in range(len(xi)):
                env = rl.make_cartpole()
                env.kinematics_integrator = "euler" if euler else "semi-implicit"
                env.set_task(*xi[m])
                env.state = obs[t].copy()
                for k in range(lam):
                    s, _, _, _ = env.step(int(act[t + k]))
                    env.state = np.array(s)                              # keep stepping past the thresholds
                assert tuple(np.asarray(s, dtype=np.float64)) == tuple(pred[m]), (euler, lam, t, m)
