"""Offline DR fitting: the log-likelihood of candidate task distributions on recorded cart-pole transitions.

DROPO-style fitting (offline ADR) scores a candidate distribution p(xi) against transitions (s_t, a_t, s_{t+1}) recorded
on the real system: draw M tasks xi_m ~ p, put the simulator in state s_t with task xi_m, apply the recorded action(s),
fit a Gaussian to the M predicted states and sum the log-density of the observed next state over all transitions.
Around the reference env that is one set_task / state assignment / step per (candidate, transition, sample, step);
here it is one fp64 kernel per call (include/renv.h renv_cartpole_transition_loglik_f64)::

    data = TransitionDataset(obs, actions, next_obs, episode_starts=starts)
    ll = data.log_likelihood(xi, lam=1, epsilon=2e-4)                         # xi (C, M, 4) -> total (C,)
    ll = data.dr_log_likelihood("truncnorm", distrs, num_samples=1024, seed=0)  # what an optimiser calls

For a window starting at t (lam transitions t .. t+lam-1 of one episode), candidate c and sample m:
    s_m = lam applications of RandomCartPoleEnv's dynamics (fp64, the arithmetic of step; termination ignored: no
          TimeLimit, no reset) under xi[c, m] and actions[t .. t+lam-1], starting from obs[t]
    y = next_obs[t+lam-1],  mu = mean_m s_m,  Sigma = numpy.cov(s, rowvar=False) (ddof 1),  S = Sigma + diag(epsilon)
    l[c, w] = scipy.stats.multivariate_normal.logpdf(y, mu, S)   (-inf when the Cholesky factorisation of S fails)
    total[c] = sum_w l[c, w]
Results are bitwise reproducible: l[c] and total[c] depend only on the data, the windows, xi[c], epsilon, lam and the
integrator -- not on how many candidates share the call or where c sits among them.
"""
import ctypes

import numpy as np

from . import _device, _lib
from .random_env import TaskSampler

__all__ = ["TransitionDataset"]


def _host(x, name, dtype):
    t = _device.torch()
    if isinstance(x, t.Tensor):
        x = x.detach().cpu().numpy()
    a = np.asarray(x)
    if dtype is not None:
        if a.dtype.kind not in "biuf":
            raise TypeError("%s must be numeric, got %s" % (name, a.dtype))
        a = a.astype(dtype)
    return a


def _epsilon(epsilon):
    eps = np.broadcast_to(np.asarray(epsilon, dtype=np.float64), (4,)) if np.ndim(epsilon) == 0 else \
        np.asarray(epsilon, dtype=np.float64)
    if eps.shape != (4,):
        raise ValueError("epsilon must be a scalar or a 4-vector, got shape %s" % (eps.shape,))
    if not (np.all(np.isfinite(eps)) and np.all(eps >= 0)):
        raise ValueError("epsilon must be finite and >= 0, got %s" % eps)
    return eps


def _integrator(kinematics_integrator):
    # random_cartpole.py:187-196: 'euler' selects Euler, anything else the semi-implicit update
    return _lib.EULER if kinematics_integrator == "euler" else _lib.SEMI_IMPLICIT


class TransitionDataset:
    """T recorded transitions (obs[i], actions[i], next_obs[i]) of the cart-pole, uploaded once as float64.

    obs, next_obs: (T, 4) x, x_dot, theta, theta_dot; actions: (T,) in {0, 1}; numpy arrays or torch tensors.
    episode_starts: indices of the transitions that begin an episode (or a boolean mask of length T); None = one
    episode.  A window of lam transitions starting at t is scored iff t + lam <= T and no episode starts at
    t+1 .. t+lam-1, so a multi-step prediction never crosses a reset.  Transitions whose next_obs is not the dynamics'
    successor of obs (e.g. the reset observation an auto-resetting vector env returns on `done`) belong out of the data.
    """

    def __init__(self, obs, actions, next_obs, episode_starts=None, device="cuda"):
        t = _device.torch()
        obs = _host(obs, "obs", np.float64)
        next_obs = _host(next_obs, "next_obs", np.float64)
        act = _host(actions, "actions", None)
        if obs.ndim != 2 or obs.shape[1] != 4 or obs.shape[0] < 1:
            raise ValueError("obs must have shape (T, 4) with T >= 1, got %s" % (obs.shape,))
        T = obs.shape[0]
        if next_obs.shape != obs.shape:
            raise ValueError("next_obs must have the shape of obs %s, got %s" % (obs.shape, next_obs.shape))
        if act.shape != (T,):
            raise ValueError("actions must have shape (%d,), got %s" % (T, act.shape))
        if not (np.all(np.isfinite(obs)) and np.all(np.isfinite(next_obs))):
            raise ValueError("obs and next_obs must be finite")
        bad = ~np.isin(act, (0, 1))
        if bad.any():
            a = act[np.argmax(bad)].item()
            raise AssertionError("%r (%s) invalid" % (a, type(a)))        # random_cartpole.py:173-174
        starts = np.zeros(T, dtype=bool)
        starts[0] = True
        if episode_starts is not None:
            es = _host(episode_starts, "episode_starts", None)
            if es.dtype == bool:
                if es.shape != (T,):
                    raise ValueError("an episode_starts mask must have shape (%d,), got %s" % (T, es.shape))
                starts |= es
            else:
                es = es.reshape(-1)
                if es.size and (es.dtype.kind not in "iu" or es.min() < 0 or es.max() >= T):
                    raise ValueError("episode_starts must be indices in [0, %d)" % T)
                starts[es] = True
        self.num_transitions = T
        self.episode_starts = np.flatnonzero(starts)
        self._starts_cum = np.cumsum(starts)
        self.device = _device.require_cuda(device)
        self.obs = t.as_tensor(obs, dtype=t.float64).to(self.device).contiguous()
        self.next_obs = t.as_tensor(next_obs, dtype=t.float64).to(self.device).contiguous()
        self.actions = t.as_tensor(act.astype(np.uint8)).to(self.device).contiguous()
        self._windows = {}

    def window_starts(self, lam=1):
        """Start indices of the windows of lam transitions (host int32 array)."""
        lam = int(lam)
        if lam < 1:
            raise ValueError("lam must be >= 1")
        T = self.num_transitions
        if lam > T:
            return np.zeros(0, dtype=np.int32)
        t0 = np.arange(T - lam + 1)
        # episode starts at t+1 .. t+lam-1: cum[t+lam-1] - cum[t]
        inside = self._starts_cum[t0 + lam - 1] - self._starts_cum[t0]
        return t0[inside == 0].astype(np.int32)

    def num_windows(self, lam=1):
        return int(self.window_starts(lam).size)

    def _window_tensor(self, lam):
        w = self._windows.get(lam)
        if w is None:
            starts = self.window_starts(lam)
            if starts.size == 0:
                raise ValueError("no window of %d transitions lies inside one episode" % lam)
            w = self._windows[lam] = _device.torch().as_tensor(starts).to(self.device)
        return w

    def log_likelihood(self, xi, lam=1, epsilon=2e-4, kinematics_integrator="euler", per_window=False):
        """Log-likelihood of the data under C candidates, each given by M >= 2 task samples.

        xi: (C, M, 4) or (M, 4) float64 tensor on the dataset's device (gravity, cart_mass, pole_mass, pole_length).
        epsilon: scalar or 4-vector >= 0 added to the diagonal of each predicted covariance.  Under Euler with lam = 1
        x and theta of the prediction do not depend on xi, so two rows of the covariance are exactly zero and
        epsilon keeps S invertible; with observation noise of std sigma, 2 sigma^2 is the natural floor.
        Returns total (C,) float64 -- or, with per_window=True, (total, l) with l (C, W) the per-window values in the
        order of window_starts(lam).  A (M, 4) xi drops the candidate dimension from both.
        """
        t = _device.torch()
        if not isinstance(xi, t.Tensor) or xi.dtype != t.float64 or xi.device != self.device:
            raise ValueError("xi must be a float64 tensor on %s" % self.device)
        single = xi.dim() == 2
        x = xi.unsqueeze(0) if single else xi
        if x.dim() != 3 or x.shape[2] != 4:
            raise ValueError("xi must have shape (C, M, 4) or (M, 4), got %s" % (tuple(xi.shape),))
        C, M = int(x.shape[0]), int(x.shape[1])
        if C < 1 or M < 2:
            raise ValueError("xi needs C >= 1 candidates of M >= 2 samples, got %s" % (tuple(xi.shape),))
        lam = int(lam)
        if not 1 <= lam <= self.num_transitions:
            raise ValueError("lam must lie in [1, T = %d]" % self.num_transitions)
        eps = _epsilon(epsilon)
        windows = self._window_tensor(lam)
        x = x.contiguous()
        W = int(windows.numel())
        loglik = t.empty((C, W), dtype=t.float64, device=self.device)
        total = t.empty(C, dtype=t.float64, device=self.device)
        data = _lib.Transitions()
        data.obs, data.next_obs = self.obs.data_ptr(), self.next_obs.data_ptr()
        data.action, data.window = self.actions.data_ptr(), windows.data_ptr()
        data.T, data.W = self.num_transitions, W
        with t.cuda.device(self.device):
            _lib.call("renv_cartpole_transition_loglik_f64", ctypes.byref(data), lam, _integrator(kinematics_integrator),
                      _device.ptr(x), C, M, (ctypes.c_double * 4)(*eps), _device.ptr(loglik), _device.ptr(total),
                      _device.stream_ptr(self.device))
        if single:
            total, loglik = total[0], loglik[0]
        return (total, loglik) if per_window else total

    def sample_candidates(self, dr_type, distrs, num_samples=1024, seed=0):
        """(C, M, 4) float64 task samples of C distributions, each drawn as TaskSampler('RandomCartPole-v0') with
        seed_dr(seed) then sample_tasks_tensor(M, float64) draws them: every candidate uses the same Philox counters
        (common random numbers).  distrs: the `distr` arguments of set_dr_distribution (interleaved pairs, or
        {"mean", "cov"} for fullgaussian).  Raises the reference's Exception when a gaussian dim stays below 0.1."""
        t = _device.torch()
        distrs = list(distrs)
        if not distrs:
            raise ValueError("distrs must hold at least one distribution")
        M = int(num_samples)
        if M < 2:
            raise ValueError("num_samples must be >= 2")
        xi = t.empty((len(distrs), M, 4), dtype=t.float64, device=self.device)
        sampler = TaskSampler("RandomCartPole-v0")
        for c, distr in enumerate(distrs):
            sampler.set_dr_distribution(dr_type, distr)
            sampler.seed_dr(seed)
            sampler.sample_tasks_tensor(M, dtype=t.float64, device=self.device, out=xi[c])
        sampler.check_dr_violations()
        return xi

    def dr_log_likelihood(self, dr_type, distrs, num_samples=1024, seed=0, lam=1, epsilon=2e-4,
                          kinematics_integrator="euler", per_window=False):
        """log_likelihood of C candidate distributions (the objective an optimiser such as CMA-ES evaluates for its
        population): sample_candidates(dr_type, distrs, num_samples, seed), then log_likelihood on them."""
        xi = self.sample_candidates(dr_type, distrs, num_samples, seed)
        return self.log_likelihood(xi, lam, epsilon, kinematics_integrator, per_window)
