"""Float64 numpy restatement of the offline-DR log-likelihood (include/renv.h renv_cartpole_transition_loglik_f64).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Predictions come from ``cartpole_port.dynamics_step``, which is
bit-exact against the reference's step; the Gaussian fit is ``np.cov`` (ddof 1) plus a Cholesky factorisation, so
``loglik`` equals ``scipy.stats.multivariate_normal.logpdf(y, mu, S)`` wherever S is positive definite.
"""
import math

import numpy as np

from .cartpole_port import dynamics_step

LOG_2PI = math.log(2.0 * math.pi)


def window_starts(T, lam, episode_starts=()):
    """Starts t with t + lam <= T and no episode start in t+1 .. t+lam-1 (plain loops, independent of the product)."""
    starts = set(int(s) for s in episode_starts)
    return np.array([t for t in range(T - lam + 1) if not any(u in starts for u in range(t + 1, t + lam))], np.int32)


def predict(obs, actions, t, lam, xi, euler):
    """(M, 4) predictions: obs[t] pushed through lam dynamics steps under each row of xi (termination ignored)."""
    out = np.empty((len(xi), 4))
    s0 = tuple(float(v) for v in obs[t])
    acts = [int(a) for a in actions[t:t + lam]]
    for m, x in enumerate(xi):
        s, x = s0, tuple(float(v) for v in x)
        for a in acts:
            s, _ = dynamics_step(s, x, a, euler)
        out[m] = s
    return out


def gauss_logpdf(y, pred, eps):
    """log N(y; mean(pred), cov(pred) + diag(eps)); -inf when the Cholesky factorisation meets a pivot <= 0 or NaN."""
    mu = pred.mean(axis=0)
    S = np.cov(pred, rowvar=False, ddof=1) + np.diag(np.asarray(eps, dtype=np.float64))
    L = np.zeros((4, 4))
    for j in range(4):
        piv = S[j, j] - L[j, :j] @ L[j, :j]
        if not piv > 0:
            return -math.inf
        L[j, j] = math.sqrt(piv)
        for i in range(j + 1, 4):
            L[i, j] = (S[i, j] - L[i, :j] @ L[j, :j]) / L[j, j]
    r = np.asarray(y, dtype=np.float64) - mu
    z = np.zeros(4)
    for j in range(4):
        z[j] = (r[j] - L[j, :j] @ z[:j]) / L[j, j]
    return -0.5 * float(z @ z) - float(np.sum(np.log(np.diag(L)))) - 2.0 * LOG_2PI


def loglik(obs, actions, next_obs, windows, xi, lam, eps, euler=True):
    """(C, W) log-likelihoods and (C,) totals (math.fsum) of candidates xi (C, M, 4); NaN for a window out of range."""
    obs, next_obs, xi = np.asarray(obs, np.float64), np.asarray(next_obs, np.float64), np.asarray(xi, np.float64)
    eps = np.broadcast_to(np.asarray(eps, np.float64), (4,))
    T = len(obs)
    out = np.empty((len(xi), len(windows)))
    for c in range(len(xi)):
        for w, t in enumerate(windows):
            t = int(t)
            if t < 0 or t + lam > T:
                out[c, w] = math.nan
                continue
            out[c, w] = gauss_logpdf(next_obs[t + lam - 1], predict(obs, actions, t, lam, xi[c], euler), eps)
    return out, np.array([math.fsum(row) if np.all(np.isfinite(row)) else float(np.sum(row)) for row in out])
