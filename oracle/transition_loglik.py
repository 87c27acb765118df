"""Float64 numpy restatement of the offline-DR log-likelihood (include/renv.h renv_cartpole_transition_loglik_f64).

TEST INFRASTRUCTURE (see oracle/__init__.py).  Predictions come from ``cartpole_port.dynamics_step``, which is
bit-exact against the reference's step; the Gaussian fit is ``np.cov`` (ddof 1) plus a Cholesky factorisation, so
``loglik`` equals ``scipy.stats.multivariate_normal.logpdf(y, mu, S)`` wherever S is positive definite.

``loglik(..., exact=True)`` (``gauss_logpdf_exact``) fits the Gaussian without cancellation error: mu, Sigma (ddof 1)
and r = y - mu are computed exactly from the float64 predictions (integer arithmetic on their binary expansions) and
rounded once to float64; S = Sigma + diag(eps), the Cholesky factorisation, the solve and the log-determinant then run
in float64 as in ``gauss_logpdf``.  ``np.cov``'s two-pass float64 moments lose accuracy as the predicted states move
away from 0 -- about 3e-8 relative in l at x = 1e6 with a spread of 1e-4 -- while the exact mode stays within 1e-13 of
a rational evaluation of the whole objective there, so it can judge a kernel that claims more than the float64 form
delivers.  It costs a few ms per (candidate, window) at M = 1024.
"""
import math
from fractions import Fraction

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
    return _chol_logpdf(S, np.asarray(y, dtype=np.float64) - mu)


def exact_moments(pred):
    """(M, 4) finite float64 predictions -> (sum, cross, e): for every column i, pred[:, i] = n_i * 2**e[i] with
    integers n_i, sum[i] = sum_m n_i[m] and cross[i][j] = sum_m n_i[m] n_j[m], all exact Python ints."""
    pred = np.asarray(pred, dtype=np.float64)
    if not np.all(np.isfinite(pred)):
        raise ValueError("exact moments need finite predictions")
    mant, ex = np.frexp(pred)                         # pred = mant * 2**ex, |mant| in [0.5, 1) or 0
    mant = (mant * 2.0 ** 53).astype(np.int64)        # exact: 53 significant bits
    ex = ex.astype(np.int64) - 53
    cols, e = [], []
    for i in range(4):
        e0 = int(ex[:, i].min())
        cols.append([int(a) << int(b - e0) for a, b in zip(mant[:, i], ex[:, i])])
        e.append(e0)
    sums = [sum(c) for c in cols]
    cross = [[sum(a * b for a, b in zip(cols[i], cols[j])) if j >= i else None for j in range(4)] for i in range(4)]
    return sums, cross, e


def exact_fit(y, pred):
    """mu (4,), Sigma (4, 4) (ddof 1) and r = y - mu (4,), each the float64 rounding of the exact value."""
    M = len(pred)
    sums, cross, e = exact_moments(pred)
    scale = [Fraction(2) ** k for k in e]
    mu = [Fraction(sums[i], M) * scale[i] for i in range(4)]
    Sigma = np.empty((4, 4))
    for i in range(4):
        for j in range(i, 4):
            Sigma[i, j] = Sigma[j, i] = float(Fraction(M * cross[i][j] - sums[i] * sums[j], M * (M - 1))
                                              * scale[i] * scale[j])
    r = np.array([float(Fraction(float(y[i])) - mu[i]) for i in range(4)])
    return np.array([float(m) for m in mu]), Sigma, r


def gauss_logpdf_exact(y, pred, eps):
    """gauss_logpdf with mu, Sigma and y - mu computed exactly and rounded once; S, the Cholesky factorisation, the
    solve and the log-determinant in float64 (-inf on a pivot <= 0 or NaN)."""
    _, Sigma, r = exact_fit(y, pred)
    return _chol_logpdf(Sigma + np.diag(np.asarray(eps, dtype=np.float64)), r)


def _chol_logpdf(S, r):
    """-1/2 r' S^-1 r - 1/2 log det S - 2 log 2 pi by a float64 Cholesky factorisation; -inf on a pivot <= 0 or NaN."""
    L = np.zeros((4, 4))
    for j in range(4):
        piv = S[j, j] - L[j, :j] @ L[j, :j]
        if not piv > 0:
            return -math.inf
        L[j, j] = math.sqrt(piv)
        for i in range(j + 1, 4):
            L[i, j] = (S[i, j] - L[i, :j] @ L[j, :j]) / L[j, j]
    z = np.zeros(4)
    for j in range(4):
        z[j] = (r[j] - L[j, :j] @ z[:j]) / L[j, j]
    return -0.5 * float(z @ z) - float(np.sum(np.log(np.diag(L)))) - 2.0 * LOG_2PI


def loglik(obs, actions, next_obs, windows, xi, lam, eps, euler=True, exact=False):
    """(C, W) log-likelihoods and (C,) totals (math.fsum) of candidates xi (C, M, 4); NaN for a window out of range.
    exact=True fits each Gaussian with gauss_logpdf_exact instead of gauss_logpdf."""
    obs, next_obs, xi = np.asarray(obs, np.float64), np.asarray(next_obs, np.float64), np.asarray(xi, np.float64)
    eps = np.broadcast_to(np.asarray(eps, np.float64), (4,))
    T = len(obs)
    logpdf = gauss_logpdf_exact if exact else gauss_logpdf
    out = np.empty((len(xi), len(windows)))
    for c in range(len(xi)):
        for w, t in enumerate(windows):
            t = int(t)
            if t < 0 or t + lam > T:
                out[c, w] = math.nan
                continue
            out[c, w] = logpdf(next_obs[t + lam - 1], predict(obs, actions, t, lam, xi[c], euler), eps)
    return out, np.array([math.fsum(row) if np.all(np.isfinite(row)) else float(np.sum(row)) for row in out])
