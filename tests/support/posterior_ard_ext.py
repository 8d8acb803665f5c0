"""Extended-precision reference of the batched ARD posterior draws (gpb200_posterior_draws_ard_batched) -- TEST
INFRASTRUCTURE ONLY.

The ARD twin of oracle/posterior_ext.py: the joint prior covariance of (y, f(Xs)) under QQard (R/kernels.R:19) is
factored by that file's unblocked LLT, in np.longdouble (posterior_ard_ext) or in float64 through LAPACK
(posterior_ard_f64, the baseline whose own error scales the tolerances of tests/test_posterior_draws_ard_gpu.py), and
turned into (mu, L22, info, draws) by the same _result.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

from oracle.chol_deriv_ext import LONGDOUBLE_OK
from oracle.posterior_ext import _forward_ld, _result, llt


def ard_joint_cov(X, Xs, theta, jitter, dtype=np.float64):
    """The (n+m) x (n+m) joint prior covariance of (y, f(Xs)) under QQard in `dtype`:
    k(p, q) = alpha^2 exp(-0.5 sum_d (p_d - q_d)^2 / rho_d^2) off the diagonal; the diagonal is alpha^2 + sigma^2 on the
    first n entries and alpha^2 + jitter on the last m, as the GPU kernel writes it.  X: (n, D), Xs: (m, D) or None
    (predict on X); theta = (alpha, rho_1 .. rho_D, sigma)."""
    X = np.atleast_2d(np.asarray(X, dtype=np.float64))
    Xs = X if Xs is None else np.atleast_2d(np.asarray(Xs, dtype=np.float64))
    theta = [dtype(float(v)) for v in theta]
    alpha, rho, sigma = theta[0], np.array(theta[1:-1], dtype=dtype), theta[-1]
    n, m = X.shape[0], Xs.shape[0]
    P = np.vstack([X, Xs]).astype(dtype) / rho[None, :]
    r2 = np.zeros((n + m, n + m), dtype=dtype)
    for d in range(P.shape[1]):
        diff = P[:, d][:, None] - P[:, d][None, :]
        r2 += diff * diff
    J = alpha * alpha * np.exp(-r2 / dtype(2))
    J[np.arange(n + m), np.arange(n + m)] = alpha * alpha   # no exponential on the diagonal: a NaN point fails off it
    J[np.arange(n), np.arange(n)] += sigma * sigma
    J[np.arange(n, n + m), np.arange(n, n + m)] += dtype(jitter)
    return J


def posterior_ard_ext(X, Xs, y, theta, jitter, eps=None):
    """Posterior(mu, L22, info, draws) from the long-double LLT of ard_joint_cov, as float64 arrays.  eps: optional
    (k, m) normals; draws[i] = mu + L22 eps[i].  Failed factorisations give NaN outputs and info != 0."""
    if not LONGDOUBLE_OK:
        raise RuntimeError("np.longdouble carries %d mantissa bits; the reference LLT needs 63" % np.finfo(np.longdouble).nmant)
    n = np.shape(X)[0]
    m = n if Xs is None else np.shape(Xs)[0]
    L, info = llt(ard_joint_cov(X, Xs, theta, jitter, np.longdouble))
    y = np.asarray(y, dtype=np.float64).astype(np.longdouble)
    eps = None if eps is None else np.atleast_2d(np.asarray(eps, dtype=np.float64)).astype(np.longdouble)
    return _result(L, info, n, m, y, eps, _forward_ld)


def posterior_ard_f64(X, Xs, y, theta, jitter, eps=None):
    """The same in float64 through LAPACK (dpotrf and a triangular solve): the baseline."""
    n = np.shape(X)[0]
    m = n if Xs is None else np.shape(Xs)[0]
    L, info = sla.lapack.dpotrf(ard_joint_cov(X, Xs, theta, jitter), lower=1, clean=1)
    eps = None if eps is None else np.atleast_2d(np.asarray(eps, dtype=np.float64))
    solve = lambda A, b: sla.solve_triangular(A, b, lower=True, check_finite=False)
    return _result(L, int(info), n, m, np.asarray(y, dtype=np.float64), eps, solve)
