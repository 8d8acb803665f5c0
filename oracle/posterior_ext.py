"""Extended-precision reference of the batched posterior draws (gpb200_posterior_draws_batched) -- TEST
INFRASTRUCTURE ONLY.

The entry point factors, per item, the joint prior covariance of (y, f^(p)(s))
    J = [[alpha^2 QQ(t, t) + sigma^2 I,   .                                ],
         [alpha^2 k_{p,0}(s, t),          alpha^2 k_{p,p}(s, s) + jitter I ]]
with the kernel pairs (QQ, QQ), (RQ, RR), (TQ, TT) for p = 0, 1, 2 (gram_cond_batched_kernel, gram.cu).  Its factor is
[[L11, 0], [L21, L22]]: mu = L21 L11^-1 y is the posterior mean and L22 the unique Cholesky factor of the posterior
covariance + jitter I, so L22 can be compared element by element.

posterior_ext runs the unblocked LLT of J (the value half of chol_deriv_ext.llt_dual) in np.longdouble, which on x86
carries a 64-bit significand: 11 bits more than the float64 result it is compared with.  posterior_f64 is the same
computation in float64 through LAPACK, the baseline whose own error against posterior_ext scales the tolerances of
the GPU tests.  Cost of the long-double LLT: about 0.1 s at n + m = 516, 0.6 s at 1024, 2.3 s at 1536, 20 s at 3072.
"""
from __future__ import annotations

from collections import namedtuple

import numpy as np
import scipy.linalg as sla

from oracle.chol_deriv_ext import LONGDOUBLE_OK

KINDS = {0: ("QQ", "QQ"), 1: ("RQ", "RR"), 2: ("TQ", "TT")}

# derivative_kernels.R:39-73 as functions of e = exp(-d^2 / (2 l^2)), d = tj - tk and l; RQ, TQ and TR are QR, QT and
# RT with the points swapped (as in oracle.gp_oracle)
_BASE = {
    "QQ": lambda e, d, l: e,
    "QR": lambda e, d, l: (e * d) / l ** 2,
    "RR": lambda e, d, l: e / l ** 2 - (e * d ** 2) / l ** 4,
    "QT": lambda e, d, l: -(e / l ** 2) + (e * d ** 2) / l ** 4,
    "RT": lambda e, d, l: (3 * e * d) / l ** 4 - (e * d ** 3) / l ** 6,
    "TT": lambda e, d, l: (3 * e) / l ** 4 - (6 * e * d ** 2) / l ** 6 + (e * d ** 4) / l ** 8,
}
_SWAPPED = {"RQ": "QR", "TQ": "QT", "TR": "RT"}

Posterior = namedtuple("Posterior", "mu L22 info draws")


def outer_kernel(name, tj, tk, l, dtype):
    """oracle.gp_oracle.outer_kernel evaluated in `dtype` from the float64 points and length scale."""
    tj = np.asarray(tj, dtype=np.float64).astype(dtype)
    tk = np.asarray(tk, dtype=np.float64).astype(dtype)
    if name in _SWAPPED:
        name, tj, tk = _SWAPPED[name], tk, tj
        d = tj[None, :] - tk[:, None]
    else:
        d = tj[:, None] - tk[None, :]
    l = dtype(l)
    return _BASE[name](np.exp(-(d ** 2 / (2 * l ** 2))), d, l)


def joint_cov(t, s, theta, order, jitter, dtype=np.float64):
    """The (n+m) x (n+m) joint prior covariance J of (y, f^(order)(s)) in `dtype`; s = None predicts on t."""
    s = t if s is None else s
    alpha, rho, sigma = (dtype(float(v)) for v in theta)
    a2 = alpha * alpha
    n, m = len(t), len(s)
    kc, kss = KINDS[order]
    J = np.empty((n + m, n + m), dtype=dtype)
    J[:n, :n] = a2 * outer_kernel("QQ", t, t, rho, dtype)
    J[n:, :n] = a2 * outer_kernel(kc, s, t, rho, dtype)
    J[:n, n:] = J[n:, :n].T
    J[n:, n:] = a2 * outer_kernel(kss, s, s, rho, dtype)
    J[np.arange(n), np.arange(n)] += sigma * sigma
    J[np.arange(n, n + m), np.arange(n, n + m)] += dtype(jitter)
    return J


def llt(J):
    """Unblocked left-looking LLT in the dtype of J; returns (L, info) with info the 1-based index of the first pivot
    that is not > 0 (0 when J is positive definite; L is then incomplete)."""
    N = J.shape[0]
    L = np.zeros_like(J)
    for j in range(N):
        lj = L[j, :j]
        d = J[j, j] - lj @ lj
        if not d > 0:
            return L, j + 1
        d = np.sqrt(d)
        L[j, j] = d
        if j + 1 < N:
            L[j + 1:, j] = (J[j + 1:, j] - L[j + 1:, :j] @ lj) / d
    return L, 0


def _result(L, info, n, m, y, eps, solve):
    if info:
        nan = np.full(m, np.nan)
        return Posterior(nan, np.full((m, m), np.nan), info, None if eps is None else np.full((len(eps), m), np.nan))
    mu = L[n:, :n] @ solve(L[:n, :n], y)
    L22 = L[n:, n:]
    draws = None if eps is None else mu[None, :] + eps @ L22.T
    f = lambda a: None if a is None else np.asarray(a, dtype=np.float64)
    return Posterior(f(mu), f(L22), 0, f(draws))


def _forward_ld(L, b):
    x = np.zeros_like(b)
    for i in range(len(b)):
        x[i] = (b[i] - L[i, :i] @ x[:i]) / L[i, i]
    return x


def posterior_ext(t, s, y, theta, order, jitter, eps=None):
    """Posterior(mu, L22, info, draws) from the long-double LLT of J, as float64 arrays.  eps: optional (k, m) normals;
    draws[i] = mu + L22 eps[i], formed in long double.  Failed factorisations give NaN outputs and info != 0."""
    if not LONGDOUBLE_OK:
        raise RuntimeError("np.longdouble carries %d mantissa bits; the reference LLT needs 63" % np.finfo(np.longdouble).nmant)
    n, m = len(t), len(t) if s is None else len(s)
    L, info = llt(joint_cov(t, s, theta, order, jitter, np.longdouble))
    y = np.asarray(y, dtype=np.float64).astype(np.longdouble)
    eps = None if eps is None else np.atleast_2d(np.asarray(eps, dtype=np.float64)).astype(np.longdouble)
    return _result(L, info, n, m, y, eps, _forward_ld)


def posterior_f64(t, s, y, theta, order, jitter, eps=None):
    """The same in float64 through LAPACK (dpotrf and a triangular solve): the baseline."""
    n, m = len(t), len(t) if s is None else len(s)
    L, info = sla.lapack.dpotrf(joint_cov(t, s, theta, order, jitter), lower=1, clean=1)
    eps = None if eps is None else np.atleast_2d(np.asarray(eps, dtype=np.float64))
    solve = lambda A, b: sla.solve_triangular(A, b, lower=True, check_finite=False)
    return _result(L, int(info), n, m, np.asarray(y, dtype=np.float64), eps, solve)
