"""mpmath (50-digit) arbiter for the oracle at N <= 64 -- TEST INFRASTRUCTURE ONLY.
Restates models/fit_hyperparameters.stan:18-31 and the gradient formulas of SURVEY Appendix B in
arbitrary precision so that NumPy, C and CUDA results can be ranked against a value that is not
subject to float64 rounding."""
from __future__ import annotations

import mpmath as mp

mp.mp.dps = 50


def _gram(x, alpha, rho, diag_add):
    n = len(x)
    K = mp.matrix(n, n)
    for i in range(n):
        for j in range(n):
            d = mp.mpf(x[i]) - mp.mpf(x[j])
            K[i, j] = mp.mpf(alpha) ** 2 * mp.exp(-d * d / (2 * mp.mpf(rho) ** 2))
        K[i, i] += diag_add
    return K


def lml_grad(x, y, alpha, rho, sigma, jitter=0.0):
    n = len(x)
    alpha, rho, sigma = mp.mpf(alpha), mp.mpf(rho), mp.mpf(sigma)
    K = _gram(x, alpha, rho, sigma ** 2 + mp.mpf(jitter))
    L = mp.cholesky(K)
    yv = mp.matrix([mp.mpf(v) for v in y])
    z = mp.lu_solve(L, yv)
    Kinv = mp.inverse(K)
    a = Kinv * yv
    lml = -mp.mpf(n) / 2 * mp.log(2 * mp.pi) - sum(mp.log(L[i, i]) for i in range(n)) - (z.T * z)[0] / 2
    g = [mp.mpf(0)] * 3
    for i in range(n):
        for j in range(n):
            d = mp.mpf(x[i]) - mp.mpf(x[j])
            kse = alpha ** 2 * mp.exp(-d * d / (2 * rho ** 2))
            m = a[i] * a[j] - Kinv[i, j]
            g[0] += m * 2 * kse / alpha / 2
            g[1] += m * kse * d * d / rho ** 3 / 2
            if i == j:
                g[2] += m * 2 * sigma / 2
    return float(lml), [float(v) for v in g]


def chol_tangent(x, alpha, rho, diag_add, wrt):
    """L = chol(alpha^2 E + diag_add I) and dL/dtheta (theta = alpha for wrt == "alpha", rho for wrt == "rho") by the
    dual-number LLT of covariance.cpp:13-39 carried in 50 digits; returned as nested lists of floats."""
    n = len(x)
    alpha, rho = mp.mpf(alpha), mp.mpf(rho)
    K = [[None] * n for _ in range(n)]
    Kd = [[None] * n for _ in range(n)]
    for i in range(n):
        for j in range(n):
            d2 = (mp.mpf(x[i]) - mp.mpf(x[j])) ** 2
            e = mp.exp(-d2 / (2 * rho ** 2))
            K[i][j] = alpha ** 2 * e + (mp.mpf(diag_add) if i == j else 0)
            Kd[i][j] = 2 * alpha * e if wrt == "alpha" else alpha ** 2 * e * d2 / rho ** 3
    Lv = [[mp.mpf(0)] * n for _ in range(n)]
    Lt = [[mp.mpf(0)] * n for _ in range(n)]
    for j in range(n):
        sv = K[j][j] - sum(Lv[j][k] ** 2 for k in range(j))
        st = Kd[j][j] - 2 * sum(Lv[j][k] * Lt[j][k] for k in range(j))
        dv = mp.sqrt(sv)
        dt = st / (2 * dv)
        Lv[j][j], Lt[j][j] = dv, dt
        for i in range(j + 1, n):
            cv = K[i][j] - sum(Lv[i][k] * Lv[j][k] for k in range(j))
            ct = Kd[i][j] - sum(Lv[i][k] * Lt[j][k] + Lt[i][k] * Lv[j][k] for k in range(j))
            Lv[i][j] = cv / dv
            Lt[i][j] = (ct - Lv[i][j] * dt) / dv
    return [[float(v) for v in r] for r in Lv], [[float(v) for v in r] for r in Lt]
