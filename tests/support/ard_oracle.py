"""NumPy float64 reference of the ARD LML + gradient (gpb200_lml_grad_ard_batched): Cholesky, explicit inverse and
the trace formula, written from the model, independent of the CUDA code."""
import numpy as np
import scipy.linalg as sla

from oracle import gp_oracle as o


def lml_grad_ard(X, y, alpha, rho, sigma, jitter=0.0):
    """K = alpha^2 exp(-0.5 sum_d (X_id - X_jd)^2 / rho_d^2) + (sigma^2 + jitter) I (QQard, R/kernels.R:19);
    returns (lml, grad) with grad = d lml / d (alpha, rho_1 .. rho_D, sigma), from
    d lml / d theta = 0.5 tr((a a^T - K^-1) dK/dtheta), a = K^-1 y.  Raises o.NotPositiveDefinite on a failed pivot."""
    X = np.asarray(X, dtype=np.float64)
    if X.ndim == 1:
        X = X[:, None]
    y = np.asarray(y, dtype=np.float64)
    rho = np.asarray(rho, dtype=np.float64).reshape(-1)
    n, D = X.shape
    diff2 = (X[:, None, :] - X[None, :, :]) ** 2                  # (n, n, D)
    Kse = alpha * alpha * np.exp(-0.5 * np.sum(diff2 / (rho * rho), axis=2))
    K = o.add_diag(Kse, sigma * sigma + jitter)
    L = o.cholesky_decompose(K)
    z = o.mdivide_left_tri_low(L, y)
    a = o.mdivide_right_tri_low_T(L, z)
    val = -0.5 * n * o.LOG_TWO_PI - np.sum(np.log(np.diag(L))) - 0.5 * float(z @ z)
    Linv = sla.solve_triangular(L, np.eye(n), lower=True, check_finite=False)
    M = np.outer(a, a) - Linv.T @ Linv
    g = np.empty(D + 2)
    g[0] = 0.5 * np.sum(M * (2.0 * Kse / alpha))
    for d in range(D):
        g[1 + d] = 0.5 * np.sum(M * (Kse * diff2[:, :, d] / rho[d] ** 3))
    g[D + 1] = 0.5 * np.trace(M) * 2.0 * sigma
    return float(val), g


def pivot(X, alpha, rho, sigma, jitter=0.0):
    """1-based index of the first pivot of the ARD covariance that is not > 0 (0 when it factors).  A NaN pivot counts
    as a failure, as in the library; column-by-column Cholesky rather than dpotrf, whose NaN handling differs between
    LAPACK builds (OpenBLAS's does not stop at a NaN pivot)."""
    X = np.asarray(X, dtype=np.float64)
    if X.ndim == 1:
        X = X[:, None]
    rho = np.asarray(rho, dtype=np.float64).reshape(-1)
    diff2 = (X[:, None, :] - X[None, :, :]) ** 2
    K = o.add_diag(alpha * alpha * np.exp(-0.5 * np.sum(diff2 / (rho * rho), axis=2)), sigma * sigma + jitter)
    n = K.shape[0]
    L = np.zeros_like(K)
    for j in range(n):
        d = K[j, j] - L[j, :j] @ L[j, :j]
        if not d > 0.0:
            return j + 1
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (K[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return 0


def synth_ard(n, D, B, seed, per_item=False):
    """Inputs on a scale where every length-scale matters: X ~ U(0, 3)^D, y a smooth function + noise,
    theta rows (alpha, rho_1 .. rho_D, sigma)."""
    rng = np.random.default_rng(seed)
    shape = (B, n, D) if per_item else (n, D)
    X = rng.uniform(0.0, 3.0, size=shape)
    w = rng.standard_normal(D)
    f = np.sin(X @ w) + 0.3 * np.cos(2.0 * X[..., 0])
    y = f + 0.2 * rng.standard_normal(f.shape)
    theta = np.empty((B, D + 2))
    theta[:, 0] = np.abs(rng.standard_normal(B)) + 0.3
    theta[:, 1:D + 1] = rng.uniform(0.4, 2.5, size=(B, D))
    theta[:, D + 1] = rng.uniform(0.1, 0.5, size=B)
    return X, y, theta

