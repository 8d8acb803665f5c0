"""Host-side mirror of the Stan Math functions the reference's exact-GP models call
(models/fit_hyperparameters.stan:18-31, exact_gp.stan:16-26, heteroscedastic_centered.stan:24-34):
same names and argument meaning, arithmetic on the GPU through the C ABI.

fit_hyperparameters_lp reproduces the model block of models/fit_hyperparameters.stan as the
(lp__, gradient) pair NUTS asks for on the unconstrained scale -- the value a Stan external function
built on include/gp_lml_stan.hpp returns.
"""
from __future__ import annotations

import math

import numpy as np

from . import capi


def cov_exp_quad(x, alpha, rho, diag_add=0.0, handle=None):
    """cov_exp_quad(x, alpha, rho) (+ diag_add on the diagonal, fused: fit_hyperparameters.stan:19-24)."""
    return (handle or capi.default_handle()).gram_se(x, float(alpha), float(rho), float(diag_add))


def cholesky_decompose(K, handle=None):
    """Lower factor; raises NotPositiveDefiniteError where Stan throws std::domain_error."""
    K = np.asarray(K, dtype=np.float64)
    if K.ndim != 2 or K.shape[0] != K.shape[1]:
        raise capi.GpB200Error("cholesky_decompose: matrix is not square")
    if K.size and np.max(np.abs(K - K.T)) > 1e-8:   # Stan's check_symmetric tolerance
        raise capi.GpB200Error("cholesky_decompose: matrix is not symmetric")
    return (handle or capi.default_handle()).potrf(K)


def mdivide_left_tri_low(L, b, handle=None):
    return (handle or capi.default_handle()).trsm_lower(L, b)


def multi_normal_cholesky_lpdf(y, mu, L, drop_constants=False, handle=None):
    return (handle or capi.default_handle()).mvn_chol_lpdf(y, mu, L, drop_constants)


def multiply_lower_tri(L, z, handle=None):
    """f = L * z of the non-centred latent models (exact_gp.stan:25)."""
    return (handle or capi.default_handle()).trmv_lower(L, z)


def gp_lml_grad(x, y, alpha, rho, sigma, jitter=0.0, handle=None):
    """LML (with constants) and d/d(alpha, rho, sigma)."""
    return (handle or capi.default_handle()).lml_grad(x, y, [alpha, rho, sigma], jitter)


def gp_lml_grad_draws(x, y, theta, jitter=0.0, want_grad=True, handle=None):
    """Batched over hyper-parameter draws / groups: theta (B, 3); x, y shared (n,) or per item (B, n)."""
    return (handle or capi.default_handle()).lml_grad_batched(x, y, theta, jitter, want_grad)


def gp_lml_grad_ard_draws(X, y, theta, jitter=0.0, want_grad=True, handle=None):
    """The same with the ARD covariance (QQard) on multi-column inputs: X (n, D) shared or (B, n, D) per item,
    theta (B, D + 2) = (alpha, rho_1 .. rho_D, sigma); y (n,) or (B, n)."""
    return (handle or capi.default_handle()).lml_grad_ard_batched(X, y, theta, jitter, want_grad)


def gp_lml_grad_groups(xs, ys, theta, jitter=0.0, want_grad=True, handle=None):
    """One GP per group with the group's own size (multiple_players.stan:59-63): xs, ys lists of B 1-D arrays,
    theta (B, 3).  All B LMLs and gradients in one call; returns lml[B], grad[B,3], info[B]."""
    return (handle or capi.default_handle()).lml_grad_ragged(xs, ys, theta, jitter, want_grad)


def fit_hyperparameters_lp(x, y, log_rho, log_alpha, log_sigma, handle=None):
    """lp__ and its gradient w.r.t. the unconstrained (log rho, log alpha, log sigma) for
    models/fit_hyperparameters.stan: `~` likelihood (constant dropped, :31), gamma(4,4) and
    normal(0,1) priors (:27-29), log-Jacobians of the <lower=0> transforms (:13-15)."""
    rho, alpha, sigma = math.exp(log_rho), math.exp(log_alpha), math.exp(log_sigma)
    n = len(x)
    lml, g = gp_lml_grad(x, y, alpha, rho, sigma, handle=handle)
    lp = lml + 0.5 * n * math.log(2.0 * math.pi)
    lp += 3.0 * math.log(rho) - 4.0 * rho - 0.5 * alpha * alpha - 0.5 * sigma * sigma
    lp += log_rho + log_alpha + log_sigma
    d_rho = g[1] + 3.0 / rho - 4.0
    d_alpha = g[0] - alpha
    d_sigma = g[2] - sigma
    grad = np.array([d_rho * rho + 1.0, d_alpha * alpha + 1.0, d_sigma * sigma + 1.0])
    return lp, grad
