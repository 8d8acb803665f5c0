"""Host-side mirror of the reference's non-centred latent exact-GP models (SURVEY CS-E):
models/exact_gp.stan:16-33 and, with an amplitude, models/fit_full_gp.stan:18-26 /
westbrook_exact.stan:17-24.

    Sigma = cov_exp_quad(x, alpha, l) + jitter I ;  L = cholesky_decompose(Sigma) ;  f = L z
    z ~ normal(0, 1) ;  l ~ gamma(4, 4) ;  y ~ normal(f, sigma)

Stan differentiates THROUGH the Cholesky.  Default route (reverse mode, what Stan itself does): gpb200_latent_forward
gives f = L z and keeps L on the device, gpb200_latent_backward turns fbar = d lp / d f into zbar = L^T fbar and
d lp / d (alpha, l) with ONE pass of the Cholesky adjoint  Kbar = L^-T Phi(L^T tril(fbar z^T)) L^-1  contracted with
dK/dtheta (N^3 flops for all parameters).  The forward-mode route of round 1 is kept (reverse=False): the factor and its
tangent from gpb200_se_chol_tangent (for alpha = 1, jitter = 1e-10 exactly rbf_cov_chol, covariance.cpp:9-47), one
5 N^3 / 3 pass per parameter, d lp / d l = fbar^T (dL/dl z).  Both must agree -- tests/test_host_mirror_gpu.py.
exact_gp_log_prob_batched evaluates B parameter states (chains of a vectorised sampler, or posterior draws) with one
batched forward and one batched backward call.
"""
from __future__ import annotations

import numpy as np

from . import capi


def transformed_parameters(x, l, z, alpha=1.0, jitter=1e-10, handle=None):
    """f = L z and df/dl = (dL/dl) z  (exact_gp.stan:16-26)."""
    h = handle or capi.default_handle()
    L, dL = h.se_chol_tangent(x, float(alpha), float(l), float(jitter), 1)
    f = h.trmv_lower(L, z)
    dfdl = h.trmv_lower(dL, z)
    return f, dfdl, L


def exact_gp_log_prob(x, y, l, sigma, z, alpha=1.0, jitter=1e-10, handle=None, reverse=True):
    """lp (constants dropped as Stan's `~` does) of models/exact_gp.stan and its gradient with
    respect to the constrained parameters (l, sigma, z) -- and alpha, for fit_full_gp.stan."""
    h = handle or capi.default_handle()
    y = np.asarray(y, dtype=np.float64)
    z = np.asarray(z, dtype=np.float64)
    n = y.shape[0]
    if reverse:
        f = h.latent_forward(x, float(alpha), float(l), float(jitter), z)
    else:
        f, dfdl, L = transformed_parameters(x, l, z, alpha, jitter, h)
    r = y - f
    lp = -0.5 * float(z @ z) + 3.0 * np.log(l) - 4.0 * l - n * np.log(sigma) - 0.5 * float(r @ r) / sigma ** 2
    fbar = r / sigma ** 2
    if reverse:
        (g_alpha, g_l_through), zbar = h.latent_backward(x, float(alpha), float(l), float(jitter), z, fbar)
        g_l = float(g_l_through) + 3.0 / l - 4.0
        g_z = -z + zbar
    else:
        g_alpha = None
        g_l = float(fbar @ dfdl) + 3.0 / l - 4.0
        g_z = -z + h.trmv_lower_t(L, fbar)
    g_sigma = -n / sigma + float(r @ r) / sigma ** 3
    return lp, {"l": g_l, "sigma": g_sigma, "z": g_z, "f": f, "alpha": g_alpha}


def exact_gp_log_prob_batched(x, y, l, sigma, z, alpha=1.0, jitter=1e-10, handle=None):
    """exact_gp_log_prob (reverse mode) for B parameter states in one forward and one backward call
    (gpb200_latent_forward_batched / _backward_batched): l, sigma and alpha are scalars or (B,), z is (B, n), x and y
    are (n,) or (B, n).  Returns lp (B,) and the gradients as arrays with one row per state ("l", "sigma", "alpha" (B,);
    "z", "f" (B, n)).  A state whose covariance is not positive definite gets NaN in every output; the others are
    unaffected."""
    h = handle or capi.default_handle()
    z = np.atleast_2d(np.asarray(z, dtype=np.float64))
    B, n = z.shape
    y = np.asarray(y, dtype=np.float64)
    l = np.broadcast_to(np.asarray(l, dtype=np.float64), (B,))
    sigma = np.broadcast_to(np.asarray(sigma, dtype=np.float64), (B,))
    alpha = np.broadcast_to(np.asarray(alpha, dtype=np.float64), (B,))
    f, _ = h.latent_forward_batched(x, np.stack([alpha, l], axis=1), float(jitter), z)
    r = y - f
    rr = np.einsum("bi,bi->b", r, r)
    lp = -0.5 * np.einsum("bi,bi->b", z, z) + 3.0 * np.log(l) - 4.0 * l - n * np.log(sigma) - 0.5 * rr / sigma ** 2
    fbar = r / sigma[:, None] ** 2
    tb, zbar = h.latent_backward_batched(fbar)
    g_l = tb[:, 1] + 3.0 / l - 4.0
    g_sigma = -n / sigma + rr / sigma ** 3
    return lp, {"l": g_l, "sigma": g_sigma, "z": -z + zbar, "f": f, "alpha": tb[:, 0]}
