"""Extended-precision references for the derivatives of the SE Cholesky factor -- TEST INFRASTRUCTURE ONLY.

Covers the entry points that differentiate through the factor of
    K = alpha^2 E + diag_add I,   E_ij = exp(-(x_i - x_j)^2 / (2 rho^2))   (E_ii = 1 exactly):
  * forward mode (rbf_cov_chol[_batched], se_chol_tangent): L and Ldot = dL/dtheta for theta = alpha or rho;
  * reverse mode (latent_forward / latent_backward): f_m = L z_m, zbar_m = L^T fbar_m and
    thetabar = sum_ij Kbar_ij dK_ij/dtheta with Kbar the adjoint of the Cholesky.

Forward mode, up to DUAL_MAX_N: the unblocked dual-number LLT of covariance.cpp:13-39 (as
oracle.gp_oracle.rbf_cov_chol_dual restates it), run in np.longdouble.  On x86 that is the 80-bit format with a
64-bit significand, so the reference carries 11 more bits than the float64 result it is compared with.  It costs
O(n^3) interpreted work (about 0.5 s at n = 600).  Above DUAL_MAX_N: the float64 closed form
Ldot = L Phi(L^-1 Kdot L^-T) through LAPACK.

Reverse mode (float64, LAPACK), the formulas of the header of gp_b200/csrc/api_latent.cu:
    Lbar = sum_m tril(fbar_m z_m^T),  Kbar = L^-T Phi(L^T Lbar) L^-1,  thetabar = sum Kbar o dK/dtheta.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

from oracle import gp_oracle as o

LONGDOUBLE_OK = np.finfo(np.longdouble).nmant >= 63
DUAL_MAX_N = 1100
TILE = 128


def se_gram_tangent(x, alpha, rho, diag_add, wrt, dtype=np.float64):
    """K = alpha^2 E + diag_add I and dK/dtheta: 2 alpha E for wrt == "alpha", alpha^2 E d^2 / rho^3 for
    wrt == "rho" (the length-scale l of rbf_cov_chol is rho with alpha = 1).  x is taken as float64 and widened."""
    if wrt not in ("alpha", "rho"):
        raise ValueError("wrt must be 'alpha' or 'rho'")
    x = np.asarray(x, dtype=np.float64).astype(dtype)
    alpha, rho, diag_add = dtype(alpha), dtype(rho), dtype(diag_add)
    d2 = np.subtract.outer(x, x) ** 2
    E = np.exp(-d2 / (2 * rho * rho))
    np.fill_diagonal(E, 1)
    K = alpha * alpha * E
    K[np.diag_indices_from(K)] += diag_add
    Kdot = 2 * alpha * E if wrt == "alpha" else alpha * alpha * E * d2 / rho ** 3
    return K, Kdot


def llt_dual(K, Kdot):
    """Unblocked left-looking LLT carried on (value, tangent) pairs in the dtype of K (covariance.cpp:13-39)."""
    n = K.shape[0]
    Lv = np.zeros_like(K)
    Lt = np.zeros_like(K)
    for j in range(n):
        lv, lt = Lv[j, :j], Lt[j, :j]
        sv = K[j, j] - lv @ lv
        st = Kdot[j, j] - 2 * (lv @ lt)
        if not sv > 0:
            raise o.NotPositiveDefinite("llt_dual: not positive definite", j + 1)
        dv = np.sqrt(sv)
        dt = st / (2 * dv)
        Lv[j, j], Lt[j, j] = dv, dt
        if j + 1 < n:
            cv = K[j + 1:, j] - Lv[j + 1:, :j] @ lv
            ct = Kdot[j + 1:, j] - Lv[j + 1:, :j] @ lt - Lt[j + 1:, :j] @ lv
            Lv[j + 1:, j] = cv / dv
            Lt[j + 1:, j] = (ct - Lv[j + 1:, j] * dt) / dv
    return Lv, Lt


def chol_tangent_closed_form(K, Kdot):
    """float64: L = chol(K), Ldot = L Phi(L^-1 Kdot L^-T)."""
    L = o.cholesky_decompose(K)
    T = sla.solve_triangular(L, Kdot, lower=True, check_finite=False)
    A = sla.solve_triangular(L, T.T, lower=True, check_finite=False).T
    return L, np.tril(L @ o.phi_lower(A))


def chol_tangent(x, alpha, rho, diag_add, wrt):
    """(L, Ldot) as float64 arrays: the longdouble dual LLT up to DUAL_MAX_N (raises when long double is not
    the 64-bit-significand format), the float64 closed form above."""
    n = len(x)
    if n > DUAL_MAX_N:
        return chol_tangent_closed_form(*se_gram_tangent(x, alpha, rho, diag_add, wrt))
    if not LONGDOUBLE_OK:
        raise RuntimeError("np.longdouble carries %d mantissa bits; the dual LLT needs 63" % np.finfo(np.longdouble).nmant)
    Lv, Lt = llt_dual(*se_gram_tangent(x, alpha, rho, diag_add, wrt, np.longdouble))
    return Lv.astype(np.float64), Lt.astype(np.float64)


def latent_adjoint(x, alpha, rho, diag_add, z, fbar):
    """Reverse sweep through f_m = L z_m and the Cholesky for general z_m, fbar_m (rows of z, fbar).
    Returns a dict: L, f (nvec x n), zbar (nvec x n), theta_bar = (d/dalpha, d/drho), scale = (sum |Kbar o dK/dalpha|,
    sum |Kbar o dK/drho|) -- the size of the terms theta_bar sums, for a tolerance -- and the term matrices
    terms = (Kbar o dK/dalpha, Kbar o dK/drho)."""
    z = np.atleast_2d(np.asarray(z, dtype=np.float64))
    fbar = np.atleast_2d(np.asarray(fbar, dtype=np.float64))
    K, dKa = se_gram_tangent(x, alpha, rho, diag_add, "alpha")
    _, dKr = se_gram_tangent(x, alpha, rho, diag_add, "rho")
    L = o.cholesky_decompose(K)
    Lbar = np.tril(fbar.T @ z)
    P = o.phi_lower(L.T @ Lbar)
    T = sla.solve_triangular(L, P, lower=True, trans="T", check_finite=False)           # L^-T P
    Kbar = sla.solve_triangular(L, T.T, lower=True, trans="T", check_finite=False).T    # L^-T P L^-1
    terms = (Kbar * dKa, Kbar * dKr)
    return {"L": L, "f": z @ L.T, "zbar": fbar @ L,
            "theta_bar": np.array([t.sum() for t in terms]),
            "scale": np.array([np.abs(t).sum() for t in terms]),
            "terms": terms}


def tile_blocks(n):
    """(I, J, row slice, column slice) of the 128 x 128 tiles of an n x n matrix."""
    nt = (n + TILE - 1) // TILE
    for I in range(nt):
        for J in range(nt):
            yield I, J, slice(I * TILE, (I + 1) * TILE), slice(J * TILE, (J + 1) * TILE)


def far_gap(n):
    """Tile distance that counts as far: 2, or 1 when the matrix has only two tile rows."""
    return 2 if n > 2 * TILE else 1


def far_tile_share(A, gap=None):
    """Largest |entry| over the tile pairs at least `gap` apart (|I - J| >= gap, default far_gap(n)), relative to
    the largest |entry|."""
    A = np.abs(np.asarray(A, dtype=np.float64))
    gap = far_gap(A.shape[0]) if gap is None else gap
    far = max((float(A[r, c].max()) for I, J, r, c in tile_blocks(A.shape[0]) if abs(I - J) >= gap), default=0.0)
    return far / max(float(A.max()), 1e-300)


def far_tile_sum(A):
    """Sum of the entries over the tile pairs at least far_gap(n) apart."""
    A = np.asarray(A, dtype=np.float64)
    gap = far_gap(A.shape[0])
    return sum(float(A[r, c].sum()) for I, J, r, c in tile_blocks(A.shape[0]) if abs(I - J) >= gap)


def worst_tile(err):
    """(I, J) of the tile that holds the largest entry of err."""
    i, j = np.unravel_index(int(np.argmax(err)), err.shape)
    return int(i) // TILE, int(j) // TILE
