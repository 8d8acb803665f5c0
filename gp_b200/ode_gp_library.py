"""Host-side mirror of R/ode_gp_library.R (and of the older R/ode_gp.R): the conditioning API.

p_Xn / p_dotXn keep the reference signatures (tn, Xn, phi_n, sigma_n) and return what
condMVNorm::condMVN returns, {"condMean", "condVar"} (R/ode_gp_library.R:17,32).  UU/UD/DD, which
the reference never defines, are QQ/QR/RR of R/kernels.R as R/ode_gp.R:5-8,23-26 shows
(SURVEY Appendix A.2).  p_dotXn_mnKn is the R/ode_gp.R:19-32 variant returning {"mn", "Kn"}.
sample_derivs is pendulum_fit.R:227-255.  The joint matrix is assembled by one Gram kernel and
conditioned by the tiled Cholesky; nothing is computed on the host.
"""
from __future__ import annotations

import numpy as np
import scipy.linalg as sla

from . import capi


def condMVN(mean, sigma, dependent_ind, given_ind, X_given, handle=None):
    """condMVNorm::condMVN for the layout the reference uses: given indices 0..ng-1 first, dependent
    indices ng..N-1 after (R/ode_gp_library.R:17: condMVN(m, K, (N+1):(2*N), 1:N, Xn))."""
    ng = len(given_ind)
    N = np.asarray(sigma).shape[0]
    if list(given_ind) != list(range(ng)) or list(dependent_ind) != list(range(ng, N)):
        raise capi.GpB200Error("condMVN: only the reference's block layout (given block first) is supported")
    cm, cv = (handle or capi.default_handle()).cond_mvn(mean, sigma, ng, X_given)
    return {"condMean": cm, "condVar": cv}


def p_dotXn(tn, Xn, phi_n, sigma_n, quirk=True, handle=None):  # R/ode_gp_library.R:23-33
    h = handle or capi.default_handle()
    tn = np.asarray(tn, dtype=np.float64)
    n = tn.shape[0]
    K = h.gram_deriv(tn, float(phi_n[0]), float(phi_n[1]), [float(sigma_n), 0.0], 1e-6, nblocks=2, quirk=quirk)
    cm, cv = h.cond_mvn(np.zeros(2 * n), K, n, Xn)
    return {"condMean": cm, "condVar": cv}


def p_Xn(tn, Xn, phi_n, sigma_n, handle=None):  # R/ode_gp_library.R:3-18
    h = handle or capi.default_handle()
    tn = np.asarray(tn, dtype=np.float64)
    n = tn.shape[0]
    UU = h.gram_outer("QQ", tn, tn, float(phi_n[1]), float(phi_n[0]) ** 2)
    K = np.empty((2 * n, 2 * n), order="F")
    K[:n, :n] = UU + float(sigma_n) ** 2 * np.eye(n)
    K[:n, n:] = UU.T
    K[n:, :n] = UU.T
    K[n:, n:] = UU
    K[np.diag_indices(2 * n)] += 1e-6
    cm, cv = h.cond_mvn(np.zeros(2 * n), K, n, Xn)
    return {"condMean": cm, "condVar": cv}


def p_dotXn_mnKn(tn, Xn, phi_n, sigma_n, quirk=True, handle=None):  # R/ode_gp.R:19-32
    h = handle or capi.default_handle()
    a2, l = float(phi_n[0]) ** 2, float(phi_n[1])
    QQ = h.gram_outer("QQ", tn, tn, l, a2)
    RQ = h.gram_outer("QR", tn, tn, l, a2).T
    RR = h.gram_outer("RR_QUIRK" if quirk else "RR", tn, tn, l, a2)
    mn, Kn = h.gp_condition(QQ, RQ, RR, Xn, float(sigma_n) ** 2, 0.0)
    return {"mn": mn, "Kn": Kn}


def sample_derivs_moments(params, ynoise, ti, handle=None):
    """pendulum_fit.R:227-251: params = (l, a, sy); returns build_mu / build_cov."""
    h = handle or capi.default_handle()
    l, a, sy = (float(v) for v in params)
    K = h.gram_outer("QQ", ti, ti, l, a * a)
    KsK = h.gram_outer("RQ", ti, ti, l, a * a)
    KsKs = h.gram_outer("RR", ti, ti, l, a * a)
    return h.gp_condition(K, KsK, KsKs, ynoise, sy * sy, 1e-8)


def sample_derivs(params, ynoise, ti, rng=None, seed=None, handle=None):
    """pendulum_fit.R:227-255 including the MASS::mvrnorm(1, mu, Sigma) draw (:253): the draw is
    mu + L z with L the GPU Cholesky factor of the posterior covariance.  With `seed` the normals come
    from the device generator (gpb200_mvrnorm: Philox, reproducible per seed); with `rng` (a NumPy
    Generator) they are drawn on the host and only the factorisation and L z run on the GPU."""
    h = handle or capi.default_handle()
    mu, cov = sample_derivs_moments(params, ynoise, ti, handle=h)
    if seed is not None:
        return h.mvrnorm(1, mu, cov, int(seed))
    rng = rng or np.random.default_rng()
    L = h.potrf(cov)
    return mu + h.trmv_lower(L, rng.standard_normal(mu.shape[0]))


def sample_derivs_draws(params, ynoise, ti, seed=None, rng=None, handle=None):
    """The loop of pendulum_fit.R:259-268 over sample_derivs, batched: one draw of the posterior derivative per
    row of params = (l, a, sy) (B, 3), in one call (gpb200_posterior_draws_batched, order 1, predicting on ti,
    jitter 1e-8).  ynoise: (n,) shared or (B, n).  Normals: the device stream of `seed`, or drawn on the host from
    `rng` (a NumPy Generator; a fresh one when both are None).  Returns a (B, n) array."""
    p = np.asarray(params, dtype=np.float64)
    if p.ndim != 2 or p.shape[1] != 3:
        raise ValueError("sample_derivs_draws: params must be (B, 3) = (l, a, sy) per row")
    ti = np.asarray(ti, dtype=np.float64)
    y = np.asarray(ynoise, dtype=np.float64)
    if ti.ndim != 1 or y.ndim not in (1, 2) or y.shape[-1] != ti.shape[0] or (y.ndim == 2 and y.shape[0] != p.shape[0]):
        raise ValueError("sample_derivs_draws: ynoise must be (n,) or (B, n) with n = len(ti)")
    h = handle or capi.default_handle()
    theta = p[:, [1, 0, 2]]  # (l, a, sy) -> (alpha, rho, sigma)
    z = None
    if seed is None:
        z = (rng or np.random.default_rng()).standard_normal((p.shape[0], ti.shape[0]))
    draws, _, info = h.posterior_draws_batched(ti, y, theta, order=1, jitter=1e-8, seed=seed, z=z)
    bad = np.flatnonzero(info)
    if bad.size:
        raise capi.NotPositiveDefiniteError("sample_derivs_draws (item %d)" % bad[0], int(info[bad[0]]))
    return draws


def create_p_dotXnS(Xn_list, mn, Kn, theta, rng=None, handle=None, incremental=True):
    """R/ode_gp_library.R:43-93: closure that, given a new state x*, returns the conditional normal
    of the derivative there given the data and every derivative already drawn, then draws from it.

    Same values as the R text, less work per call (incremental=True, the default; row f-4 of SURVEY 8): the reference
    rebuilds the whole i x i joint covariance of the star points, re-solves all i cross-covariance columns against
    K_XX and inverts the (i-1) x (i-1) leading block inside condMVN on EVERY call (O(i N^2 + i^3)).  Here each call
    solves only for the NEW column (one GPU potrs, N^2) and extends the lower Cholesky factor of the star points'
    covariance by one row -- a bordered ("rank-1 growth") update, O(i^2) -- from which the conditional mean and
    variance of the new point given all earlier draws drop out:  l = Lc^-1 k,  mean = m_i + l.w,  var = k_ii - l.l,
    with w = Lc^-1 (dot_Xs - m) grown the same way.  incremental=False is the literal re-solve (kept for the test).

    Other differences from the R text, all benign: the pre-factorisation of K_XX + 1e-6 I is a GPU Cholesky instead
    of qr() (:55-57); `rnorm(1, mean, condVar)` passes a VARIANCE as sd (:84, SURVEY Appendix A.3) -- reproduced by
    default (sd_is_variance=True on the returned closure).  Each call returns {"mu", "sigma", "dot_xs"} (:91).
    """
    h = handle or capi.default_handle()
    rng = rng or np.random.default_rng()
    X = np.column_stack([np.asarray(c, dtype=np.float64) for c in Xn_list])
    N, D = X.shape
    mn = np.asarray(mn, dtype=np.float64)
    Kn = np.asarray(Kn, dtype=np.float64)
    K_XX = h.gram_ard(X, X, float(theta[0]), theta[1])
    L = h.potrf(K_XX + 1e-6 * np.eye(N))
    K_XX_1_mn = h.potrs(L, mn)
    K_XX_1_Kn = h.potrs(L, Kn)
    state = {"i": 1, "K_XsX": np.zeros((0, N)), "K_XsXs": np.zeros((0, 0)), "Xs": np.zeros((0, D)),
             "dot_Xs": np.zeros(0), "S": np.zeros((N, 0)), "Lc": np.zeros((0, 0)), "w": np.zeros(0)}

    def step_literal(xs, st):
        st["K_XsX"] = np.vstack([st["K_XsX"], h.gram_ard(xs, X, float(theta[0]), theta[1])])
        kss = h.gram_ard(xs, xs, float(theta[0]), theta[1])
        if st["Xs"].shape[0]:
            cross = h.gram_ard(st["Xs"], xs, float(theta[0]), theta[1])
            st["K_XsXs"] = np.block([[st["K_XsXs"], cross], [cross.T, kss]])
        else:
            st["K_XsXs"] = kss
        A = st["K_XsX"]
        S = h.potrs(L, np.asfortranarray(A.T))            # solve(K_XX_qr, t(K_XsX))
        m = A @ K_XX_1_mn
        K = st["K_XsXs"] - A @ S + A @ K_XX_1_Kn @ S
        K = (K + K.T) / 2 + 1e-6 * np.eye(K.shape[0])
        i = st["i"]
        if i == 1:
            return m[0], K[0, 0]
        # condMVN(m, K, i, 1:(i-1), c(dot_Xs)): last point given all earlier draws
        cm, cv = h.cond_mvn(m, K, i - 1, st["dot_Xs"])
        return cm[0], cv[0, 0]

    def step_incremental(xs, st):
        i = st["i"]
        a = h.gram_ard(xs, X, float(theta[0]), theta[1])              # 1 x N
        s = h.potrs(L, a.ravel().copy())                              # the NEW column of solve(K_XX, t(K_XsX))
        A = np.vstack([st["K_XsX"], a])
        S = np.column_stack([st["S"], s])
        m_new = float(a.ravel() @ K_XX_1_mn)
        kss = h.gram_ard(st["Xs"], xs, float(theta[0]), theta[1]).ravel() if st["Xs"].shape[0] else np.zeros(0)
        kself = float(h.gram_ard(xs, xs, float(theta[0]), theta[1])[0, 0])
        aK = a @ K_XX_1_Kn                                            # 1 x N
        left = (a @ S - aK @ S).ravel()                               # row i of  K_XsX (I - K_XX^-1 Kn) K_XX^-1 K_XXs
        right = (A @ s - A @ (K_XX_1_Kn @ s)).ravel()                 # column i of the same (not symmetric before averaging)
        krow = np.concatenate([kss, [kself]]) - 0.5 * (left + right)
        krow[i - 1] += 1e-6
        if i == 1:
            l_row = np.zeros(0)
            cmean, cvar = m_new, krow[0]
        else:
            l_row = sla.solve_triangular(st["Lc"], krow[:i - 1], lower=True, check_finite=False)
            cmean = m_new + float(l_row @ st["w"])
            cvar = krow[i - 1] - float(l_row @ l_row)
        if not cvar > 0.0:
            # the bordered factor's new pivot: the joint covariance of the star points is not positive definite
            # (condMVN's explicit inverse would go on and return a negative variance, SURVEY Appendix A)
            raise capi.NotPositiveDefiniteError("create_p_dotXnS", i)
        st["K_XsX"], st["S"] = A, S
        st["_pending"] = (l_row, cvar, cmean)
        return cmean, cvar

    def p_dotXnS(xs_vec, sd_is_variance=True):
        xs = np.asarray(xs_vec, dtype=np.float64).reshape(1, D)
        st = state
        cmean, cvar = (step_incremental if incremental else step_literal)(xs, st)
        sd = cvar if sd_is_variance else np.sqrt(max(cvar, 0.0))
        dot_xs = cmean + sd * rng.standard_normal()
        i = st["i"]
        if incremental:
            l_row, cv, cm = st.pop("_pending")
            d = np.sqrt(max(cv, 0.0))
            Lc = np.zeros((i, i))
            Lc[:i - 1, :i - 1] = st["Lc"]
            Lc[i - 1, :i - 1] = l_row
            Lc[i - 1, i - 1] = d
            st["Lc"] = Lc
            st["w"] = np.append(st["w"], (dot_xs - cm) / d if d > 0 else 0.0)
        st["i"] = i + 1
        st["Xs"] = np.vstack([st["Xs"], xs])
        st["dot_Xs"] = np.append(st["dot_Xs"], dot_xs)
        return {"mu": float(cmean), "sigma": float(cvar), "dot_xs": float(dot_xs)}

    return p_dotXnS
