"""CPU tests of the oracle itself (runs everywhere, no GPU):
  * the NumPy restatement against the golden vectors produced by the reference's OWN gp_derivs.py
    (tests/golden/make_golden.py) -- the only reference-generated numbers that exist for this path;
  * NumPy <-> plain-C <-> mpmath (50 digits) cross-checks for the Stan-Math rows, which the reference
    does not pin ("parity unpinned", SURVEY 8c);
  * analytic gradient vs central finite differences; forward-mode Cholesky tangent vs the literal
    dual-number LLT of covariance.cpp:13-29; Hermite end-point identities (cubic_spline_test.R)."""
import numpy as np
import pytest

from oracle import c_oracle as c
from oracle import gp_oracle as o


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


@pytest.mark.parametrize("name", ["QQ", "QR", "RQ", "RR", "QT", "TQ", "RT", "TR", "TT"])
def test_oracle_kernels_match_reference_golden(golden, name):
    ts, tts, l, a = golden["ts"], golden["tts"], float(golden["l"]), float(golden["a"])
    assert relerr(a * a * o.outer_kernel(name, tts, ts, l), golden["kern_" + name]) < 1e-14
    assert relerr(c.outer_kernel(name, tts, ts, l, a * a), golden["kern_" + name]) < 1e-14


def test_oracle_conditioning_matches_reference_golden(golden):
    s = float(golden["s"])
    mu, cov = o.gp_condition(golden["K"], golden["KsK"], golden["KsKs"], golden["y"], s * s, 0.0)
    assert relerr(mu, golden["mu_d"]) < 1e-12 and relerr(cov, golden["cov_d"]) < 1e-12
    mu, cov = o.gp_condition(golden["K"], golden["KsKi"], golden["KsKsi"], golden["y"], s * s, 0.0)
    assert relerr(mu, golden["mu_i"]) < 1e-12 and relerr(cov, golden["cov_i"]) < 1e-12
    # known closed-form spot values quoted in SURVEY 8c: TT(0,0) = 3, RR(0,0.5) = 0.66187...
    assert o.dk_TT(0.0, 0.0, 1.0) == 3.0
    assert abs(o.dk_RR(0.0, 0.5, 1.0) - 0.75 * np.exp(-0.125)) < 1e-15


def test_numpy_c_mpmath_agree_on_lml_and_gradient():
    from oracle import gp_oracle_mp as m
    rng = np.random.default_rng(1)
    x = np.linspace(0, 10, 48)
    y = np.sin(x) + 0.2 * rng.standard_normal(48)
    for th in ([1.1, 0.8, 0.3], [0.6, 1.7, 0.15]):
        v, g = o.lml_grad(x, y, *th)
        v2, g2, info = c.lml_grad(x, y, th)
        v3, g3 = m.lml_grad(x, y, *th)
        assert info == 0
        assert abs(v - v3) < 1e-11 * abs(v3) and abs(v2 - v3) < 1e-11 * abs(v3)
        assert relerr(g, g3) < 1e-10 and relerr(g2, g3) < 1e-10


def test_gradient_matches_finite_differences():
    x, y = o.synth_xy(100, 3)
    th = np.array([1.0, 1.0, 0.3])
    _, g = o.lml_grad(x, y, *th)
    for k in range(3):
        tp, tm = th.copy(), th.copy()
        tp[k] += 1e-6; tm[k] -= 1e-6
        fd = (o.lml(x, y, *tp) - o.lml(x, y, *tm)) / 2e-6
        assert abs(fd - g[k]) < 1e-6 * max(1, abs(g[k]))


def test_c_oracle_matches_numpy_at_moderate_n():
    x, y = o.synth_xy(300, 5)
    th = o.synth_theta(4, 9)
    out = c.lml_grad_draws(x, y, th, nthreads=2)
    for b in range(4):
        v, g = o.lml_grad(x, y, *th[b])
        assert abs(out[b, 0] - v) < 1e-10 * abs(v)
        assert relerr(out[b, 1:4], g) < 1e-9
        assert out[b, 4] == 0
    K = o.gram_se(x, 1.0, 1.0, 0.09)
    assert relerr(c.cov_exp_quad(x, 1.0, 1.0) + 0.09 * np.eye(300), K) < 1e-15
    L, info = c.llt(K)
    assert info == 0 and relerr(L, o.cholesky_decompose(K)) < 1e-11


def test_cholesky_semantics():
    K = o.gram_se(np.linspace(0, 1, 20), 1.0, 0.5, 1e-3)
    L = o.cholesky_decompose(K)
    assert np.all(np.triu(L, 1) == 0)
    Kbad = K.copy(); Kbad[3, 7] += 1e-6
    with pytest.raises(o.NotPositiveDefinite):
        o.cholesky_decompose(Kbad)          # symmetry check (abs tol 1e-8)
    Kneg = K.copy(); Kneg[10, 10] = -1.0
    with pytest.raises(o.NotPositiveDefinite) as ei:
        o.cholesky_decompose(Kneg)
    assert ei.value.info == 11
    _, info = c.llt(Kneg)
    assert info == 11
    # cov_exp_quad puts alpha^2 exactly on the diagonal
    assert np.all(np.diag(o.cov_exp_quad(np.linspace(0, 3, 9), 1.7, 0.3)) == 1.7 * 1.7)


def test_rbf_cov_chol_closed_form_vs_literal_duals():
    xs = np.arange(14) * 0.8
    L, dL = o.rbf_cov_chol(xs, 0.5)
    L2, dL2 = o.rbf_cov_chol_dual(xs, 0.5)
    L3, dL3, info = c.rbf_cov_chol(xs, 0.5)
    assert info == 0
    assert relerr(L, L2) < 1e-12 and relerr(dL, dL2) < 1e-10
    assert relerr(L3, L2) < 1e-13 and relerr(dL3, dL2) < 1e-12
    h = 1e-6
    Lp, _ = o.rbf_cov_chol(xs, 0.5 + h); Lm, _ = o.rbf_cov_chol(xs, 0.5 - h)
    assert relerr((Lp - Lm) / (2 * h), dL) < 1e-6


def test_hermite_identities_cubic_spline_test_constants():
    # cubic_spline_test.R:4-18 : y1=5, y2=2, k1=-5, k2=3, x1=1, x2=1.75
    y1, y2, k1, k2, x1, x2 = 5.0, 2.0, -5.0, 3.0, 1.0, 1.75
    lp = [x1, x2]
    Ls = [np.array([[y1]]), np.array([[y2]])]
    dLs = [np.array([[k1]]), np.array([[k2]])]
    assert o.approx_L(x1, lp, Ls, dLs)[0, 0] == y1
    assert abs(o.approx_L(x2, lp, Ls, dLs)[0, 0] - y2) < 1e-15
    z = np.array([1.0])
    h = 1e-6
    for x, k in ((x1, k1), (x2, k2)):
        _, d = o.approx_Lz(x, lp, Ls, dLs, z)
        assert abs(d[0] - k) < 1e-12
    v1, d1 = o.approx_Lz(1.3, lp, Ls, dLs, z)
    vp, _ = o.approx_Lz(1.3 + h, lp, Ls, dLs, z); vm, _ = o.approx_Lz(1.3 - h, lp, Ls, dLs, z)
    assert abs((vp[0] - vm[0]) / (2 * h) - d1[0]) < 1e-7


def test_condmvn_and_p_dotXn_consistency():
    tn = np.arange(-2, 2.0001, 0.2)
    Xn = np.exp(tn)
    # with alpha = 1 the R/kernels.R quirk vanishes and the two API generations agree up to the 1e-6 jitter
    cm, cv = o.p_dotXn(tn, Xn, (1.0, 0.9), 0.1)
    mn, Kn = o.p_dotXn_solve(tn, Xn, (1.0, 0.9), 0.1)
    assert relerr(cm, mn) < 1e-3
    assert cm.shape == (len(tn),) and cv.shape == (len(tn), len(tn))
    assert relerr(o.rk_RR(tn, tn, (1.0, 0.9), True), o.rk_RR(tn, tn, (1.0, 0.9), False)) == 0.0
    assert relerr(o.rk_RR(tn, tn, (1.5, 0.9), True), o.rk_RR(tn, tn, (1.5, 0.9), False)) > 1e-3


def test_lp_matches_lml_plus_priors():
    x, y = o.synth_xy(50, 1)
    lp = o.lp_fit_hyperparameters(x, y, np.log(0.9), np.log(1.2), np.log(0.3))
    base = o.lml(x, y, 1.2, 0.9, 0.3, drop_constants=True)
    extra = 3 * np.log(0.9) - 4 * 0.9 - 0.5 * 1.2 ** 2 - 0.5 * 0.3 ** 2 + np.log(0.9) + np.log(1.2) + np.log(0.3)
    assert abs(lp - (base + extra)) < 1e-12


def test_lapack_route_matches_plain_route():
    x, y = o.synth_xy(400, 3)
    for th in o.synth_theta(3, 1):
        v, g = o.lml_grad(x, y, *th)
        v2, g2 = o.lml_grad_lapack(x, y, *th)
        assert abs(v - v2) < 1e-12 * abs(v) and relerr(g2, g) < 1e-11


def test_latent_gp_reverse_mode_adjoint_matches_finite_differences():
    rng = np.random.default_rng(0)
    x = np.arange(30) * 0.8
    y = np.sin(x) + 0.1 * rng.standard_normal(30)
    z = rng.standard_normal(30)
    lp, g = o.exact_gp_lp_grad(x, y, 0.9, 0.3, z)
    h = 1e-6
    fd_l = (o.exact_gp_lp_grad(x, y, 0.9 + h, 0.3, z)[0] - o.exact_gp_lp_grad(x, y, 0.9 - h, 0.3, z)[0]) / (2 * h)
    fd_s = (o.exact_gp_lp_grad(x, y, 0.9, 0.3 + h, z)[0] - o.exact_gp_lp_grad(x, y, 0.9, 0.3 - h, z)[0]) / (2 * h)
    assert abs(fd_l - g["l"]) < 1e-6 * abs(g["l"]) and abs(fd_s - g["sigma"]) < 1e-6 * abs(g["sigma"])


def test_oracle_matches_reference_ch2_golden(ch2_golden):
    # the reference's ch2.py:55-91 in its l2 parametrisation: alpha^2 = eta2, rho = sqrt(l2 / 2)
    g = ch2_golden
    phi = (float(np.sqrt(g["eta2"])), float(np.sqrt(g["l2"] / 2.0)))
    xs, xd, idx = g["xs"], g["xd"], g["idx"]
    assert relerr(o.rk_QQ(xs, xd, phi), g["Ksd"]) < 1e-13
    assert relerr(o.rk_QQ(xs[idx], xs[idx], phi), g["Kss_sub"]) < 1e-13
    mu, cov = o.gp_condition(g["Kdd"], g["Ksd"], o.rk_QQ(xs, xs, phi), g["f"], 0.0, 0.0)
    assert relerr(mu, g["m"]) < 1e-10
    assert np.max(np.abs(cov[np.ix_(idx, idx)] - g["Kt_sub"])) < 1e-10


def test_westbrook_fixture_shape(westbrook):
    x = westbrook["x"]
    assert x.shape == (1438,) and len(np.unique(x)) == 1073 and abs(x.min() + 0.4976) < 1e-3 and x.max() == 0.5
    # duplicated inputs: the exact-GP Gram is singular without jitter (SURVEY 2.1 "Data")
    assert o.potrf_info(o.gram_se(x, 1.0, 0.3, 0.0)) > 0


# ---- derivative-observation LML (gpderivs.py:62-83; design_notes.Rmd:25-46) ------------------------
def test_kernel_length_scale_derivatives_match_central_differences():
    rng = np.random.default_rng(0)
    a = rng.uniform(0, 3, 64); b = rng.uniform(0, 3, 64)
    l, h = 0.9, 1e-6
    for name, f in o.DERIV_KERNELS.items():
        fd = (f(a, b, l + h) - f(a, b, l - h)) / (2 * h)
        an = o.DERIV_KERNELS_DL[name](a, b, l)
        assert np.max(np.abs(fd - an)) <= 1e-8 * np.max(np.abs(an)), name


def test_lml_grad_deriv_gradient_vs_finite_differences_and_reference_parametrisation():
    rng = np.random.default_rng(1)
    t = np.linspace(0, 5, 40)
    y = np.concatenate([np.sin(t), np.cos(t), -np.sin(t)]) + 0.1 * rng.standard_normal(120)
    th = np.array([1.2, 0.8, 0.1, 0.2, 0.3])
    v, g = o.lml_grad_deriv(t, y, th[0], th[1], th[2:], 1e-6)
    for i in range(5):
        tp = th.copy(); tm = th.copy(); tp[i] += 1e-6; tm[i] -= 1e-6
        fd = (o.lml_grad_deriv(t, y, tp[0], tp[1], tp[2:], 1e-6)[0] - o.lml_grad_deriv(t, y, tm[0], tm[1], tm[2:], 1e-6)[0]) / 2e-6
        assert abs(fd - g[i]) <= 1e-6 * max(1.0, abs(g[i]))
    # the reference's own covdd in its l2 parametrisation (gpderivs.py:35-37), typed out literally
    sf2, l2, s2 = 1.3, 2.2, 0.04
    d = t[:, None] - t[None, :]
    Sigma = sf2 * 2 * np.exp(-d ** 2 / l2) * (l2 - 2 * d ** 2) / l2 ** 2 + s2 * np.eye(40)
    dx = np.cos(t) + 0.15 * rng.standard_normal(40)
    ref = -0.5 * (40 * np.log(2 * np.pi) + np.linalg.slogdet(Sigma)[1] + dx @ np.linalg.solve(Sigma, dx))
    v, g = o.gpderivs_log_prob_grad(t, dx, sf2, l2, s2)
    assert abs(v - ref) <= 1e-10 * abs(ref)
    for i, hh in enumerate(np.eye(3) * 1e-6):
        fd = (o.gpderivs_log_prob_grad(t, dx, *(np.array([sf2, l2, s2]) + hh))[0] -
              o.gpderivs_log_prob_grad(t, dx, *(np.array([sf2, l2, s2]) - hh))[0]) / 2e-6
        assert abs(fd - g[i]) <= 1e-6 * max(1.0, abs(g[i]))


# ---- f-4: the device random-number stream restated (oracle/philox.py) -------------------------------
def test_philox_known_answer_and_normal_moments():
    from oracle import philox
    # Random123 known-answer vector: philox4x32-10, counter = 0, key = 0
    r = philox.philox4x32_10(np.array([0], dtype=np.uint64), 0)
    assert [int(v) for v in r[0]] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    z = philox.normals(42, 200001)
    assert abs(z.mean()) < 0.01 and abs(z.std() - 1.0) < 0.01
    assert abs(np.mean(z ** 3)) < 0.03 and abs(np.mean(z ** 4) - 3.0) < 0.06
    assert np.array_equal(philox.normals(42, 100, offset=1000), philox.normals(42, 1100)[1000:])
    assert not np.array_equal(philox.normals(43, 100), z[:100])


# ---- independent third-party corroboration of the "parity unpinned" rows (a4-a7) ---------------------
def test_lml_and_gradient_agree_with_scikit_learn_gpr():
    """The reference pins no output for the Stan-Math rows and Stan Math cannot run here, so besides
    NumPy <-> C <-> mpmath <-> finite differences the oracle is checked against an independent,
    widely used implementation of the same quantity: scikit-learn's GaussianProcessRegressor
    (ConstantKernel * RBF + WhiteKernel = alpha^2 exp(-d^2 / 2 rho^2) + sigma^2 I), whose
    log_marginal_likelihood(theta, eval_gradient=True) works in log-parameters."""
    pytest.importorskip("sklearn")
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel, WhiteKernel
    for n, (a, r, s) in ((100, (1.0, 1.0, 0.2)), (257, (1.3, 0.8, 0.25)), (400, (0.6, 2.1, 0.45))):
        x, y = o.synth_xy(n, 3)
        k = ConstantKernel(a * a) * RBF(r) + WhiteKernel(s * s)
        g = GaussianProcessRegressor(k, alpha=0.0, optimizer=None).fit(x[:, None], y)
        v, gr = g.log_marginal_likelihood(np.log([a * a, r, s * s]), eval_gradient=True)
        rv, rg = o.lml_grad(x, y, a, r, s)
        assert abs(v - rv) <= 1e-11 * abs(rv)
        chain = np.array([rg[0] * a / 2.0, rg[1] * r, rg[2] * s / 2.0])   # d/dlog(alpha^2), d/dlog(rho), d/dlog(sigma^2)
        assert np.max(np.abs(gr - chain)) <= 1e-9 * np.max(np.abs(chain))
        rv2, rg2 = o.lml_grad_lapack(x, y, a, r, s)
        assert abs(v - rv2) <= 1e-11 * abs(rv2) and np.max(np.abs(rg2 - rg)) <= 1e-9 * np.max(np.abs(rg))


# ---- property-based checks of the restatement (hypothesis) -------------------------------------------
def test_oracle_properties_hold_for_random_inputs():
    """Size-independent properties of the LML path, over random sizes / inputs / hyper-parameters:
    permutation invariance, gradient vs central differences, the sigma-gradient identity
    alpha dL/dalpha + sigma dL/dsigma = y^T K^-1 y - n (K is homogeneous of degree 2 in (alpha, sigma)),
    and NumPy <-> C agreement."""
    hyp = pytest.importorskip("hypothesis")
    from hypothesis import given, settings, strategies as st
    from oracle import c_oracle as c

    @settings(max_examples=25, deadline=None, derandomize=True)
    @given(n=st.integers(2, 60), seed=st.integers(0, 10_000), alpha=st.floats(0.3, 2.0), rho=st.floats(0.3, 3.0),
           sigma=st.floats(0.1, 0.8))
    def check(n, seed, alpha, rho, sigma):
        rng = np.random.default_rng(seed)
        x = np.sort(rng.uniform(0, 0.3 * n, n)); y = rng.standard_normal(n)
        v, g = o.lml_grad(x, y, alpha, rho, sigma)
        perm = rng.permutation(n)
        vp, gp = o.lml_grad(x[perm], y[perm], alpha, rho, sigma)
        assert abs(v - vp) <= 1e-10 * max(1.0, abs(v)) and np.max(np.abs(g - gp)) <= 1e-8 * max(1.0, np.max(np.abs(g)))
        th = np.array([alpha, rho, sigma])
        for i in range(3):
            h = 1e-6 * th[i]
            tp, tm = th.copy(), th.copy(); tp[i] += h; tm[i] -= h
            fd = (o.lml(x, y, *tp) - o.lml(x, y, *tm)) / (2 * h)
            assert abs(fd - g[i]) <= 2e-5 * max(1.0, abs(g[i]))
        K = o.gram_se(x, alpha, rho, sigma * sigma)
        quad = float(y @ np.linalg.solve(K, y))
        assert abs(alpha * g[0] + sigma * g[2] - (quad - n)) <= 1e-8 * max(1.0, abs(quad))
        cv, cg, info = c.lml_grad(x, y, th)
        assert info == 0 and abs(cv - v) <= 1e-10 * max(1.0, abs(v)) and np.max(np.abs(cg - g)) <= 1e-8 * max(1.0, np.max(np.abs(g)))

    check()


# ---- extended-precision references of the Cholesky derivatives (oracle/chol_deriv_ext.py) ---------------------
def _need_longdouble():
    from oracle import chol_deriv_ext as X
    if not X.LONGDOUBLE_OK:
        pytest.skip("np.longdouble has %d mantissa bits here; the dual LLT reference needs 63" % np.finfo(np.longdouble).nmant)
    return X


def test_longdouble_dual_llt_matches_float64_duals_and_mpmath():
    X = _need_longdouble()
    from oracle import gp_oracle_mp as m
    # rbf_cov_chol's inputs: the float64 literal duals agree to rounding
    xs = np.random.default_rng(4).permutation(30).astype(float)
    L, dL = X.chol_tangent(xs, 1.0, 0.7, o.RBF_JITTER, "rho")
    L2, dL2 = o.rbf_cov_chol_dual(xs, 0.7)
    assert relerr(L, L2) < 1e-14 and relerr(dL, dL2) < 1e-13
    # dense SE inputs, both tangents: the 50-digit duals agree to the float64 rounding of the result
    x = np.sort(np.random.default_rng(5).uniform(0, 10, 36))
    for wrt in ("alpha", "rho"):
        L, dL = X.chol_tangent(x, 1.3, 2.0, 0.1, wrt)
        Lm, dLm = m.chol_tangent(x, 1.3, 2.0, 0.1, wrt)
        assert relerr(L, Lm) < 4e-16 and relerr(dL, dLm) < 4e-16, wrt
        assert np.all(np.triu(L, 1) == 0) and np.all(np.triu(dL, 1) == 0)


def test_longdouble_dual_llt_matches_closed_form_at_n300():
    X = _need_longdouble()
    x = np.sort(np.random.default_rng(6).uniform(0, 10, 300))
    for wrt in ("alpha", "rho"):
        L, dL = X.chol_tangent(x, 1.3, 2.0, 0.1, wrt)
        Lc, dLc = X.chol_tangent_closed_form(*X.se_gram_tangent(x, 1.3, 2.0, 0.1, wrt))
        assert relerr(L, Lc) < 1e-13 and relerr(dL, dLc) < 1e-12, wrt
    assert X.far_tile_share(L) >= 1e-2 and X.far_tile_share(dL) >= 1e-2


def test_latent_adjoint_matches_central_differences():
    from oracle import chol_deriv_ext as X
    rng = np.random.default_rng(7)
    n, theta, da = 200, np.array([1.3, 1.5]), 0.1
    x = np.sort(rng.uniform(0, 10, n))
    z = rng.standard_normal((3, n)); fbar = rng.standard_normal((3, n))
    r = X.latent_adjoint(x, *theta, da, z, fbar)
    L = o.cholesky_decompose(o.gram_se(x, *theta, da))
    assert relerr(r["L"], L) == 0.0 and relerr(r["f"], z @ L.T) < 1e-15 and relerr(r["zbar"], fbar @ L) < 1e-15

    def objective(th):   # sum_m fbar_m^T L(theta) z_m
        Lt = o.cholesky_decompose(o.gram_se(x, th[0], th[1], da))
        return float(np.sum(fbar * (z @ Lt.T)))
    for k in range(2):
        h = 1e-6 * theta[k]
        tp, tm = theta.copy(), theta.copy()
        tp[k] += h; tm[k] -= h
        fd = (objective(tp) - objective(tm)) / (2 * h)
        assert abs(fd - r["theta_bar"][k]) <= 1e-6 * r["scale"][k], (k, fd, r["theta_bar"][k], r["scale"][k])
        assert r["scale"][k] >= abs(r["theta_bar"][k])
    # the symmetrised adjoint of gp_oracle.exact_gp_lp_grad gives the same rho component for nvec = 1
    y = rng.standard_normal(n)
    _, g = o.exact_gp_lp_grad(x, y, 1.0, 0.3, z[0], jitter=da)
    f = o.cholesky_decompose(o.gram_se(x, 1.0, 1.0, da)) @ z[0]
    r1 = X.latent_adjoint(x, 1.0, 1.0, da, z[0], (y - f) / 0.3 ** 2)
    assert abs(r1["theta_bar"][1] - (g["l"] - 3.0 + 4.0)) <= 1e-10 * r1["scale"][1]


# ---- extended-precision reference of the batched posterior draws (oracle/posterior_ext.py) -------------------------
def _joint_mp(t, s, theta, order, jitter):
    """J of posterior_ext.joint_cov in 50-digit mpmath, with the kernel formulas of posterior_ext"""
    import mpmath as mp
    from oracle import posterior_ext as P
    mp.mp.dps = 50
    n, m = len(t), len(s)
    pts = [mp.mpf(float(v)) for v in t] + [mp.mpf(float(v)) for v in s]
    alpha, rho, sigma = (mp.mpf(float(v)) for v in theta)
    J = mp.matrix(n + m, n + m)
    for i in range(n + m):
        for j in range(i + 1):
            name = "QQ" if i < n else P.KINDS[order][0 if j < n else 1]
            a, b = pts[i], pts[j]
            if name in P._SWAPPED:
                name, a, b = P._SWAPPED[name], b, a
            d = a - b
            J[i, j] = J[j, i] = alpha ** 2 * P._BASE[name](mp.exp(-(d ** 2 / (2 * rho ** 2))), d, rho)
        J[i, i] += sigma ** 2 if i < n else mp.mpf(jitter)
    return J


@pytest.mark.parametrize("order", [0, 1, 2])
def test_posterior_ext_matches_mpmath_llt(order):
    _need_longdouble()
    import mpmath as mp
    from oracle import posterior_ext as P
    rng = np.random.default_rng(10 + order)
    for n, m in ((1, 1), (7, 12), (19, 21)):
        t, s = np.sort(rng.uniform(0, 4, n)), np.sort(rng.uniform(-0.5, 4.5, m))
        y = np.sin(t) + 0.1 * rng.standard_normal(n)
        theta = (1.2, 0.8, 0.15)
        J = _joint_mp(t, s, theta, order, 1e-8)
        L = mp.cholesky(J)
        z1 = mp.lu_solve(L[:n, :n], mp.matrix([mp.mpf(float(v)) for v in y]))
        mu = np.array([float(v) for v in L[n:, :n] * z1])
        L22 = np.array([[float(L[n + i, n + j]) for j in range(m)] for i in range(m)])
        ext = P.posterior_ext(t, s, y, theta, order, 1e-8)
        base = P.posterior_f64(t, s, y, theta, order, 1e-8)
        assert ext.info == 0 and base.info == 0
        assert np.all(np.triu(ext.L22, 1) == 0)
        # with jitter 1e-8 the posterior block is ill-conditioned: the float64 baseline's L22 is off by up to 1e-8
        # relative here, and the long-double factor must be at least 100 times closer (measured: about 2000 times)
        for got, want, b in ((ext.mu, mu, base.mu), (ext.L22, L22, base.L22)):
            assert relerr(got, want) <= 1e-2 * relerr(b, want) + 4e-16, (n, m, relerr(got, want), relerr(b, want))
        # the long-double J is the 50-digit one to its own rounding
        Jl = P.joint_cov(t, s, theta, order, 1e-8, np.longdouble)
        Jm = np.array([[float(J[i, j]) for j in range(n + m)] for i in range(n + m)])
        dJ = max(abs(mp.mpf(float(Jl[i, j])) + mp.mpf(float(Jl[i, j] - np.longdouble(float(Jl[i, j])))) - J[i, j])
                 for i in range(n + m) for j in range(n + m))
        assert float(dJ) <= 1e-18 * np.max(np.abs(Jm)), (n, m, float(dJ))
        # the float64 J of the restated kernels is the oracle's blocks
        Jf = P.joint_cov(t, s, theta, order, 1e-8)
        a2 = theta[0] ** 2
        assert relerr(Jf[n:, :n], a2 * o.outer_kernel(P.KINDS[order][0], s, t, theta[1])) < 1e-15
        assert relerr(Jf[n:, n:] - 1e-8 * np.eye(m), a2 * o.outer_kernel(P.KINDS[order][1], s, s, theta[1])) < 1e-15


def test_posterior_ext_matches_gp_condition_at_n300_m515():
    _need_longdouble()
    from oracle import posterior_ext as P
    rng = np.random.default_rng(11)
    t, s = np.sort(rng.uniform(0, 6, 300)), np.sort(rng.uniform(-0.5, 6.5, 515))
    y = np.sin(t) + 0.1 * rng.standard_normal(300)
    theta, jitter = (1.3, 0.9, 0.1), 1e-8
    for order in (0, 1, 2):
        a2 = theta[0] ** 2
        mu, cov = o.gp_condition(a2 * o.outer_kernel("QQ", t, t, theta[1]),
                                 a2 * o.outer_kernel(P.KINDS[order][0], s, t, theta[1]),
                                 a2 * o.outer_kernel(P.KINDS[order][1], s, s, theta[1]), y, theta[2] ** 2, jitter)
        ext = P.posterior_ext(t, s, y, theta, order, jitter)
        assert ext.info == 0
        assert relerr(ext.mu, mu) < 1e-11, order
        assert relerr(ext.L22 @ ext.L22.T, cov) < 1e-11, order


def test_posterior_ext_reports_the_first_bad_pivot():
    _need_longdouble()
    from oracle import posterior_ext as P
    n, m = 30, 25
    t, s = np.linspace(0, 3, n), np.linspace(-0.2, 3.2, m)
    y = np.cos(t)
    for order in (0, 1, 2):
        for k in (0, 11, n - 1):
            tt = t.copy(); tt[k] = np.nan
            r = P.posterior_ext(tt, s, y, (1.0, 0.7, 0.1), order, 1e-8)
            assert r.info == k + 1 and np.all(np.isnan(r.mu)) and np.all(np.isnan(r.L22)), (order, k)
        for k in (0, 9, m - 1):
            ss = s.copy(); ss[k] = np.nan
            r = P.posterior_ext(t, ss, y, (1.0, 0.7, 0.1), order, 1e-8, eps=np.ones((2, m)))
            assert r.info == n + k + 1 and np.all(np.isnan(r.draws)), (order, k)
