"""CPU checks of the ARD LML + gradient reference (tests/support/ard_oracle.py) that the GPU tests of
gpb200_lml_grad_ard_batched compare against: scikit-learn's GP marginal likelihood, central differences, the
one-dimensional SE reference, and the exact zero of a constant column."""
import os
import sys

import numpy as np
import pytest

from oracle import gp_oracle as o
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import ard_oracle  # noqa: E402


@pytest.mark.parametrize("D", [2, 3, 8])
def test_oracle_matches_sklearn_log_marginal_likelihood(D):
    gp = pytest.importorskip("sklearn.gaussian_process")
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel, WhiteKernel
    X, y, th = ard_oracle.synth_ard(60, D, 1, seed=10 + D)
    alpha, rho, sigma = th[0, 0], th[0, 1:D + 1], th[0, D + 1]
    kern = ConstantKernel(alpha ** 2, (1e-5, 1e5)) * RBF(length_scale=rho, length_scale_bounds=(1e-5, 1e5)) + \
        WhiteKernel(sigma ** 2, noise_level_bounds=(1e-10, 1e5))
    model = gp.GaussianProcessRegressor(kernel=kern, optimizer=None, normalize_y=False, alpha=0.0)
    model.fit(X, y)
    # sklearn's hyper-parameters are log(alpha^2), log(rho_d), log(sigma^2): chain rule back to (alpha, rho, sigma)
    ref, dlog = model.log_marginal_likelihood(model.kernel_.theta, eval_gradient=True)
    got, g = ard_oracle.lml_grad_ard(X, y, alpha, rho, sigma)
    assert abs(got - ref) <= 1e-11 * abs(ref)
    want = np.concatenate([[dlog[0] * 2.0 / alpha], dlog[1:D + 1] / rho, [dlog[D + 1] * 2.0 / sigma]])
    np.testing.assert_allclose(g, want, rtol=1e-9, atol=1e-9 * np.max(np.abs(want)))


def test_oracle_gradient_matches_central_differences():
    D = 3
    X, y, th = ard_oracle.synth_ard(40, D, 1, seed=3)
    t0 = th[0]
    _, g = ard_oracle.lml_grad_ard(X, y, t0[0], t0[1:D + 1], t0[D + 1])
    for k in range(D + 2):
        h = 1e-5 * t0[k]
        tp, tm = t0.copy(), t0.copy()
        tp[k] += h
        tm[k] -= h
        fp, _ = ard_oracle.lml_grad_ard(X, y, tp[0], tp[1:D + 1], tp[D + 1])
        fm, _ = ard_oracle.lml_grad_ard(X, y, tm[0], tm[1:D + 1], tm[D + 1])
        assert abs((fp - fm) / (2 * h) - g[k]) <= 1e-6 * max(1.0, abs(g[k])), k


def test_oracle_at_one_dimension_is_the_se_reference():
    x, y = o.synth_xy(80, 5)
    for alpha, rho, sigma in o.synth_theta(4, 6):
        v1, g1 = ard_oracle.lml_grad_ard(x[:, None], y, alpha, [rho], sigma, jitter=1e-9)
        v0, g0 = o.lml_grad(x, y, alpha, rho, sigma, jitter=1e-9)
        assert abs(v1 - v0) <= 1e-12 * abs(v0)
        np.testing.assert_allclose(g1, g0, rtol=1e-10, atol=1e-12 * np.max(np.abs(g0)))


def test_constant_column_gives_exactly_zero_gradient_for_its_length_scale():
    X, y, th = ard_oracle.synth_ard(50, 3, 1, seed=8)
    X[:, 1] = 0.7
    t0 = th[0]
    v, g = ard_oracle.lml_grad_ard(X, y, t0[0], t0[1:4], t0[4])
    assert g[2] == 0.0
    v2, g2 = ard_oracle.lml_grad_ard(X[:, [0, 2]], y, t0[0], t0[[1, 3]], t0[4])
    assert abs(v - v2) <= 1e-12 * abs(v2)
    np.testing.assert_allclose(g[[0, 1, 3, 4]], g2, rtol=1e-11)


def test_reference_pivot_matches_lapack_and_stops_at_a_nan():
    X, _, th = ard_oracle.synth_ard(40, 2, 1, seed=9)
    t0 = th[0]
    assert ard_oracle.pivot(X, t0[0], t0[1:3], t0[3]) == 0
    Xs = X.copy()
    Xs[7] = Xs[3]                                   # duplicate point, no noise: singular at the second copy
    K = 1.0 * np.exp(-0.5 * np.sum(((Xs[:, None] - Xs[None]) / t0[1:3]) ** 2, axis=2))
    assert ard_oracle.pivot(Xs, 1.0, t0[1:3], 0.0) == o.potrf_info(K) == 8
    Xn = X.copy()
    Xn[11, 1] = np.nan
    assert ard_oracle.pivot(Xn, t0[0], t0[1:3], t0[3]) == 12
