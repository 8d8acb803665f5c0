"""The ARD posterior of tests/support/posterior_ard_ext.py (the yardstick of tests/test_posterior_draws_ard_gpu.py)
against scikit-learn's Gaussian-process regression, against the 1-D joint matrix of oracle/posterior_ext.py at D = 1,
and long double against float64."""
import os
import sys

import numpy as np
import pytest

from oracle import posterior_ext as P
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import posterior_ard_ext as A  # noqa: E402


def _data(n, m, D, seed):
    rng = np.random.default_rng(seed)
    X = rng.uniform(-2.0, 2.0, (n, D))
    Xs = rng.uniform(-2.5, 2.5, (m, D))
    y = np.sin(X).sum(axis=1) + 0.1 * rng.standard_normal(n)
    theta = np.r_[1.3, rng.uniform(0.7, 1.6, D), 0.2]
    return X, Xs, y, theta


@pytest.mark.parametrize("D", [1, 2, 3, 8])
def test_f64_posterior_agrees_with_scikit_learn(D):
    from sklearn.gaussian_process import GaussianProcessRegressor
    from sklearn.gaussian_process.kernels import RBF, ConstantKernel
    n, m, jitter = 60, 25, 1e-8
    X, Xs, y, th = _data(n, m, D, 10 + D)
    alpha, rho, sigma = th[0], th[1:-1], th[-1]
    gp = GaussianProcessRegressor(kernel=ConstantKernel(alpha ** 2, "fixed") * RBF(rho, "fixed"), alpha=sigma ** 2,
                                  optimizer=None).fit(X, y)
    mu_sk, cov_sk = gp.predict(Xs, return_cov=True)
    cov_sk = cov_sk + jitter * np.eye(m)
    post = A.posterior_ard_f64(X, Xs, y, th, jitter)
    assert post.info == 0
    assert np.max(np.abs(post.mu - mu_sk)) <= 1e-9 * np.max(np.abs(mu_sk))
    cov = post.L22 @ post.L22.T
    assert np.max(np.abs(cov - cov_sk)) <= 1e-9 * np.max(np.abs(cov_sk))


def test_ard_joint_matrix_at_one_dimension_is_the_order_zero_joint_matrix():
    rng = np.random.default_rng(3)
    t, s = np.sort(rng.uniform(0, 6, 40)), np.sort(rng.uniform(-0.5, 6.5, 30))
    theta = np.array([1.4, 0.8, 0.15])
    for S in (s, None):
        Ja = A.ard_joint_cov(t[:, None], None if S is None else S[:, None], theta, 1e-8)
        Js = P.joint_cov(t, S, theta, 0, 1e-8)
        assert Ja.shape == Js.shape
        assert np.max(np.abs(Ja - Js)) <= 4 * np.finfo(float).eps * np.max(np.abs(Js))


def test_ard_joint_matrix_predicting_on_the_inputs():
    X, _, y, th = _data(20, 1, 3, 4)
    J = A.ard_joint_cov(X, None, th, 1e-6)
    assert np.array_equal(J, A.ard_joint_cov(X, X, th, 1e-6))
    K = J[:20, :20] - th[-1] ** 2 * np.eye(20)
    assert np.array_equal(K, J[20:, 20:] - 1e-6 * np.eye(20))


def test_long_double_posterior_agrees_with_f64_when_well_conditioned():
    if not A.LONGDOUBLE_OK:
        pytest.skip("np.longdouble is not an extended type on this platform")
    X, Xs, y, th = _data(70, 45, 3, 5)
    th[-1] = 0.5                     # noise and jitter well away from the rounding of the kernel values
    eps = np.random.default_rng(6).standard_normal((2, 45))
    e = A.posterior_ard_ext(X, Xs, y, th, 1e-3, eps)
    b = A.posterior_ard_f64(X, Xs, y, th, 1e-3, eps)
    assert e.info == 0 and b.info == 0
    for u, v in ((e.mu, b.mu), (e.L22, b.L22), (e.draws, b.draws)):
        assert np.max(np.abs(u - v)) <= 1e-12 * np.max(np.abs(u))


def test_nan_coordinate_fails_at_its_pivot():
    X, Xs, y, th = _data(30, 20, 2, 7)
    Xb = X.copy()
    Xb[11, 1] = np.nan
    post = A.posterior_ard_ext(Xb, Xs, y, th, 1e-8)
    assert post.info == 12 and np.all(np.isnan(post.mu))
    Xsb = Xs.copy()
    Xsb[4, 0] = np.nan
    assert A.posterior_ard_ext(X, Xsb, y, th, 1e-8).info == 30 + 5
