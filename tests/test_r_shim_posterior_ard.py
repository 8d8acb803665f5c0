"""gp_posterior_draws_ard of r/shim.c, executed through the functional mock of the R C API (tests/support/mock_r.py):
shape and type errors are R errors before any GPU work, a failed draw is an R error naming it, and on the GPU the
m x B result equals the Python binding bit for bit."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import mock_r  # noqa: E402


@pytest.fixture(scope="module")
def R():
    return mock_r.MockR()


def _inputs(n=40, m=25, D=3, B=4, seed=1):
    rng = np.random.default_rng(seed)
    X = rng.uniform(0, 4, (n, D))
    Xs = rng.uniform(0, 4, (m, D))
    y = np.sin(X).sum(axis=1)
    theta = np.column_stack([rng.uniform(0.8, 1.5, B), rng.uniform(1.0, 2.5, (B, D)), rng.uniform(0.1, 0.3, B)])
    return X, Xs, y, theta


def test_entry_is_registered_and_shape_and_type_errors_are_r_errors(R):
    assert R.registered("gp_posterior_draws_ard") > 0
    X, Xs, y, th = _inputs()
    T = np.asfortranarray(th.T)
    z = np.zeros((25, 4))
    call = lambda *a: R.call("gp_posterior_draws_ard", *a)
    with pytest.raises(mock_r.RError, match=r"\(ncol\(X\) \+ 2\) x B"):
        call(X, y, T[:4], Xs, 1e-8, 1.0, None)                       # theta rows must be D + 2
    with pytest.raises(mock_r.RError, match=r"length\(y\)"):
        call(X, y[:7], T, Xs, 1e-8, 1.0, None)
    with pytest.raises(mock_r.RError, match="1 to 8 columns"):
        call(np.ones((40, 9)), y, np.ones((11, 4)), None, 1e-8, 1.0, None)
    with pytest.raises(mock_r.RError, match="Xs must be a matrix with ncol"):
        call(X, y, T, Xs[:, :2], 1e-8, 1.0, None)
    with pytest.raises(mock_r.RError, match="z must be a 25 x 4"):
        call(X, y, T, Xs, 1e-8, None, z[:, :3])                      # seed NULL: normals z of m x B
    with pytest.raises(mock_r.RError, match="needed when seed is NULL"):
        call(X, y, T, Xs, 1e-8, None, None)
    with pytest.raises(mock_r.RError, match="must not be NULL"):
        call(None, y, T, Xs, 1e-8, 1.0, None)
    with pytest.raises(mock_r.RError, match="cannot coerce"):
        call([X], y, T, Xs, 1e-8, 1.0, None)                          # a list is not a numeric matrix


@pytest.mark.gpu
def test_r_result_equals_the_python_binding_bit_for_bit(R):
    from gp_b200 import capi
    X, Xs, y, th = _inputs(n=300, m=213, D=3, B=6, seed=2)
    B, m = th.shape[0], Xs.shape[0]
    Z = np.random.default_rng(3).standard_normal((B, m))
    h = capi.Handle(0)
    try:
        for xs in (Xs, None):
            mm = m if xs is not None else X.shape[0]
            Zb = Z if xs is not None else np.random.default_rng(4).standard_normal((B, mm))
            out = R.call("gp_posterior_draws_ard", np.asfortranarray(X), y, np.asfortranarray(th.T),
                         None if xs is None else np.asfortranarray(xs), 1e-8, None, np.asfortranarray(Zb.T))
            ref, _, info = h.posterior_draws_ard_batched(X, y, th, Xs=xs, jitter=1e-8, z=Zb)
            assert np.all(info == 0) and out.shape == (mm, B)
            assert np.array_equal(out.T.view(np.uint64), ref.view(np.uint64))
            out_s = R.call("gp_posterior_draws_ard", np.asfortranarray(X), y, np.asfortranarray(th.T),
                           None if xs is None else np.asfortranarray(xs), 1e-8, 5.0, None)
            ref_s, _, _ = h.posterior_draws_ard_batched(X, y, th, Xs=xs, jitter=1e-8, seed=5)
            assert np.array_equal(np.ascontiguousarray(out_s.T).view(np.uint64), ref_s.view(np.uint64))
        bad = th.copy()
        bad[2, 1] = np.nan                                            # a NaN length-scale fails draw 3 at pivot 2
        with pytest.raises(mock_r.RError, match="draw 3: .* pivot at 2"):
            R.call("gp_posterior_draws_ard", np.asfortranarray(X), y, np.asfortranarray(bad.T), np.asfortranarray(Xs),
                   1e-8, 5.0, None)
    finally:
        h.close()
