"""gp_lml_grad_ard_draws of r/shim.c, executed through the functional mock of the R C API (tests/support/mock_r.py,
the build helper tests/test_r_shim.py uses): shape errors are R errors before any GPU work, and on the GPU the
(D + 2) x B result matches the float64 reference."""
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import ard_oracle  # noqa: E402
import mock_r  # noqa: E402


@pytest.fixture(scope="module")
def R():
    return mock_r.MockR()


def test_ard_entry_is_registered_and_shape_errors_are_r_errors(R):
    assert R.registered("gp_lml_grad_ard_draws") > 0
    X = np.ones((8, 3))
    y = np.zeros(8)
    with pytest.raises(mock_r.RError, match=r"\(ncol\(X\) \+ 2\) x B"):
        R.call("gp_lml_grad_ard_draws", X, y, np.ones((4, 2)), 0.0)      # theta rows must be D + 2
    with pytest.raises(mock_r.RError, match=r"length\(y\)"):
        R.call("gp_lml_grad_ard_draws", X, y[:5], np.ones((5, 2)), 0.0)
    with pytest.raises(mock_r.RError, match="1 to 8 columns"):
        R.call("gp_lml_grad_ard_draws", np.ones((8, 9)), y, np.ones((11, 2)), 0.0)


@pytest.mark.gpu
def test_ard_lml_grad_draws_through_the_shim(R):
    n, D, B = 300, 3, 5
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=12)
    out = R.call("gp_lml_grad_ard_draws", np.asfortranarray(X), y, np.asfortranarray(th.T), 1e-8)
    assert out["grad"].shape == (D + 2, B) and np.all(out["info"] == 0)
    for b in range(B):
        rv, rg = ard_oracle.lml_grad_ard(X, y, th[b, 0], th[b, 1:D + 1], th[b, D + 1], 1e-8)
        assert abs(out["lml"][b] - rv) <= 1e-9 * abs(rv)
        assert np.max(np.abs(out["grad"][:, b] - rg)) <= 1e-9 * np.max(np.abs(rg))
