"""gpb200_posterior_draws_batched: B posterior draws of f^(p) on a prediction grid, one per hyper-parameter
draw, from one Cholesky factorisation of the joint prior covariance of (y, f^(p)(s)) per item.

The factor L22 of the posterior covariance is never returned; it is recovered through the draws.  With y = 0
(mu is then exactly 0) and the caller's normals z_k = e_k for items k = 0 .. m-1 with one theta, draw k is
column k of L22.  So "L22 L22^T = cov + jitter I" and "L22 is lower triangular" are checked on what a caller
receives.  References: the oracle's dense solve (oracle.gp_condition) and the reference's own goldens
(gp_derivs.py, ch2.py)."""
import os
import sys

import numpy as np
import pytest

from gp_b200 import capi, ode_gp_library as lib
from oracle import gp_oracle as o

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import mock_r  # noqa: E402

gpu = pytest.mark.gpu
KINDS = {0: ("QQ", "QQ"), 1: ("RQ", "RR"), 2: ("TQ", "TT")}


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def reference(t, s, y, theta, order):
    """mu and cov (without jitter) of f^(order)(s) given y = f(t) + N(0, sigma^2) on t, by a dense solve"""
    alpha, rho, sigma = (float(v) for v in theta)
    a2 = alpha * alpha
    K = a2 * o.outer_kernel("QQ", t, t, rho)
    Ks = a2 * o.outer_kernel(KINDS[order][0], s, t, rho)
    Kss = a2 * o.outer_kernel(KINDS[order][1], s, s, rho)
    return o.gp_condition(K, Ks, Kss, y, sigma * sigma, 0.0)


def recover_factor(h, t, s, theta, order, jitter):
    """L22 of one theta: column k is the draw with y = 0 and normals e_k"""
    n = np.shape(t)[-1]
    m = n if s is None else np.shape(s)[-1]
    draws, mu, info = h.posterior_draws_batched(t, np.zeros(n), np.tile(theta, (m, 1)), order=order, s=s, jitter=jitter,
                                                z=np.eye(m))
    assert np.all(info == 0), info
    assert np.all(mu == 0.0)
    return draws.T.copy()


def grid(n, seed, lo=0.0, hi=6.0):
    return np.sort(np.random.default_rng(seed).uniform(lo, hi, n))


@pytest.fixture(scope="module")
def h():
    hd = capi.Handle(0)
    yield hd
    hd.close()


@pytest.fixture(scope="module")
def golden():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "gp_derivs_golden.npz"))


@pytest.fixture(scope="module")
def ch2():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ch2_golden.npz"))


# ---- 1. the reference's own outputs ------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("order, which", [(0, "d"), (2, "i")])
def test_reference_gp_derivs_golden(h, golden, order, which):
    # gp_derivs.py:97-113 on ts = tts = linspace(0, 5, 25), a = l = 1, s = 0.1.  Its "d" pair (KsK, KsKs) are QQ
    # Grams (the golden's KsK equals its K), so mu_d / cov_d are the order-0 posterior; mu_i / cov_i condition TQ / TT.
    ts, tts, y = golden["ts"], golden["tts"], golden["y"]
    theta = np.array([[float(golden["a"]), float(golden["l"]), float(golden["s"])]])
    s = ts if order == 0 else tts
    _, mu, info = h.posterior_draws_batched(ts, y, theta, order=order, s=s, jitter=1e-8, seed=3)
    assert info[0] == 0
    assert relerr(mu[0], golden["mu_" + which]) < 1e-10
    L = recover_factor(h, ts, s, theta[0], order, 1e-8)
    assert relerr(L @ L.T - 1e-8 * np.eye(25), golden["cov_" + which]) < 1e-10


@gpu
def test_reference_ch2_golden(h, ch2):
    # ch2.py:55-91: 1000-point posterior of an SE GP (eta2 exp(-d^2 / l2)) on 4 noise-free observations, Cholesky of
    # the posterior + 1e-10 I; here alpha^2 = eta2, rho = sqrt(l2 / 2), sigma = 0
    g = ch2
    theta = np.array([np.sqrt(float(g["eta2"])), np.sqrt(float(g["l2"]) / 2.0), 0.0])
    xs, xd = g["xs"], g["xd"]
    _, mu, info = h.posterior_draws_batched(xd, g["f"], theta[None, :], order=0, s=xs, jitter=1e-10, seed=1)
    assert info[0] == 0
    assert relerr(mu[0], g["m"]) < 1e-9
    draws, mu0, info = h.posterior_draws_batched(xd, np.zeros(4), np.tile(theta, (5, 1)), order=0, s=xs, jitter=1e-10,
                                                 z=np.eye(1000)[:5])
    assert np.all(info == 0) and np.all(mu0 == 0.0)
    assert relerr(np.diag(draws[:, :5]), g["L_diag"][:5]) < 1e-6


# ---- 2. parity with the dense-solve oracle -----------------------------------------------------------------------------
SHAPES = [(1, 1), (5, 5), (127, 128), (128, 129), (129, 127), (300, 515), (515, 300)]


@gpu
@pytest.mark.parametrize("order", [0, 1, 2])
@pytest.mark.parametrize("n, m", SHAPES)
def test_oracle_parity_separate_grid(h, order, n, m):
    t, s = grid(n, n), grid(m, 1000 + m, -0.5, 6.5)
    y = np.sin(t) + 0.1 * np.random.default_rng(n + m).standard_normal(n)
    theta = np.array([1.3, 0.9, 0.1 + 0.05 * order])
    check_item(h, t, s, y, theta, order, jitter=1e-8)


@gpu
@pytest.mark.parametrize("order", [0, 1, 2])
@pytest.mark.parametrize("n", [1, 5, 128, 129, 300])
def test_oracle_parity_on_the_training_grid(h, order, n):
    t = grid(n, 7 * n)
    y = np.cos(t) + 0.1 * np.random.default_rng(n).standard_normal(n)
    check_item(h, t, None, y, np.array([0.8, 1.1, 0.2]), order, jitter=1e-8)


def check_item(h, t, s, y, theta, order, jitter):
    n = t.shape[0]
    m = n if s is None else s.shape[0]
    mu_ref, cov_ref = reference(t, t if s is None else s, y, theta, order)
    _, mu1, info = h.posterior_draws_batched(t, y, theta[None, :], order=order, s=s, jitter=jitter, seed=2)
    assert info[0] == 0
    assert relerr(mu1[0], mu_ref) < 1e-9
    # items 0 .. m-1 recover L22; item m (same theta, in the same launches) draws with the data and random normals
    z = np.random.default_rng(m).standard_normal(m)
    Y = np.zeros((m + 1, n)); Y[m] = y
    draws, mu, info = h.posterior_draws_batched(t, Y, np.tile(theta, (m + 1, 1)), order=order, s=s, jitter=jitter,
                                                z=np.vstack([np.eye(m), z]))
    assert np.all(info == 0) and np.all(mu[:m] == 0.0)
    L = draws[:m].T
    assert np.all(np.triu(L, 1) == 0.0)                      # the mat-vecs read j <= i only
    A = cov_ref + jitter * np.eye(m)
    assert np.linalg.norm(L @ L.T - A) / np.linalg.norm(A) < 1e-10
    assert relerr(mu[m], mu_ref) < 1e-9
    assert relerr(draws[m], mu[m] + L @ z) < 1e-12


@gpu
@pytest.mark.parametrize("order", [0, 1, 2])
def test_strided_and_shared_inputs_per_item(h, order):
    # per-item t, s and y (strides n, m, n) and every shared / strided mix: each item against its own oracle, and the
    # batch against the same items called one at a time with the same normals
    B, n, m = 6, 130, 97
    rng = np.random.default_rng(order)
    T = np.sort(rng.uniform(0, 6, (B, n)), axis=1)
    S = np.sort(rng.uniform(-0.5, 6.5, (B, m)), axis=1)
    Y = np.sin(T) + 0.1 * rng.standard_normal((B, n))
    th = np.column_stack([rng.uniform(0.5, 2.0, B), rng.uniform(0.6, 1.5, B), rng.uniform(0.1, 0.3, B)])
    z = rng.standard_normal((B, m))
    for tt, ss, yy in ((T, S, Y), (T[0], S, Y), (T, S[0], Y[0]), (T[0], S[0], Y)):
        draws, mu, info = h.posterior_draws_batched(tt, yy, th, order=order, s=ss, z=z)
        assert np.all(info == 0)
        for b in range(B):
            tb, sb, yb = (a[b] if a.ndim == 2 else a for a in (tt, ss, yy))
            mu_ref, _ = reference(tb, sb, yb, th[b], order)
            assert relerr(mu[b], mu_ref) < 1e-9
            d1, m1, _ = h.posterior_draws_batched(tb, yb, th[b:b + 1], order=order, s=sb, z=z[b:b + 1])
            assert relerr(d1[0], draws[b]) < 1e-10 and relerr(m1[0], mu[b]) < 1e-10


# ---- 3. the seeded normal stream ----------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("m", [128, 129])
def test_seed_stream_is_normal_fill_per_item_and_independent_of_chunking(h, m):
    B, n, seed = 9, 64, 77
    t, s = grid(n, 3), grid(m, 4)
    y = np.sin(t)
    rng = np.random.default_rng(m)
    th = np.column_stack([rng.uniform(0.5, 2.0, B), rng.uniform(0.6, 1.5, B), rng.uniform(0.1, 0.3, B)])
    d_seed, mu_seed, info = h.posterior_draws_batched(t, y, th, order=1, s=s, seed=seed)
    assert np.all(info == 0)
    z = h.normal_fill(seed, B * m).reshape(B, m)
    d_z, mu_z, _ = h.posterior_draws_batched(t, y, th, order=1, s=s, z=z)
    assert np.array_equal(d_seed, d_z) and np.array_equal(mu_seed, mu_z)
    # chunks of 3 items (np = 256: 1 MiB of factor and inverse tiles per item): with m = 129 the chunks start at odd
    # offsets of the stream
    hc = capi.Handle(0)
    try:
        hc.set_workspace_limit(4 << 20)
        d_c, mu_c, info_c = hc.posterior_draws_batched(t, y, th, order=1, s=s, seed=seed)
    finally:
        hc.close()
    assert np.all(info_c == 0)
    assert relerr(d_c, d_seed) < 1e-12 and relerr(mu_c, mu_seed) < 1e-12


@gpu
def test_single_draw_uses_the_normals_of_mvrnorm(h):
    n, m, seed = 40, 33, 1234
    t, s = grid(n, 1), grid(m, 2)
    th = np.array([[1.1, 0.7, 0.2]])
    eps = h.mvrnorm(1, None, np.eye(m), seed)          # chol(I) eps = the normals mvrnorm draws with
    d_seed, _, _ = h.posterior_draws_batched(t, np.sin(t), th, order=2, s=s, seed=seed)
    d_z, _, _ = h.posterior_draws_batched(t, np.sin(t), th, order=2, s=s, z=eps[None, :])
    assert np.array_equal(d_seed, d_z)


# ---- 4. failed items and bad arguments ------------------------------------------------------------------------------------
@gpu
def test_failed_items_get_nan_and_leave_their_neighbours_bit_identical(h):
    n, m, B = 50, 40, 8
    t = grid(n, 5)
    t[1] = t[0]                                         # duplicated point: with sigma = 0 the second pivot is exactly 0
    s = grid(m, 6)
    y = np.sin(t)
    rng = np.random.default_rng(2)
    th = np.column_stack([np.ones(B), rng.uniform(0.6, 1.5, B), rng.uniform(0.1, 0.3, B)])
    good_d, good_mu, info = h.posterior_draws_batched(t, y, th, order=1, s=s, seed=5)
    assert np.all(info == 0)
    bad = th.copy()
    bad[1, 1] = np.nan                                  # NaN theta
    bad[4, 2] = 0.0                                     # K singular
    d, mu, info = h.posterior_draws_batched(t, y, bad, order=1, s=s, seed=5)
    assert info[1] != 0 and 1 <= info[4] <= n
    for b in (1, 4):
        assert np.all(np.isnan(d[b])) and np.all(np.isnan(mu[b]))
    keep = [b for b in range(B) if b not in (1, 4)]
    assert np.all(info[keep] == 0)
    assert np.array_equal(d[keep], good_d[keep]) and np.array_equal(mu[keep], good_mu[keep])
    # a negative jitter larger than the posterior variance: cov is not positive definite
    d, mu, info = h.posterior_draws_batched(t, y, th[:3], order=1, s=s, seed=5, jitter=-100.0)
    assert np.all((info > n) & (info <= n + m)) and np.all(np.isnan(d)) and np.all(np.isnan(mu))


@gpu
def test_bad_arguments_return_negative_and_leave_outputs_untouched(h):
    n, m, B = 6, 5, 2
    t, s, y = np.linspace(0, 1, n), np.linspace(0, 1, m), np.ones(n)
    th = np.tile([1.0, 0.5, 0.1], (B, 1))
    draws, mu, info = np.full(B * 8, 7.0), np.full(B * 8, 7.0), np.full(B, 7, dtype=np.int32)
    f = h.lib.gpb200_posterior_draws_batched
    p = lambda a: a.ctypes.data
    base = dict(n=n, m=m, order=1, B=B, ts=0, s=p(s), ss=0, ys=0)
    for change in (dict(n=0), dict(m=0), dict(order=3), dict(order=-1), dict(s=None), dict(ts=n - 1), dict(ss=m - 1),
                   dict(ys=n - 1), dict(B=-1)):
        a = dict(base, **change)
        rc = f(h._h, a["n"], a["m"], a["order"], a["B"], p(t), a["ts"], a["s"], a["ss"], p(y), a["ys"], p(th), 1e-8, None, 1,
               p(draws), p(mu), p(info))
        assert rc < 0, change
        assert np.all(draws == 7.0) and np.all(mu == 7.0) and np.all(info == 7), change
    assert f(h._h, n, m, 1, 0, p(t), 0, p(s), 0, p(y), 0, p(th), 1e-8, None, 1, p(draws), p(mu), p(info)) == 0
    assert np.all(draws == 7.0)


# ---- 5. device-pointer mode ------------------------------------------------------------------------------------------------
@gpu
def test_device_pointer_mode_is_bit_identical_and_runs_on_the_handles_stream(h):
    import torch
    B, n, m = 5, 90, 70
    rng = np.random.default_rng(9)
    T = np.sort(rng.uniform(0, 6, (B, n)), axis=1)
    s = grid(m, 8)
    Y = np.sin(T)
    th = np.column_stack([rng.uniform(0.5, 2.0, B), rng.uniform(0.6, 1.5, B), rng.uniform(0.1, 0.3, B)])
    th[2, 0] = np.nan
    z = rng.standard_normal((B, m))
    ref = [h.posterior_draws_batched(T, Y, th, order=1, s=s, seed=11), h.posterior_draws_batched(T, Y, th, order=1, s=s, z=z)]
    hd = capi.Handle(0)
    try:
        hd.set_pointer_mode(True)
        stream = torch.cuda.Stream()
        hd.set_stream(stream.cuda_stream)
        dev = lambda a: torch.as_tensor(np.ascontiguousarray(a), device="cuda")
        dT, ds, dY, dth, dz = dev(T), dev(s), dev(Y), dev(th), dev(z)
        torch.cuda.synchronize()
        for k, (zz, seed) in enumerate(((None, 11), (dz, 0))):
            draws = torch.empty((B, m), dtype=torch.float64, device="cuda")
            mu = torch.empty_like(draws)
            info = torch.full((B,), -5, dtype=torch.int32, device="cuda")
            hd.posterior_draws_batched_device(n, m, 1, B, dT, n, ds, 0, dY, n, dth, 1e-8, zz, seed, draws, mu, info)
            stream.synchronize()
            assert np.array_equal(draws.cpu().numpy(), ref[k][0], equal_nan=True)
            assert np.array_equal(mu.cpu().numpy(), ref[k][1], equal_nan=True)
            assert np.array_equal(info.cpu().numpy(), ref[k][2])
    finally:
        hd.close()


# ---- 6. the Python and R mirrors -----------------------------------------------------------------------------------------
@gpu
def test_sample_derivs_draws_mirror(h):
    n, B = 120, 7
    ti = np.linspace(0, 10, n)
    rng = np.random.default_rng(3)
    params = np.column_stack([rng.uniform(0.8, 2.0, B), rng.uniform(0.5, 1.5, B), rng.uniform(0.05, 0.2, B)])  # (l, a, sy)
    y = np.sin(ti) + 0.1 * rng.standard_normal(n)
    got = lib.sample_derivs_draws(params, y, ti, seed=21, handle=h)
    want, mu, _ = h.posterior_draws_batched(ti, y, params[:, [1, 0, 2]], order=1, jitter=1e-8, seed=21)
    assert np.array_equal(got, want)
    for b in range(B):                                  # the per-draw route of pendulum_fit.R:227-251
        mu_ref, _ = lib.sample_derivs_moments(params[b], y, ti, handle=h)
        assert relerr(mu[b], mu_ref) < 1e-9
    Yb = y + 0.01 * rng.standard_normal((B, n))
    got_r = lib.sample_derivs_draws(params, Yb, ti, rng=np.random.default_rng(4), handle=h)
    z = np.random.default_rng(4).standard_normal((B, n))
    want_r, _, _ = h.posterior_draws_batched(ti, Yb, params[:, [1, 0, 2]], order=1, jitter=1e-8, z=z)
    assert np.array_equal(got_r, want_r)


@gpu
def test_r_sample_derivs_draws_through_the_mock_r_equals_the_python_mirror(h):
    R = mock_r.MockR()
    n, B = 64, 5
    ti = np.linspace(0, 6, n)
    rng = np.random.default_rng(8)
    params = np.column_stack([rng.uniform(0.8, 2.0, B), rng.uniform(0.5, 1.5, B), rng.uniform(0.05, 0.2, B)])
    y = np.sin(ti)
    out = R.call("gp_sample_derivs_draws", np.asfortranarray(params.T), y, ti, 17.0, None)
    assert out.shape == (n, B)
    assert np.array_equal(out, lib.sample_derivs_draws(params, y, ti, seed=17, handle=h).T)
    Y = np.sin(ti)[:, None] + 0.01 * rng.standard_normal((n, B))          # n x B ynoise, R's normals as z
    z = np.random.default_rng(1).standard_normal((B, n))
    out = R.call("gp_sample_derivs_draws", np.asfortranarray(params.T), np.asfortranarray(Y), ti, None, np.asfortranarray(z.T))
    got = lib.sample_derivs_draws(params, Y.T.copy(), ti, rng=np.random.default_rng(1), handle=h)
    assert np.array_equal(out, got.T)


def test_mirror_shape_errors_raise_without_a_gpu():
    ti = np.linspace(0, 1, 8)
    with pytest.raises(ValueError, match="params"):
        lib.sample_derivs_draws(np.ones(3), np.zeros(8), ti, seed=1)
    with pytest.raises(ValueError, match="ynoise"):
        lib.sample_derivs_draws(np.ones((2, 3)), np.zeros(7), ti, seed=1)
    with pytest.raises(ValueError, match="ynoise"):
        lib.sample_derivs_draws(np.ones((2, 3)), np.zeros((3, 8)), ti, seed=1)


def test_r_shape_and_type_errors_are_r_errors_before_any_gpu_work():
    R = mock_r.MockR()
    ti = np.linspace(0, 1, 8)
    with pytest.raises(mock_r.RError, match="3 x B matrix"):
        R.call("gp_sample_derivs_draws", np.ones((4, 2)), np.zeros(8), ti, 1.0, None)
    with pytest.raises(mock_r.RError, match="ynoise must be a 8 x 2"):
        R.call("gp_sample_derivs_draws", np.ones((3, 2)), np.zeros((8, 3)), ti, 1.0, None)
    with pytest.raises(mock_r.RError, match="z must be a 8 x 2"):
        R.call("gp_sample_derivs_draws", np.ones((3, 2)), np.zeros(8), ti, None, np.zeros((8, 3)))
    with pytest.raises(mock_r.RError, match="must not be NULL"):
        R.call("gp_sample_derivs_draws", np.ones((3, 2)), np.zeros(8), ti, None, None)
