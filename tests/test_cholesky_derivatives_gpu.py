"""The entry points that differentiate through the Cholesky factor, on covariances that are dense across tiles:
gpb200_rbf_cov_chol[_batched] and gpb200_se_chol_tangent (forward mode: the three tangent GEMM task lists of
tasks_tangent and launch_phi_lower, api_gp.cu) and gpb200_latent_forward / _backward (reverse mode: the nt x nt
TK_LATENT_G task list with TF_FULL_WEIGHT and latent_pw_kernel, api_latent.cu).

The other tests of these entry points use inputs whose factor and tangent vanish beyond the first off-diagonal
tile, so a wrong contraction length, triangular flag or missing task there goes unnoticed.  Every test below
asserts its own premise: the reference result carries weight in the tile pairs at least two apart
(oracle.chol_deriv_ext.far_tile_share >= 1e-2), and, where a GEMM configuration or Cholesky schedule is the point,
that the host code picks it (helpers mirroring the C conditions).

References (oracle/chol_deriv_ext.py): the dual-number LLT in long double up to n = 1100, the float64 closed form
above; the float64 reverse-mode adjoint.  They are computed once per input and cached for the module.
Bar: max |got - ref| <= 1e-9 max |ref|; a failure names the worst 128 x 128 tile (I, J).
"""
import functools

import numpy as np
import pytest

from gp_b200 import capi
from oracle import chol_deriv_ext as X
from oracle import gp_oracle as o

pytestmark = pytest.mark.gpu

RTOL = 1e-9
NSM = 148
ALPHA, RHO_TAN, DIAG_ADD = 1.3, 2.0, 0.1
WRT = {"alpha": 0, "rho": 1}


# ---- branch predicates, mirrored from the C host code --------------------------------------------------------
def tiles(n):
    return (n + 127) // 128


def gemm_cfg(ntasks, batch, override=0):
    """gemm_pick_cfg (gemm.cu:480-484) with the default knobs: 1 = whole tiles, 2 = half tiles, 3 = quarter tiles."""
    if override:
        return override
    return 3 if ntasks * batch * 2 < 2 * NSM * 2 else 2


def tangent_tasks(n):
    """tasks_tangent (api_gp.cu:229-247): one task per lower tile in each of the three lists; the batch is P."""
    nt = tiles(n)
    return nt * (nt + 1) // 2


def latent_tasks(n):
    """TK_LATENT_G (api_latent.cu:141-153): every tile pair, the upper ones included."""
    return tiles(n) ** 2


def chol_schedule(n, batch):
    """chol_batched (engine.cu:171-174, 196-200, 272-275) with the default knobs."""
    nt = tiles(n)
    if batch <= 64 and batch * nt <= 256 and nt >= 3:
        return "lookahead"
    return "left-looking" if (batch >= 64 or nt <= 8) else "panels"


# ---- inputs and cached references ----------------------------------------------------------------------------
def dense_x(n):
    """Sorted uniform on [0, 10] (on [0, 20] above 1100 points): cond(K) ~ 1e3 .. 2e4 with diag_add = 0.1."""
    return np.sort(np.random.default_rng(1000 + n).uniform(0.0, 10.0 if n <= 1100 else 20.0, n))


def shuffled_x(n):
    """A random permutation of 0, 1, ..., n-1: rbf_cov_chol's well-conditioned grid, dense across tiles."""
    return np.random.default_rng(2000 + n).permutation(n).astype(np.float64)


def need_reference(n):
    if n <= X.DUAL_MAX_N and not X.LONGDOUBLE_OK:
        pytest.skip("np.longdouble has %d mantissa bits here; the dual LLT reference needs 63" % np.finfo(np.longdouble).nmant)


@functools.lru_cache(maxsize=None)
def tangent_ref(grid, n, alpha, rho, diag_add, wrt):
    need_reference(n)
    x = dense_x(n) if grid == "dense" else shuffled_x(n)
    return X.chol_tangent(x, alpha, rho, diag_add, wrt)


def rbf_ref(n, l):
    return tangent_ref("shuffled", n, 1.0, l, o.RBF_JITTER, "rho")


def rho_lat(n):
    """The latent tests' length-scale: 2.5 on [0, 10], 1.5 on [0, 20] (the far tiles of Kbar o dK/dtheta stay
    above 1e-2 of its largest entry)."""
    return 2.5 if n <= 1100 else 1.5


def latent_inputs(n, nvec):
    rng = np.random.default_rng(3000 + 10 * n + nvec)
    return dense_x(n), rng.standard_normal((nvec, n)), rng.standard_normal((nvec, n))


@functools.lru_cache(maxsize=None)
def latent_ref(n, nvec):
    x, z, fbar = latent_inputs(n, nvec)
    return X.latent_adjoint(x, ALPHA, rho_lat(n), DIAG_ADD, z, fbar)


# ---- assertions ------------------------------------------------------------------------------------------------
def assert_close(got, ref, what, rtol=RTOL):
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    assert got.shape == ref.shape, (what, got.shape, ref.shape)
    err = np.abs(got - ref)
    bound = rtol * float(np.max(np.abs(ref)))
    worst = float(np.max(err))
    if not worst <= bound:   # also catches NaN
        where = "worst tile (I, J) = %s" % (X.worst_tile(np.nan_to_num(err, nan=np.inf)),) if got.ndim == 2 else \
            "worst entry %s" % (np.unravel_index(int(np.argmax(np.nan_to_num(err, nan=np.inf))), err.shape),)
        pytest.fail("%s: max |got - ref| = %.3e > %.3e (%.0e of max |ref|); %s" % (what, worst, bound, rtol, where))


def assert_factor(L, dL, Lr, dLr, what):
    assert_close(L, Lr, what + " L")
    assert_close(dL, dLr, what + " dL")
    assert np.all(np.triu(L, 1) == 0.0) and np.all(np.triu(dL, 1) == 0.0), what + ": strict upper triangle is not 0"


def assert_far(ref, what):
    share = X.far_tile_share(ref)
    assert share >= 1e-2, "%s: premise broken, far-tile share %.2e < 1e-2 (the test would not see far tiles)" % (what, share)


def assert_theta_bar(got, ref, scale, what):
    for k, name in enumerate(("alpha", "rho")):
        assert abs(got[k] - ref[k]) <= RTOL * scale[k], \
            "%s: theta_bar_%s = %r, reference %r, bound %.3e" % (what, name, got[k], ref[k], RTOL * scale[k])


def rbf_tables(h, x, ls):
    """gpb200_rbf_cov_chol_batched: (L, dL) as (P, n, n) arrays of row-major slices (each slice is the transpose of
    the table) and the info array, unchecked."""
    x = np.ascontiguousarray(x, dtype=np.float64)
    ls = np.ascontiguousarray(ls, dtype=np.float64)
    n, P = x.shape[0], ls.shape[0]
    L = np.empty((P, n, n)); dL = np.empty((P, n, n)); info = np.full(P, -7, dtype=np.int32)
    rc = h.lib.gpb200_rbf_cov_chol_batched(h._h, n, x.ctypes.data, P, ls.ctypes.data, L.ctypes.data, dL.ctypes.data,
                                           info.ctypes.data)
    assert rc == 0, (rc, h.lib.gpb200_last_error(h._h))
    return L, dL, info


def batched_ls(P):
    """P length-scales in [0.5, 0.7] with 0.5 first, 0.6 in the middle (index P // 2) and 0.7 last."""
    if P == 1:
        return np.array([0.7])
    ls = np.linspace(0.5, 0.7, P)
    ls[P // 2] = 0.6
    return ls


# ---- se_chol_tangent ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("wrt", ["alpha", "rho"])
@pytest.mark.parametrize("n", [129, 257, 300, 1000, 2100])
def test_se_chol_tangent_dense_matches_extended_precision(handle, n, wrt):
    Lr, dLr = tangent_ref("dense", n, ALPHA, RHO_TAN, DIAG_ADD, wrt)
    assert_far(Lr, "L"); assert_far(dLr, "dL")
    assert gemm_cfg(tangent_tasks(n), 1) == 3   # a single table: the tangent GEMMs run on quarter tiles
    L, dL = handle.se_chol_tangent(dense_x(n), ALPHA, RHO_TAN, DIAG_ADD, WRT[wrt])
    assert_factor(L, dL, Lr, dLr, "se_chol_tangent n=%d wrt %s" % (n, wrt))


def test_se_chol_tangent_matches_central_differences(handle):
    # an independent route: the derivative of LAPACK's float64 factor by central differences
    n = 1000
    x = dense_x(n)
    th = {"alpha": ALPHA, "rho": RHO_TAN}
    for wrt in ("alpha", "rho"):
        _, dL = handle.se_chol_tangent(x, ALPHA, RHO_TAN, DIAG_ADD, WRT[wrt])
        h = 1e-5 * th[wrt]

        def factor(s):
            t = dict(th); t[wrt] += s
            return o.cholesky_decompose(o.gram_se(x, t["alpha"], t["rho"], DIAG_ADD))
        fd = (factor(h) - factor(-h)) / (2 * h)
        assert_far(fd, "central difference of L wrt " + wrt)
        assert_close(dL, fd, "se_chol_tangent n=1000 wrt %s vs central differences" % wrt, rtol=1e-6)


# ---- rbf_cov_chol and its batched form --------------------------------------------------------------------------
@pytest.mark.parametrize("n,l", [(257, 0.7), (1000, 0.7), (2100, 0.7)])
def test_rbf_cov_chol_shuffled_grid_matches_extended_precision(handle, n, l):
    Lr, dLr = rbf_ref(n, l)
    assert_far(Lr, "L"); assert_far(dLr, "dL")
    L, dL = handle.rbf_cov_chol(shuffled_x(n), l)
    assert_factor(L, dL, Lr, dLr, "rbf_cov_chol n=%d l=%g" % (n, l))


@pytest.mark.parametrize("P", [1, 3, 9, 64])
def test_rbf_cov_chol_batched_tables_match_single_calls_and_reference(handle, P):
    n = 1000
    x = shuffled_x(n)
    ls = batched_ls(P)
    # P < 9 keeps the tangent GEMMs on quarter tiles, P >= 9 moves them to half tiles; P = 64 factors with the
    # large-batch (pure left-looking) Cholesky schedule, the others with the look-ahead schedule
    assert gemm_cfg(tangent_tasks(n), P) == (3 if P < 9 else 2)
    assert chol_schedule(n, P) == ("left-looking" if P == 64 else "lookahead")
    L, dL, info = rbf_tables(handle, x, ls)
    assert np.all(info == 0), info
    for q in range(P):
        Ls, dLs = handle.rbf_cov_chol(x, float(ls[q]))
        assert_close(L[q].T, Ls, "table %d L vs its single-table call" % q, rtol=1e-12)
        assert_close(dL[q].T, dLs, "table %d dL vs its single-table call" % q, rtol=1e-12)
    for q in sorted({0, P // 2, P - 1}):
        Lr, dLr = rbf_ref(n, float(ls[q]))
        assert_far(Lr, "L"); assert_far(dLr, "dL")
        assert_factor(L[q].T, dL[q].T, Lr, dLr, "rbf_cov_chol_batched P=%d table %d (l=%g)" % (P, q, ls[q]))


def test_rbf_cov_chol_batched_reference_grid_identities(handle):
    # the reference's own tables: x = seq(0, 10, length = N) and lp = seq(qgamma(.05, 4, 4), qgamma(.95, 4, 4),
    # length = 10) of test_interpolate.R, at N = 1000.  cond(Sigma) ~ 1e10, so L is not reproducible to 1e-9: check
    # the identities L L^T = Sigma and Ldot L^T + L Ldot^T = dSigma/dl instead, per 128 x 128 block, each within 10x
    # the LAPACK oracle's residual in that block.  The floor differs.  The backward error of L is a property of each
    # block: 1e-12 of the block's norm.  The tangent is known only to about eps cond(Sigma) of ||dSigma|| (the oracle's
    # own residual is 2e-7 .. 5e-7 ||dSigma||), and how that error spreads over the blocks depends on the order of
    # the sums: the explicit-inverse route Ldot = L Phi(W dSigma W^T) that the library takes leaves up to 1e4x the
    # oracle's residual in a block where dSigma is small (tile (0, 2) at l = 0.34), and less than the oracle overall.  So
    # there the floor is 1e-8 ||dSigma||, 20x below the oracle's overall residual, and the whole residual must be within
    # 10x the oracle's.
    from scipy.stats import gamma
    n = 1000
    x = np.linspace(0.0, 10.0, n)
    lp = np.linspace(gamma.ppf(0.05, 4, scale=0.25), gamma.ppf(0.95, 4, scale=0.25), 10)
    assert gemm_cfg(tangent_tasks(n), len(lp)) == 2
    L, dL, info = rbf_tables(handle, x, lp)
    assert np.all(info == 0), info
    for q, l in enumerate(lp):
        S, Sdot = o.rbf_gram_and_tangent(x, l)
        Lr, dLr = o.rbf_cov_chol(x, l)
        assert_far(Lr, "L (l=%g)" % l)
        Lg, dLg = L[q].T, dL[q].T
        assert np.all(np.triu(Lg, 1) == 0.0) and np.all(np.triu(dLg, 1) == 0.0)
        checks = (("L L^T - Sigma", Lg @ Lg.T - S, Lr @ Lr.T - S, lambda r, c: 1e-12 * np.linalg.norm(S[r, c])),
                  ("Ldot L^T + L Ldot^T - dSigma", dLg @ Lg.T + Lg @ dLg.T - Sdot, dLr @ Lr.T + Lr @ dLr.T - Sdot,
                   lambda r, c: 1e-8 * np.linalg.norm(Sdot)))
        for what, R, Rr, floor in checks:
            got, ref = np.linalg.norm(R), np.linalg.norm(Rr)
            assert got <= 10.0 * ref, "l=%g %s: residual %.3e > 10x the oracle's %.3e" % (l, what, got, ref)
            for I, J, r, c in X.tile_blocks(n):
                got, ref = np.linalg.norm(R[r, c]), np.linalg.norm(Rr[r, c])
                bound = 10.0 * max(ref, floor(r, c))
                assert got <= bound, "l=%g %s: tile (%d, %d) residual %.3e > %.3e (oracle %.3e)" % (l, what, I, J, got, bound, ref)


# ---- latent_forward / latent_backward ---------------------------------------------------------------------------
def check_latent(h, n, nvec, what):
    x, z, fbar = latent_inputs(n, nvec)
    r = latent_ref(n, nvec)
    assert_far(r["L"], "L")
    for k in range(2):
        assert_far(r["terms"][k], "Kbar o dK/dtheta_%d" % k)
        # deleting the far tile pairs from the adjoint would move theta_bar by far more than the bar
        assert abs(X.far_tile_sum(r["terms"][k])) >= 1e3 * RTOL * r["scale"][k], (what, k)
    f = h.latent_forward(x, ALPHA, rho_lat(n), DIAG_ADD, z)
    tb, zbar = h.latent_backward(x, ALPHA, rho_lat(n), DIAG_ADD, z, fbar)
    assert_close(f, r["f"], what + " f", rtol=1e-10)
    assert_close(zbar, r["zbar"], what + " zbar", rtol=1e-10)
    assert_theta_bar(tb, r["theta_bar"], r["scale"], what)
    return x, z, fbar, tb


@pytest.mark.parametrize("nvec", [1, 3])
@pytest.mark.parametrize("n", [300, 1000, 2200])
def test_latent_adjoint_dense_matches_reference_and_forward_mode(handle, n, nvec):
    x, z, fbar, tb = check_latent(handle, n, nvec, "latent n=%d nvec=%d" % (n, nvec))
    # the forward-mode route on the GPU's own tangents: thetabar = sum_m fbar_m^T (Ldot_theta z_m)
    fwd = []
    for wrt in ("alpha", "rho"):
        _, dL = handle.se_chol_tangent(x, ALPHA, rho_lat(n), DIAG_ADD, WRT[wrt])
        fwd.append(float(np.sum(fbar * (z @ dL.T))))
    assert_theta_bar(fwd, tb, latent_ref(n, nvec)["scale"], "latent n=%d nvec=%d: forward mode vs reverse mode" % (n, nvec))


# ---- every GEMM configuration -----------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [0, 1, 2])
def test_derivative_entry_points_under_every_gemm_configuration(handle, cfg):
    n = 1000
    # automatic choice: a single table and the latent adjoint at n = 1000 stay on quarter tiles, nine tables go to half
    expect = {"tangent": 3, "latent": 3, "batched": 2} if cfg == 0 else dict.fromkeys(("tangent", "latent", "batched"), cfg)
    assert gemm_cfg(tangent_tasks(n), 1, cfg) == expect["tangent"]
    assert gemm_cfg(latent_tasks(n), 1, cfg) == expect["latent"]
    assert gemm_cfg(tangent_tasks(n), 9, cfg) == expect["batched"]
    try:
        handle.set_gemm_config(cfg)
        Lr, dLr = tangent_ref("dense", n, ALPHA, RHO_TAN, DIAG_ADD, "rho")
        assert_far(dLr, "dL")
        L, dL = handle.se_chol_tangent(dense_x(n), ALPHA, RHO_TAN, DIAG_ADD, 1)
        assert_factor(L, dL, Lr, dLr, "cfg %d se_chol_tangent" % cfg)
        Lr, dLr = rbf_ref(n, 0.7)
        L, dL = handle.rbf_cov_chol(shuffled_x(n), 0.7)
        assert_factor(L, dL, Lr, dLr, "cfg %d rbf_cov_chol" % cfg)
        ls = batched_ls(9)
        L, dL, info = rbf_tables(handle, shuffled_x(n), ls)
        assert np.all(info == 0), info
        for q in (0, 4, 8):
            Lr, dLr = rbf_ref(n, float(ls[q]))
            assert_factor(L[q].T, dL[q].T, Lr, dLr, "cfg %d rbf_cov_chol_batched table %d" % (cfg, q))
        check_latent(handle, n, 3, "cfg %d latent" % cfg)
    finally:
        handle.set_gemm_config(0)


# ---- the latent factor cache --------------------------------------------------------------------------------------
def test_latent_factor_cache_never_serves_a_stale_factor():
    """latent_factor keeps the factor of the last successful call, keyed on an FNV hash of the host x and on
    (alpha, rho, diag_add).  Each call on one handle must equal, bit for bit, the same call on a fresh handle; each
    step changes what the previous step's factor was built from, so a stale factor would show."""
    n = 300
    x1, z, fbar = latent_inputs(n, 2)
    x2 = x1.copy()
    x2[n // 2] = np.nextafter(x2[n // 2], np.inf)   # one ulp
    good = (ALPHA, rho_lat(n), DIAG_ADD)

    def bits(res):
        return [np.asarray(a, dtype=np.float64).view(np.uint64).copy() for a in res]

    def call(h, kind, x, p):
        if kind == "forward":
            return bits([h.latent_forward(x, *p, z)])
        tb, zbar = h.latent_backward(x, *p, z, fbar)
        return bits([tb, zbar])

    def fresh(kind, x, p):
        h = capi.Handle(0)
        try:
            return call(h, kind, x, p)
        finally:
            h.close()

    steps = [("forward", x1, good), ("backward", x2, good),
             ("backward", x2, (1.25, rho_lat(n), DIAG_ADD)), ("backward", x2, (1.25, 1.45, DIAG_ADD)),
             ("backward", x2, (1.25, 1.45, 0.12))]
    h = capi.Handle(0)
    try:
        prev = None
        for kind, x, p in steps:
            ref = fresh(kind, x, p)
            if prev is not None:   # premise: the factor of the previous step gives a different answer
                stale = fresh(kind, prev[0], prev[1])
                assert any(not np.array_equal(a, b) for a, b in zip(ref, stale)), (kind, p, "premise")
            got = call(h, kind, x, p)
            assert all(np.array_equal(a, b) for a, b in zip(got, ref)), (kind, p)
            prev = (x, p)
        # a failed factorisation (alpha^2 - 2 alpha^2 < 0 at the first pivot) followed by the previous good call
        with pytest.raises(capi.NotPositiveDefiniteError) as ei:
            h.latent_backward(x2, 1.25, 1.45, -2.0 * 1.25 ** 2, z, fbar)
        assert ei.value.info == 1
        for kind in ("backward", "forward"):
            got = call(h, kind, x2, (1.25, 1.45, 0.12))
            assert all(np.array_equal(a, b) for a, b in zip(got, fresh(kind, x2, (1.25, 1.45, 0.12)))), ("after info", kind)
    finally:
        h.close()
