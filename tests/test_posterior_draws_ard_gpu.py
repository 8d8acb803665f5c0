"""gpb200_posterior_draws_ard_batched on the GPU: batched posterior draws under the ARD kernel (QQard) against the
extended-precision posterior of tests/support/posterior_ard_ext.py (posterior_ard_ext, with posterior_ard_f64 as the
float64 baseline), with the per-tile yardstick of tests/test_posterior_draws_ext_gpu.py; against the 1-D SE entry point at
D = 1; under invariances of the model; on the normal stream and its chunking; on strided inputs in both pointer modes;
on failed items in every Cholesky schedule; under every schedule knob; and on bad arguments.

L22, the Cholesky factor of the posterior covariance + jitter I, is read column by column: item k with y = 0 and normals
e_k returns column k of L22.  Each premise a test relies on (schedule, substitution kernel, chunk size) is asserted
through the mirrors of the C conditions, so a retuned threshold fails here instead of silently testing something
else."""
import os
import sys

import numpy as np
import pytest

import test_lml_ard_gpu as LA
import test_posterior_draws_ext_gpu as E
from gp_b200 import capi
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import posterior_ard_ext as A  # noqa: E402

pytestmark = pytest.mark.gpu

TILE = 128
BIG_LIMIT = E.BIG_LIMIT


# ---- mirrors of the C host code -----------------------------------------------------------------------------------------
def ard_draws_chunk(n, m, D, B, limit, x_items=False, xs_items=False, y_items=False, z=False, mu=True):
    """Items per chunk under a workspace limit > 0: posterior_draws_pipeline (api_sample.cu) with the inputs of
    gpb200_posterior_draws_ard_batched (Handle.posterior_draws_ard_batched always passes mu; Xs = None stages X's
    layout).  Returns (Bc, fixed, per_item)."""
    np_ = E.tiles(n + m) * TILE
    per_item = 2 * np_ * np_ * 8 + 2 * np_ * 8
    xl, sl, yl = (n * D if x_items else 0), (m * D if xs_items else 0), (n if y_items else 0)
    inputs = E._pad256((B * xl + n * D) * 8) + E._pad256((B * sl + m * D) * 8) + E._pad256(B * (D + 2) * 8)
    fixed = (inputs + E._pad256((B * yl + n) * 8) + (E._pad256(B * m * 8) if z else 0) + (2 if mu else 1) * E._pad256(B * m * 8)
             + E._pad256(B * 4) + 6 * 256 + 4096)
    return min(B, (limit - fixed - 8192) // per_item, 65535), fixed, per_item


def ard_limit_for_chunk(n, m, D, B, chunk, **kw):
    _, fixed, per_item = ard_draws_chunk(n, m, D, B, 1 << 62, **kw)
    limit = fixed + 8192 + chunk * per_item + per_item // 2
    assert ard_draws_chunk(n, m, D, B, limit, **kw)[0] == chunk
    return limit


def one_chunk(n, m, D, B, **kw):
    return ard_draws_chunk(n, m, D, B, BIG_LIMIT, **kw)[0] == B


@pytest.fixture(scope="module")
def h():
    hd = capi.Handle(0)
    hd.set_workspace_limit(BIG_LIMIT)
    yield hd
    hd.close()


def limited_handle(limit):
    hd = capi.Handle(0)
    hd.set_workspace_limit(limit)
    return hd


def synth(n, m, D, seed, separate=True, k=2):
    """Training inputs X (n, D), prediction inputs Xs (m, D) or None, data y and k theta rows."""
    rng = np.random.default_rng(seed)
    X = rng.uniform(0.0, 4.0, (n, D))
    Xs = rng.uniform(-0.3, 4.3, (m, D)) if separate else None
    y = np.sin(X).sum(axis=1) / np.sqrt(D) + 0.1 * rng.standard_normal(n)
    th = np.column_stack([rng.uniform(0.8, 1.5, k), rng.uniform(1.0, 2.5, (k, D)) * np.sqrt(D), rng.uniform(0.1, 0.3, k)])
    return X, Xs, y, th


class ArdCase:
    """One shape with its theta rows, the sampled L22 columns, and the long-double and float64 references of each
    theta (the ARD twin of test_posterior_draws_ext_gpu.Case)."""

    def __init__(self, X, Xs, y, jitter, thetas, cols, seed):
        self.X, self.Xs, self.y, self.jitter = X, Xs, y, jitter
        self.n, self.m = X.shape[0], X.shape[0] if Xs is None else Xs.shape[0]
        self.thetas, self.cols = np.asarray(thetas, dtype=np.float64), np.asarray(cols)
        self.eps = np.random.default_rng(seed).standard_normal((len(self.thetas), self.m))
        self.ext = [A.posterior_ard_ext(X, Xs, y, th, jitter, self.eps[k]) for k, th in enumerate(self.thetas)]
        self.base = [A.posterior_ard_f64(X, Xs, y, th, jitter, self.eps[k]) for k, th in enumerate(self.thetas)]

    def items(self):
        TH, Y, Z = [], [], []
        for k, th in enumerate(self.thetas):
            for c in self.cols:
                TH.append(th); Y.append(np.zeros(self.n)); Z.append(np.eye(1, self.m, c)[0])
            TH.append(th); Y.append(self.y); Z.append(self.eps[k])
        return np.array(TH), np.array(Y), np.array(Z)

    def run(self, hd):
        TH, Y, Z = self.items()
        return hd.posterior_draws_ard_batched(self.X, Y, TH, Xs=self.Xs, jitter=self.jitter, z=Z)

    def check(self, fails, tag, draws, mu, info):
        if not np.all(info == 0):
            fails.append("%s: info %s" % (tag, np.unique(info)))
            return
        k1 = len(self.cols) + 1
        for k in range(len(self.thetas)):
            d, u = draws[k * k1:(k + 1) * k1], mu[k * k1:(k + 1) * k1]
            if not np.all(u[:-1] == 0.0):
                fails.append("%s theta %d: mu of y = 0 is not 0" % (tag, k))
            L = d[:-1].T
            if np.any(L[np.arange(self.m)[:, None] < self.cols[None, :]] != 0.0):
                fails.append("%s theta %d: L22 has entries above the diagonal" % (tag, k))
            e, b = self.ext[k], self.base[k]
            E.check_bound(fails, "%s th%d L22" % (tag, k), L, e.L22[:, self.cols], b.L22[:, self.cols], self.cols)
            E.check_bound(fails, "%s th%d mu" % (tag, k), u[-1], e.mu, b.mu)
            E.check_bound(fails, "%s th%d draw" % (tag, k), d[-1], e.draws[0], b.draws[0])


# ---- 1. parity with the extended-precision posterior --------------------------------------------------------------------
# (n, m) on and around the tile edges of n + m with a separate Xs; n alone (m = n) when predicting on X
SEPARATE = [(100, 28), (100, 29), (127, 1), (129, 127), (300, 213)]
ON_X = [64, 129, 300]
PARITY = [(D, n, m, True) for D in (1, 2, 3, 8) for n, m in SEPARATE] + [(D, n, n, False) for D in (1, 2, 3, 8) for n in ON_X]


@pytest.mark.parametrize("D, n, m, separate", PARITY)
def test_parity_with_the_extended_posterior(h, D, n, m, separate):
    X, Xs, y, th = synth(n, m, D, 1000 * D + n + m + separate, separate)
    cols = np.arange(m) if m <= 40 else E.sampled_columns(m, 4, n + m)
    c = ArdCase(X, Xs, y, 1e-8, th, cols, D + n)
    assert one_chunk(n, m, D, len(c.items()[0]), y_items=True, z=True)
    fails = []
    c.check(fails, "D=%d n=%d m=%d %s" % (D, n, m, "Xs" if separate else "X"), *c.run(h))
    E.report(fails)


# ---- 2. D = 1 is the order-0 model of gpb200_posterior_draws_batched -------------------------------------------------------
@pytest.mark.parametrize("n, m, B", [(300, 213, 8), (512, 512, 40)])
def test_one_dimension_matches_the_se_entry_point(h, n, m, B):
    rng = np.random.default_rng(n + m)
    t = np.sort(rng.uniform(0, 8, n))
    s = np.sort(rng.uniform(-0.5, 8.5, m)) if m != n else None
    y = np.sin(t) + 0.1 * rng.standard_normal(n)
    th = np.column_stack([rng.uniform(0.8, 1.5, B), rng.uniform(0.6, 1.5, B), rng.uniform(0.1, 0.3, B)])
    Z = rng.standard_normal((B, m))
    d0, mu0, i0 = h.posterior_draws_batched(t, y, th, order=0, s=s, jitter=1e-8, z=Z)
    d1, mu1, i1 = h.posterior_draws_ard_batched(t[:, None], y, th, Xs=None if s is None else s[:, None], jitter=1e-8, z=Z)
    assert np.all(i0 == 0) and np.all(i1 == 0)
    fails = []
    for b in range(B):
        assert E.relerr(mu1[b], mu0[b]) <= 1e-9, (b, E.relerr(mu1[b], mu0[b]))
        if b in (0, B - 1):
            e = A.posterior_ard_ext(t[:, None], None if s is None else s[:, None], y, th[b], 1e-8, Z[b])
            f = A.posterior_ard_f64(t[:, None], None if s is None else s[:, None], y, th[b], 1e-8, Z[b])
            E.check_bound(fails, "ard b=%d" % b, d1[b], e.draws[0], f.draws[0])
            E.check_bound(fails, "se b=%d" % b, d0[b], e.draws[0], f.draws[0])
    E.report(fails)


# ---- 3. invariances of the model --------------------------------------------------------------------------------------------
def _inv_inputs(seed=5, n=300, m=200, D=3, B=6):
    rng = np.random.default_rng(seed)
    X = rng.uniform(0, 4, (B, n, D))
    Xs = rng.uniform(0, 4, (B, m, D))
    Y = np.sin(X).sum(axis=2) + 0.1 * rng.standard_normal((B, n))
    th = np.column_stack([rng.uniform(0.8, 1.5, B), rng.uniform(1.5, 3.0, (B, D)), rng.uniform(0.1, 0.3, B)])
    Z = rng.standard_normal((B, m))
    return X, Xs, Y, th, Z


def _close(a, b, tol=1e-9):
    for k in range(a.shape[0]):
        assert E.relerr(a[k], b[k]) <= tol, (k, E.relerr(a[k], b[k]))


KW = dict(jitter=1e-4)   # a well-conditioned posterior covariance: rounding is not amplified


def test_permuting_columns_with_rho_changes_nothing(h):
    X, Xs, Y, th, Z = _inv_inputs()
    perm = np.array([2, 0, 1])
    thp = th.copy()
    thp[:, 1:4] = th[:, 1:4][:, perm]
    d0, mu0, i0 = h.posterior_draws_ard_batched(X, Y, th, Xs=Xs, z=Z, **KW)
    d1, mu1, i1 = h.posterior_draws_ard_batched(X[:, :, perm], Y, thp, Xs=Xs[:, :, perm], z=Z, **KW)
    assert np.all(i0 == 0) and np.all(i1 == 0)
    _close(mu1, mu0); _close(d1, d0)


def test_permuting_training_rows_with_y_changes_nothing(h):
    X, Xs, Y, th, Z = _inv_inputs()
    perm = np.random.default_rng(9).permutation(X.shape[1])
    d0, mu0, _ = h.posterior_draws_ard_batched(X, Y, th, Xs=Xs, z=Z, **KW)
    d1, mu1, i1 = h.posterior_draws_ard_batched(X[:, perm], Y[:, perm], th, Xs=Xs, z=Z, **KW)
    assert np.all(i1 == 0)
    _close(mu1, mu0); _close(d1, d0)


def test_scaling_a_column_and_its_rho_changes_nothing(h):
    X, Xs, Y, th, Z = _inv_inputs()
    Xc, Xsc, thc = X.copy(), Xs.copy(), th.copy()
    Xc[:, :, 1] *= 3.7; Xsc[:, :, 1] *= 3.7; thc[:, 2] *= 3.7
    d0, mu0, _ = h.posterior_draws_ard_batched(X, Y, th, Xs=Xs, z=Z, **KW)
    d1, mu1, i1 = h.posterior_draws_ard_batched(Xc, Y, thc, Xs=Xsc, z=Z, **KW)
    assert np.all(i1 == 0)
    _close(mu1, mu0); _close(d1, d0)


def test_a_constant_column_drops_out(h):
    X, Xs, Y, th, Z = _inv_inputs()
    X[:, :, 1] = 0.37; Xs[:, :, 1] = 0.37
    keep = [0, 2]
    d0, mu0, i0 = h.posterior_draws_ard_batched(X, Y, th, Xs=Xs, z=Z, **KW)
    d1, mu1, i1 = h.posterior_draws_ard_batched(X[:, :, keep], Y, th[:, [0, 1, 3, 4]], Xs=Xs[:, :, keep], z=Z, **KW)
    assert np.all(i0 == 0) and np.all(i1 == 0)
    _close(mu1, mu0, 1e-13); _close(d1, d0, 1e-13)


# ---- 4. the normal stream -------------------------------------------------------------------------------------------------
def test_zero_normals_give_the_mean(h):
    X, Xs, Y, th, _ = _inv_inputs(B=5)
    d, mu, info = h.posterior_draws_ard_batched(X, Y, th, Xs=Xs, z=np.zeros((5, Xs.shape[1])), jitter=1e-8)
    assert np.all(info == 0) and np.all(mu != 0.0)
    assert np.array_equal(E.bits(d), E.bits(mu))


def test_seed_stream_and_chunking_are_bit_identical(h):
    # N = 251 (two tile rows) and chunks of 2399 items of a 4798-item call: every launch makes the same schedule choice
    # (LA.same_schedule, the substitution kernel), and the second chunk starts at an odd offset of the normal stream
    n, m, D, B, chunk, seed = 150, 101, 3, 4798, 2399, 77
    assert LA.same_schedule(E.tiles(n + m), chunk, B) and E.uses_trsv_blocked(chunk) == E.uses_trsv_blocked(B)
    assert E.chunks(B, chunk) == [(0, chunk), (chunk, chunk)] and (chunk * m) % 2 == 1
    rng = np.random.default_rng(3)
    X, Xs = rng.uniform(0, 4, (n, D)), rng.uniform(0, 4, (m, D))
    y = np.sin(X).sum(axis=1)
    th = np.column_stack([rng.uniform(0.8, 1.5, B), rng.uniform(1.0, 3.0, (B, D)), rng.uniform(0.1, 0.3, B)])
    assert one_chunk(n, m, D, B) and one_chunk(n, m, D, B, z=True)
    ref = h.posterior_draws_ard_batched(X, y, th, Xs=Xs, seed=seed)
    assert np.all(ref[2] == 0)
    # item b's normals are numbers [b m, (b + 1) m) of the stream
    zs = h.normal_fill(seed, B * m).reshape(B, m)
    withz = h.posterior_draws_ard_batched(X, y, th, Xs=Xs, z=zs)
    limit = ard_limit_for_chunk(n, m, D, B, chunk)
    hc = limited_handle(limit)
    try:
        chunked = hc.posterior_draws_ard_batched(X, y, th, Xs=Xs, seed=seed)
        hc.set_workspace_limit(ard_limit_for_chunk(n, m, D, B, chunk, z=True))
        chunked_z = hc.posterior_draws_ard_batched(X, y, th, Xs=Xs, z=zs)
    finally:
        hc.close()
    for got in (withz, chunked, chunked_z):
        for a, b in zip(ref, got):
            assert np.array_equal(E.bits(a), E.bits(b))


# ---- 5. strides, guards and pointer modes ------------------------------------------------------------------------------------
def _colmajor_items(A):
    """(B, rows, D) -> (B, rows * D): each item column-major."""
    return np.ascontiguousarray(np.swapaxes(A, 1, 2)).reshape(A.shape[0], -1)


def _raw_call(hd, n, m, D, B, inputs, strides, jitter, seed, device, stream=None):
    outs = {"draws": np.full(B * m + 8, E.F64_SENTINEL, np.uint64).view(np.float64),
            "mu": np.full(B * m + 8, E.F64_SENTINEL, np.uint64).view(np.float64),
            "info": np.full(B + 8, E.I32_SENTINEL, np.int32)}
    bufs = dict(inputs, **outs)
    if device:
        import torch
        bufs = {k: (None if v is None else torch.from_numpy(v).cuda()) for k, v in bufs.items()}
        torch.cuda.synchronize()
        hd.set_stream(stream.cuda_stream)
        hd.set_pointer_mode(True)
    try:
        if device:
            hd.posterior_draws_ard_batched_device(n, m, D, B, bufs["X"], strides[0], bufs["Xs"], strides[1], bufs["y"],
                                                  strides[2], bufs["theta"], jitter, bufs["z"], seed, bufs["draws"],
                                                  bufs["mu"], bufs["info"])
        else:
            p = lambda k: capi._ptr(bufs.get(k))
            rc = hd.lib.gpb200_posterior_draws_ard_batched(hd._h, n, m, D, B, p("X"), strides[0], p("Xs"), strides[1], p("y"),
                                                           strides[2], p("theta"), jitter, p("z"), seed, p("draws"), p("mu"),
                                                           p("info"))
            assert rc == 0, hd.lib.gpb200_last_error(hd._h)
    finally:
        if device:
            stream.synchronize()          # only the caller's stream
            hd.set_pointer_mode(False)
    return {k: (None if v is None else (v.cpu().numpy() if device else v)) for k, v in bufs.items()}


@pytest.mark.parametrize("x_items, xs_items, y_items", [(True, True, True), (False, True, False), (True, False, True),
                                                        (False, False, False), (True, None, True), (False, None, False)])
def test_strides_guards_and_pointer_modes(h, x_items, xs_items, y_items):
    import torch
    B, n, D, seed, jitter = 5, 130, 3, 31, 1e-8
    m = n if xs_items is None else 97
    rng = np.random.default_rng(7)
    X = rng.uniform(0, 4, (B, n, D))
    Xs = rng.uniform(0, 4, (B, m, D))
    Y = np.sin(X).sum(axis=2) + 0.1 * rng.standard_normal((B, n))
    th = np.column_stack([rng.uniform(0.5, 2.0, B), rng.uniform(1.0, 3.0, (B, D)), rng.uniform(0.1, 0.3, B)])
    Z = rng.standard_normal((B, m))
    strides = (n * D + 37 if x_items else 0, (m * D + 3 if xs_items else 0) if xs_items is not None else 0,
               n + 5 if y_items else 0)
    dense = lambda A, per_item: A if per_item else A[0]
    inputs = {"X": E._strided(_colmajor_items(X), strides[0]),
              "Xs": None if xs_items is None else E._strided(_colmajor_items(Xs), strides[1]),
              "y": E._strided(Y, strides[2]), "theta": th.ravel().copy()}
    stream = torch.cuda.Stream()
    for z in (None, Z):
        ref_d, ref_mu, ref_info = h.posterior_draws_ard_batched(dense(X, x_items), dense(Y, y_items), th,
                                                                Xs=None if xs_items is None else dense(Xs, xs_items),
                                                                jitter=jitter, seed=seed, z=z)
        assert np.all(ref_info == 0)
        ins = dict(inputs, z=None if z is None else Z.ravel().copy())
        for device in (False, True):
            ctx = ("z" if z is not None else "seed", "device" if device else "host")
            got = _raw_call(h, n, m, D, B, {k: (None if v is None else v.copy()) for k, v in ins.items()}, strides, jitter,
                            seed, device, stream)
            for k, v in ins.items():
                assert v is None or np.array_equal(E.bits(got[k]), E.bits(v)), (ctx, k, "input modified")
            assert np.array_equal(E.bits(got["draws"][:B * m]), E.bits(ref_d.ravel())), ctx
            assert np.array_equal(E.bits(got["mu"][:B * m]), E.bits(ref_mu.ravel())), ctx
            assert np.all(E.bits(got["draws"][B * m:]) == E.F64_SENTINEL), ctx
            assert np.all(E.bits(got["mu"][B * m:]) == E.F64_SENTINEL), ctx
            assert np.array_equal(got["info"][:B], ref_info) and np.all(got["info"][B:] == E.I32_SENTINEL), ctx
    h.set_stream(torch.cuda.current_stream().cuda_stream)


# ---- 6. failed items ----------------------------------------------------------------------------------------------------------
def _failing(where, B, seed):
    """(X, Xs, Y, th, jitter, bad, theta of the bad item when it is well) of a batch whose item `bad` fails:
    "X" / "Xs": a NaN coordinate; "cov": every prediction point is beyond the kernel's reach of X and of the others
    except one pair at Xs rows 200 and 201 (k = 1/2 alpha^2 between them); with jitter -0.75 the pair's 2 x 2 posterior
    covariance is positive definite for alpha = 2 and indefinite for alpha = 1, so that theta fails at pivot n + 202."""
    n, m, D = 200, 250, 3
    rng = np.random.default_rng(seed)
    bad = B * 2 // 3
    if where == "cov":
        X = np.tile(rng.uniform(0, 4, (n, D)), (B, 1, 1))
        Xs = np.tile(1000.0 + 100.0 * np.arange(m)[:, None] * np.ones(D), (B, 1, 1))
        Xs[:, 201] = Xs[:, 200]
        Xs[:, 201, 0] += np.sqrt(2 * np.log(2.0))
        th = np.column_stack([np.full(B, 2.0), np.ones((B, D)), rng.uniform(0.1, 0.3, B)])
        good_th = th[bad].copy()
        th[bad, 0] = 1.0
        return X, Xs, np.sin(X).sum(axis=2), th, -0.75, bad, good_th
    X = rng.uniform(0, 4, (B, n, D))
    Xs = rng.uniform(0, 4, (B, m, D))
    th = np.column_stack([rng.uniform(0.8, 1.5, B), rng.uniform(1.0, 2.5, (B, D)), rng.uniform(0.1, 0.3, B)])
    Xb = X if where == "X" else Xs
    Xb[bad, 150 if where == "X" else 100, 1] = np.nan
    return X, Xs, np.sin(np.nan_to_num(X)).sum(axis=2), th, 1e-2, bad, th[bad].copy()


@pytest.mark.parametrize("batch", ["lookahead", "left", "chunked"])
@pytest.mark.parametrize("where", ["X", "Xs", "cov"])
def test_failed_item_reports_the_oracle_pivot_and_leaves_the_others_alone(h, where, batch):
    n, m, D = 200, 250, 3
    B = {"lookahead": 8, "left": 100, "chunked": 70}[batch]
    X, Xs, Y, th, jitter, bad, good_th = _failing(where, B, {"X": 1, "Xs": 2, "cov": 3}[where])
    want = A.posterior_ard_ext(X[bad], Xs[bad], Y[bad], th[bad], jitter).info
    assert want == {"X": 151, "Xs": n + 101, "cov": n + 202}[where]
    assert A.posterior_ard_ext(X[bad], Xs[bad], Y[bad], good_th, jitter).info == 0 or where != "cov"
    Xg, Xsg, thg = X.copy(), Xs.copy(), th.copy()
    thg[bad] = good_th
    if where == "X":
        Xg[bad, 150, 1] = 0.5
    elif where == "Xs":
        Xsg[bad, 100, 1] = 0.5
    kw = dict(jitter=jitter, seed=9)
    hd = h
    if batch == "chunked":
        # chunks of 40 and 30 items: the failed item is in the second chunk, and both substitution kernels run
        limit = ard_limit_for_chunk(n, m, D, B, 40, x_items=True, xs_items=True, y_items=True)
        assert E.uses_trsv_blocked(40) and not E.uses_trsv_blocked(30) and E.chunks(B, 40) == [(0, 40), (40, 30)]
        hd = limited_handle(limit)
    else:
        assert E.chol_schedule(n + m, B)[0] == batch and one_chunk(n, m, D, B, x_items=True, xs_items=True, y_items=True)
    try:
        good_d, good_mu, good_info = hd.posterior_draws_ard_batched(Xg, Y, thg, Xs=Xsg, **kw)
        d, mu, info = hd.posterior_draws_ard_batched(X, Y, th, Xs=Xs, **kw)
    finally:
        if hd is not h:
            hd.close()
    assert np.all(good_info == 0)
    assert info[bad] == want, (info[bad], want)
    assert np.all(np.isnan(d[bad])) and np.all(np.isnan(mu[bad]))
    keep = np.arange(B) != bad
    assert np.all(info[keep] == 0)
    assert np.array_equal(E.bits(d[keep]), E.bits(good_d[keep])) and np.array_equal(E.bits(mu[keep]), E.bits(good_mu[keep]))


# ---- 7. schedule knobs -----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("knob", ["cfg1", "cfg2", "cfg3", "GPB200_DIAG_SPLIT", "GPB200_LOOKAHEAD"])
def test_every_schedule_knob_agrees_with_the_oracle(knob):
    hd = LA.handle_with(**({knob: 0} if knob.startswith("GPB200") else {}))
    try:
        hd.set_workspace_limit(BIG_LIMIT)
        if knob.startswith("cfg"):
            hd.set_gemm_config(int(knob[3]))
        fails = []
        for D, n, m in ((2, 300, 213), (8, 400, 350)):
            X, Xs, y, th = synth(n, m, D, 7 * D + n)
            c = ArdCase(X, Xs, y, 1e-8, th, E.sampled_columns(m, 6, m), n)
            assert E.chol_schedule(n + m, len(c.items()[0]))[0] == "lookahead"
            c.check(fails, "%s D=%d" % (knob, D), *c.run(hd))
        E.report(fails)
    finally:
        hd.close()


# ---- 8. bad arguments ---------------------------------------------------------------------------------------------------------
def test_bad_arguments_return_negative_launch_nothing_and_write_nothing(h):
    lib, p = h.lib, capi._ptr
    n, m, D, B = 50, 30, 2, 3
    X = np.zeros(n * D * B); Xs = np.zeros(m * D * B); y = np.zeros(n * B); th = np.ones((B, D + 2))
    draws = np.full(B * m, -7.25); mu = np.full(B * m, -7.25); info = np.full(B, -3, dtype=np.int32)

    def call(n_=n, m_=m, D_=D, B_=B, xs=0, xss=0, ys=0, X_=X, Xs_=Xs, y_=y, th_=th, draws_=draws, info_=info):
        return lib.gpb200_posterior_draws_ard_batched(h._h, n_, m_, D_, B_, p(X_), xs, p(Xs_), xss, p(y_), ys, p(th_), 1e-8,
                                                      None, 1, p(draws_), p(mu), p(info_))

    before = h.launch_count()
    bad = [{"n_": 0}, {"n_": -3}, {"m_": 0}, {"B_": -1}, {"D_": 0}, {"D_": 9}, {"xs": n * D - 1}, {"xss": m * D - 1},
           {"ys": n - 1}, {"Xs_": None}, {"X_": None}, {"y_": None}, {"th_": None}, {"draws_": None}, {"info_": None},
           {"n_": 40000, "m_": 30000}]
    for kw in bad:
        rc = call(**kw)
        assert rc < 0, kw
        assert lib.gpb200_last_error(h._h), kw
    assert h.launch_count() == before
    assert np.all(draws == -7.25) and np.all(mu == -7.25) and np.all(info == -3)
    assert call(B_=0) == 0 and h.launch_count() == before
    assert np.all(draws == -7.25) and np.all(info == -3)
