"""gpb200_posterior_draws_batched against the extended-precision posterior (oracle/posterior_ext.py), at the shapes the
entry point was built and measured for, on the tile boundaries of the joint matrix, on strided inputs in both pointer
modes, on failed items, and on every chunk of the normal stream.

Yardstick.  posterior_ext factors the joint prior covariance J in long double; posterior_f64 is the same computation
in float64 through LAPACK, the baseline.  A GPU result X is compared with the long-double X_ext through the
baseline's own error, so a tolerance follows the conditioning of its case: with E_gpu = |X - X_ext| and
E_base = |X_f64 - X_ext|, per 128 x 128 tile (per 128-row block of a vector)
    max E_gpu <= TILE_FACTOR max(max E_base, F max|X_ext|),   ||E_gpu||_F <= FRO_FACTOR ||E_base||_F + F ||X_ext||_F.
The factors are wider than the rounding of one float64 factorisation against another would suggest because the
posterior factor comes out of the cancellation Kss - L21 L21^T: its rounding depends on the order in which the
products are accumulated, and the GPU sums 128-deep tile products in another order than LAPACK.  Measured on a B200:
per tile up to 22 times the baseline (a diagonal tile of L22 at the lorenz shape, B = 32), in Frobenius norm up to
4.9 times (order 2, B = 32).
L22 is the unique Cholesky factor of the posterior covariance + jitter I, so it is compared element by element: item
k with y = 0 and normals e_k returns column k of L22.  A batch holds a few theta, each with the unit vectors of the
first and last column of every tile column of L22 (so every lower tile of L22 is sampled) plus random columns, and
one item with the data and random normals (mu and a draw).

Each test asserts the premise it targets (Cholesky schedule, substitution kernel, chunk sizes, far-tile share, the
identity posterior) through the mirrors of the C conditions below, so a retuned threshold fails here instead of
silently testing something else.  The checks of one test are collected and reported together."""
import itertools

import numpy as np
import pytest

from gp_b200 import capi
from oracle import chol_deriv_ext as X
from oracle import philox
from oracle import posterior_ext as P

pytestmark = pytest.mark.gpu

TILE = 128
NSM = 148
F = 1e-14                                      # floor of the bounds, relative to max|X_ext|
TILE_FACTOR = 50
FRO_FACTOR = 8
BIG_LIMIT = 8 << 30                            # workspace limit of the module's handle: every call below fits one chunk
F64_SENTINEL = np.uint64(0x7FF8DEADBEEF5A5A)   # a quiet NaN whose payload no kernel produces
I32_SENTINEL = np.int32(-1515870811)


def tiles(n):
    return (n + TILE - 1) // TILE


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a.view(np.uint32)


# ---- branch predicates, mirrored from the C host code -----------------------------------------------------------------
def chol_schedule(N, bc):
    """chol_batched (engine.cu:281-312) on a chunk of bc items with the default knobs: ("lookahead", panel tiles) when
    chol_uses_lookahead (engine.cu:204-208), with the panel of chol_lookahead_panel (engine.cu:213-216); otherwise
    chol_panel_tiles (engine.cu:179-182): ("left", nt) for one panel, ("right", 8) for 8-tile panels with
    right-looking trailing updates."""
    nt = tiles(N)
    if bc <= 64 and bc * nt <= 256 and nt >= 3:
        return "lookahead", (8 if nt >= 192 else 4 if nt >= 48 else 2 if nt >= 24 else 1)
    pt = nt if (bc >= 64 or nt <= 8) else 8
    return ("left" if pt == nt else "right"), pt


def uses_trsv_blocked(bc):
    """L11^-1 y of a chunk: trsv_blocked from 32 items on, trsv_sweep below (api_sample.cu:153-154)."""
    return bc >= 32


def _pad256(b):
    return (b + 255) & ~255


def draws_chunk(n, m, B, limit, t_items=False, s_items=False, y_items=False, z=False, mu=True):
    """Items per chunk under a workspace limit > 0: the fixed / per_item arithmetic of api_sample.cu:108-127
    (Handle.posterior_draws_batched always passes mu).  Returns (Bc, fixed, per_item)."""
    np_ = tiles(n + m) * TILE
    mat = np_ * np_
    tl, sl, yl = (n if t_items else 0), (m if s_items else 0), (n if y_items else 0)
    per_item = 2 * mat * 8 + 2 * np_ * 8
    fixed = (_pad256((B * tl + n) * 8) + _pad256((B * sl + m) * 8) + _pad256((B * yl + n) * 8) + _pad256(B * 3 * 8)
             + (_pad256(B * m * 8) if z else 0) + (2 if mu else 1) * _pad256(B * m * 8) + _pad256(B * 4) + 6 * 256 + 4096)
    return min(B, (limit - fixed - 8192) // per_item, 65535), fixed, per_item


def limit_for_chunk(n, m, B, chunk, **kw):
    _, fixed, per_item = draws_chunk(n, m, B, 1 << 62, **kw)
    limit = fixed + 8192 + chunk * per_item + per_item // 2
    assert draws_chunk(n, m, B, limit, **kw)[0] == chunk
    return limit


def chunks(B, Bc):
    return [(b0, min(Bc, B - b0)) for b0 in range(0, B, Bc)]


def normal_pairs(offset, length):
    """Box-Muller pairs normal_fill_kernel generates for a chunk (rng.cu:39-40), and the one-pass limit of its grid
    (launch_normal_fill, rng.cu:58-59: at most 148 * 8 blocks of 256 threads)."""
    return (length + (offset & 1) + 1) // 2, NSM * 8 * 256


# ---- fixtures and helpers ---------------------------------------------------------------------------------------------
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


def one_chunk(n, m, B, **kw):
    return draws_chunk(n, m, B, BIG_LIMIT, **kw)[0] == B


def check_bound(fails, what, got, ext, base, cols=None, f=F):
    """The per-tile and Frobenius bounds of the module docstring on rows x k arrays; cols are the L22 column indices
    of the k columns (None: one vector).  Appends a message per violated bound; returns the worst ratios (tile ratio
    max E_gpu / max(max E_base, f max|X_ext|), allowed TILE_FACTOR; Frobenius ratio, allowed 1)."""
    got, ext, base = (np.asarray(a, dtype=np.float64).reshape(np.shape(a)[0], -1) for a in (got, ext, base))
    cols = np.zeros(got.shape[1], dtype=int) if cols is None else np.asarray(cols)
    Eg, Eb = np.abs(got - ext), np.abs(base - ext)
    floor = f * float(np.max(np.abs(ext)))
    worst, where = 0.0, None
    for I in range(tiles(got.shape[0])):
        r = slice(I * TILE, (I + 1) * TILE)
        for J in np.unique(cols // TILE):
            c = cols // TILE == J
            ratio = float(Eg[r][:, c].max()) / max(float(Eb[r][:, c].max()), floor, 1e-300)
            if ratio > worst:
                worst, where = ratio, (I, int(J))
    fro = float(np.linalg.norm(Eg)) / max(FRO_FACTOR * float(np.linalg.norm(Eb)) + f * float(np.linalg.norm(ext)), 1e-300)
    if worst > TILE_FACTOR:
        fails.append("%s: tile %s max E_gpu = %.1f x max(E_base, floor) (allowed %d)" % (what, where, worst, TILE_FACTOR))
    if fro > 1:
        fails.append("%s: ||E_gpu||_F = %.2f x (%d ||E_base||_F + F ||X_ext||_F)" % (what, fro, FRO_FACTOR))
    print("ratios %-40s tile %7.3f at %s  fro %6.3f" % (what, worst, where, fro))
    return worst, fro


def sampled_columns(m, n_random, seed):
    """First and last column of every tile column of L22, plus n_random other columns."""
    edges = sorted({c for J in range(tiles(m)) for c in (J * TILE, min(m, (J + 1) * TILE) - 1)})
    rest = np.setdiff1d(np.arange(m), edges)
    rnd = np.random.default_rng(seed).choice(rest, min(n_random, rest.size), replace=False) if rest.size else []
    return np.array(sorted(edges + [int(c) for c in rnd]))


class Case:
    """One shape: grids, data, order, jitter, theta rows and the sampled L22 columns, with the long-double and
    float64 references of each theta (computed once)."""

    def __init__(self, t, s, y, order, jitter, thetas, cols, seed):
        self.t, self.s, self.y, self.order, self.jitter = t, s, y, order, jitter
        self.n, self.m = len(t), len(t) if s is None else len(s)
        self.thetas, self.cols = np.asarray(thetas, dtype=np.float64), np.asarray(cols)
        self.eps = np.random.default_rng(seed).standard_normal((len(self.thetas), self.m))
        self.ext = [P.posterior_ext(t, s, y, th, order, jitter, self.eps[k]) for k, th in enumerate(self.thetas)]
        self.base = [P.posterior_f64(t, s, y, th, order, jitter, self.eps[k]) for k, th in enumerate(self.thetas)]

    def items(self):
        """Per theta: the unit vectors of the sampled columns with y = 0, then the data with random normals."""
        TH, Y, Z = [], [], []
        for k, th in enumerate(self.thetas):
            for c in self.cols:
                TH.append(th); Y.append(np.zeros(self.n)); Z.append(np.eye(1, self.m, c)[0])
            TH.append(th); Y.append(self.y); Z.append(self.eps[k])
        return np.array(TH), np.array(Y), np.array(Z)

    def run(self, hd, B):
        """Every item, in calls of exactly B items (the last call padded with repeats), so each call takes the
        schedule of B."""
        TH, Y, Z = self.items()
        K = len(TH)
        idx = np.concatenate([np.arange(K), np.arange((-K) % B) % K])
        outs = [hd.posterior_draws_batched(self.t, Y[idx[i:i + B]], TH[idx[i:i + B]], order=self.order, s=self.s,
                                           jitter=self.jitter, z=Z[idx[i:i + B]]) for i in range(0, len(idx), B)]
        return tuple(np.concatenate(a)[:K] for a in zip(*outs))

    def base_errors(self):
        """Per item of items(): the baseline's largest error of that item's draw."""
        out = []
        for e, b in zip(self.ext, self.base):
            out += [float(np.max(np.abs(b.L22[:, c] - e.L22[:, c]))) for c in self.cols]
            out.append(float(np.max(np.abs(b.draws - e.draws))))
        return np.array(out)

    def check(self, fails, tag, draws, mu, info):
        if not np.all(info == 0):
            fails.append("%s: info %s" % (tag, np.unique(info)))
            return
        k1 = len(self.cols) + 1
        for k in range(len(self.thetas)):
            d, u = draws[k * k1:(k + 1) * k1], mu[k * k1:(k + 1) * k1]
            if not np.all(u[:-1] == 0.0):
                fails.append("%s theta %d: mu of y = 0 is not 0" % (tag, k))
            L = d[:-1].T                                      # m x |cols|: the sampled columns of L22
            if np.any(L[np.arange(self.m)[:, None] < self.cols[None, :]] != 0.0):
                fails.append("%s theta %d: L22 has entries above the diagonal" % (tag, k))
            e, b = self.ext[k], self.base[k]
            check_bound(fails, "%s th%d L22" % (tag, k), L, e.L22[:, self.cols], b.L22[:, self.cols], self.cols)
            check_bound(fails, "%s th%d mu" % (tag, k), u[-1], e.mu, b.mu)
            check_bound(fails, "%s th%d draw" % (tag, k), d[-1], e.draws[0], b.draws[0])


def report(fails):
    assert not fails, "\n".join(fails)


# ---- A. the reference shapes in every schedule they take ----------------------------------------------------------------
def _shape(name):
    """The shapes and theta ranges of tools/bench_posterior_draws.py, two theta each; order 2 on a gp_derivs.py-style
    grid (derivative grid wider than the data), and one wide matrix of 24 tile rows with a single theta."""
    rng = np.random.default_rng({"pendulum": 1, "lorenz": 2, "ch2": 3, "order2": 4, "wide": 5}[name])
    u = lambda lo, hi, k=2: rng.uniform(lo, hi, k)
    if name == "pendulum":
        t = np.linspace(0.0, 10.0, 512)
        y = np.sin(t) * np.exp(-0.1 * t) + 0.05 * rng.standard_normal(512)
        return Case(t, None, y, 1, 1e-8, np.column_stack([u(0.8, 1.5), u(0.8, 2.0), u(0.03, 0.1)]),
                    sampled_columns(512, 6, 1), 11)
    if name == "lorenz":
        t = np.linspace(0.0, 20.0, 512)
        y = 8.0 * np.sin(0.7 * t) + np.cos(1.9 * t) + 0.1 * rng.standard_normal(512)
        # the bench's length scales give far-tile shares of L22 below 1e-2; a longer one (rho = 1.6) is added
        th = np.vstack([np.column_stack([u(3.0, 8.0), u(0.6, 1.2), u(0.05, 0.2)]), [5.0, 1.6, 0.1]])
        return Case(t, np.linspace(0.0, 20.0, 1024), y, 1, 1e-6, th, sampled_columns(1024, 8, 2), 12)
    if name == "ch2":
        xd = np.array([-4.0, -3.0, -1.0, 2.0])
        return Case(xd, np.linspace(-5.0, 5.0, 1000), np.sin(xd), 0, 1e-10,
                    np.column_stack([u(0.8, 1.2), u(0.8, 1.5), np.zeros(2)]), sampled_columns(1000, 8, 3), 13)
    if name == "order2":
        t = np.linspace(0.0, 5.0, 500)
        y = np.sin(2 * t) + 0.1 * rng.standard_normal(500)
        return Case(t, np.linspace(-0.5, 5.5, 650), y, 2, 1e-8, np.column_stack([u(0.8, 1.5), u(0.8, 2.0), u(0.05, 0.2)]),
                    sampled_columns(650, 6, 4), 14)
    t = np.linspace(0.0, 20.0, 1024)
    y = np.sin(t) + 0.1 * rng.standard_normal(1024)
    return Case(t, np.linspace(0.0, 20.0, 2048), y, 1, 1e-6, [[1.5, 2.5, 0.1]], sampled_columns(2048, 4, 5), 15)


# shape -> (B, schedule kind, panel tiles) of every batch size it is run at
SHAPES = {
    "pendulum": [(1, "lookahead", 1), (16, "lookahead", 1), (200, "left", 8)],
    "lorenz": [(1, "lookahead", 1), (16, "lookahead", 1), (32, "right", 8), (100, "left", 12)],
    "ch2": [(1, "lookahead", 1), (64, "left", 8)],
    "order2": [(1, "lookahead", 1), (32, "right", 8)],
    "wide": [(1, "lookahead", 2)],
}
_cases = {}


@pytest.fixture(scope="module")
def shape_case():
    def get(name):
        if name not in _cases:
            _cases[name] = _shape(name)
        return _cases[name]
    return get


@pytest.mark.parametrize("name", sorted(SHAPES))
def test_reference_shapes_against_the_extended_posterior_in_every_schedule(h, shape_case, name):
    c = shape_case(name)
    N = c.n + c.m
    # the far tiles of L22 carry weight, so the per-tile bound checks them
    share = max(X.far_tile_share(e.L22) for e in c.ext)
    assert share >= 1e-2, (name, share)
    fails, runs = [], {}
    for B, kind, pt in SHAPES[name]:
        assert chol_schedule(N, B) == (kind, pt), (name, B, chol_schedule(N, B))
        assert one_chunk(c.n, c.m, B, y_items=True, z=True), (name, B)
        runs[B] = c.run(h, B)
        c.check(fails, "%s B=%d" % (name, B), *runs[B])
    # the same item in each batch size: mu to 1e-12; a draw (a column of L22, or mu + L22 eps) to 1e-12 or, where the
    # posterior covariance is ill-conditioned, to the sum of the per-tile allowances of the two (2 TILE_FACTOR times the
    # baseline's error of that item; a schedule's accumulation order moves it as much as LAPACK's does)
    B0 = SHAPES[name][0][0]
    base_err = c.base_errors()
    for B, _, _ in SHAPES[name][1:]:
        worst = 0.0
        for k in range(len(base_err)):
            if relerr(runs[B][1][k], runs[B0][1][k]) > 1e-12 and np.any(runs[B0][1][k] != 0):
                fails.append("%s item %d mu: B=%d vs B=%d differ by %.2e" % (name, k, B, B0, relerr(runs[B][1][k], runs[B0][1][k])))
            a, b = runs[B][0][k], runs[B0][0][k]
            diff, allowed = float(np.max(np.abs(a - b))), max(1e-12 * float(np.max(np.abs(b))), 2 * TILE_FACTOR * base_err[k])
            worst = max(worst, diff / allowed)
            if diff > allowed:
                fails.append("%s item %d draw: B=%d vs B=%d differ by %.2e (allowed %.2e)" % (name, k, B, B0, diff, allowed))
        print("ratios %-40s cross-batch %.3f" % ("%s B=%d vs B=%d" % (name, B, B0), worst))
    report(fails)


# ---- B. tile boundaries of the joint matrix -------------------------------------------------------------------------------
# n on / one below a multiple of 128; m and n + m on, one below and one above one
BOUNDARY = [(128, 127), (128, 129), (128, 256), (255, 128), (255, 129), (255, 130), (384, 1), (384, 127), (384, 257),
            (1, 1100), (1100, 1)]


@pytest.mark.parametrize("order", [0, 1, 2])
@pytest.mark.parametrize("n, m", BOUNDARY)
def test_tile_boundaries_of_the_joint_matrix(h, n, m, order):
    rng = np.random.default_rng(100 * n + m + order)
    t, s = np.sort(rng.uniform(0, 6, n)), np.sort(rng.uniform(-0.5, 6.5, m))
    y = np.sin(t) + 0.1 * rng.standard_normal(n)
    cols = np.arange(m) if m <= 300 else sampled_columns(m, 8, m)
    c = Case(t, s, y, order, 1e-8, [[1.3, 0.9, 0.1 + 0.05 * order]], cols, m)
    B = len(cols) + 1
    assert one_chunk(n, m, B, y_items=True, z=True)
    fails = []
    c.check(fails, "n=%d m=%d p=%d" % (n, m, order), *c.run(h, B))
    report(fails)


# ---- C. the pivot index and failed items ----------------------------------------------------------------------------------
def _failing_batch(n, m, B, seed):
    rng = np.random.default_rng(seed)
    T = np.tile(np.linspace(0.0, 8.0, n), (B, 1)) + rng.uniform(-0.01, 0.01, (B, n))
    S = np.tile(np.linspace(-0.5, 8.5, m), (B, 1))
    Y = np.sin(T) + 0.1 * rng.standard_normal((B, n))
    th = np.column_stack([rng.uniform(0.8, 1.5, B), rng.uniform(0.7, 1.5, B), rng.uniform(0.1, 0.3, B)])
    return T, S, Y, th


# (where the NaN is, n, its index, the info the header promises): a later tile row of K, a later tile of the posterior
# covariance, the first pivot of the posterior covariance
PIVOTS = [("t", 400, 300, 301), ("s", 400, 200, 601), ("s", 256, 0, 257)]


@pytest.mark.parametrize("batch", ["lookahead", "left", "chunked"])
@pytest.mark.parametrize("where, n, k, want", PIVOTS)
def test_failed_item_reports_its_pivot_and_leaves_the_others_alone(h, where, n, k, want, batch):
    m = 300
    N = n + m
    B, bad = {"lookahead": (8, 5), "left": (64, 50), "chunked": (70, 50)}[batch]
    T, S, Y, th = _failing_batch(n, m, B, n + k)
    Tb, Sb = T.copy(), S.copy()
    (Tb if where == "t" else Sb)[bad, k] = np.nan
    # a jitter that keeps the posterior covariance well-conditioned: the chunked and unchunked calls take other
    # schedules and substitution kernels, and agree to 1e-12 only where rounding is not amplified
    kw = dict(order=1, jitter=1e-2, seed=9)
    hd = h
    if batch == "chunked":
        # chunks of 40 and 30 items: the failed item is in the second chunk, and both substitution kernels run
        limit = limit_for_chunk(n, m, B, 40, t_items=True, s_items=True, y_items=True)
        assert uses_trsv_blocked(40) and not uses_trsv_blocked(30) and chunks(B, 40) == [(0, 40), (40, 30)]
        hd = limited_handle(limit)
    else:
        assert chol_schedule(N, B)[0] == batch and one_chunk(n, m, B, t_items=True, s_items=True, y_items=True)
    try:
        good_d, good_mu, good_info = hd.posterior_draws_batched(T, Y, th, s=S, **kw)
        d, mu, info = hd.posterior_draws_batched(Tb, Y, th, s=Sb, **kw)
    finally:
        if hd is not h:
            hd.close()
    assert np.all(good_info == 0)
    assert info[bad] == want, (info[bad], want)
    assert np.all(np.isnan(d[bad])) and np.all(np.isnan(mu[bad]))
    keep = np.arange(B) != bad
    assert np.all(info[keep] == 0)
    assert np.array_equal(bits(d[keep]), bits(good_d[keep])) and np.array_equal(bits(mu[keep]), bits(good_mu[keep]))
    if batch == "chunked":
        assert one_chunk(n, m, B, t_items=True, s_items=True, y_items=True)
        d1, mu1, info1 = h.posterior_draws_batched(Tb, Y, th, s=Sb, **kw)
        assert np.array_equal(info1, info)
        for b in np.flatnonzero(keep):
            assert relerr(d[b], d1[b]) < 1e-12 and relerr(mu[b], mu1[b]) < 1e-12, b


# ---- D. strides, guards and pointer modes of the C entry point --------------------------------------------------------------
def _strided(rows, stride):
    """(B, L) rows laid out `stride` apart in a NaN-filled buffer with an 8-element NaN guard; stride 0: row 0 only."""
    B, L = rows.shape
    if stride == 0:
        return np.concatenate([rows[0], np.full(8, np.nan)])
    full = np.full((B - 1) * stride + L + 8, np.nan)
    for b in range(B):
        full[b * stride:b * stride + L] = rows[b]
    return full


def _raw_call(hd, n, m, order, B, inputs, strides, jitter, seed, with_mu, device):
    """Calls the C entry point on the buffers of `inputs` (t, s or None, y, theta, z or None) with output buffers
    B * m (B for info) long plus an 8-element sentinel guard.  Returns the output buffers and the input buffers as
    they are after the call."""
    outs = {"draws": np.full(B * m + 8, F64_SENTINEL, np.uint64).view(np.float64),
            "info": np.full(B + 8, I32_SENTINEL, np.int32)}
    if with_mu:
        outs["mu"] = np.full(B * m + 8, F64_SENTINEL, np.uint64).view(np.float64)
    bufs = dict(inputs, **outs)
    if device:
        import torch
        bufs = {k: (None if v is None else torch.from_numpy(v).cuda()) for k, v in bufs.items()}
        stream = torch.cuda.current_stream()
        hd.set_stream(stream.cuda_stream)
        hd.set_pointer_mode(True)
    ptr = lambda k: None if bufs.get(k) is None else (bufs[k].data_ptr() if device else bufs[k].ctypes.data)
    try:
        rc = hd.lib.gpb200_posterior_draws_batched(hd._h, n, m, order, B, ptr("t"), strides[0], ptr("s"), strides[1], ptr("y"),
                                                   strides[2], ptr("theta"), jitter, ptr("z"), seed, ptr("draws"), ptr("mu"),
                                                   ptr("info"))
    finally:
        if device:
            stream.synchronize()
            hd.set_pointer_mode(False)
    assert rc == 0, hd.lib.gpb200_last_error(hd._h)
    return {k: (None if v is None else (v.cpu().numpy() if device else v)) for k, v in bufs.items()}


# (t, s, y) per item (True) or shared (False); s None predicts on t
LAYOUTS = [(tp, sp, yp) for tp, sp, yp in itertools.product((True, False), repeat=3)] + [(True, None, True), (False, None, False)]


@pytest.mark.parametrize("t_items, s_items, y_items", LAYOUTS)
def test_strides_guards_and_pointer_modes(h, t_items, s_items, y_items):
    B, n, order, seed, jitter = 5, 130, 1, 31, 1e-8
    m = n if s_items is None else 97
    rng = np.random.default_rng(7)
    T = np.sort(rng.uniform(0, 6, (B, n)), axis=1)
    S = np.sort(rng.uniform(-0.5, 6.5, (B, m)), axis=1)
    Y = np.sin(T) + 0.1 * rng.standard_normal((B, n))
    th = np.column_stack([rng.uniform(0.5, 2.0, B), rng.uniform(0.6, 1.5, B), rng.uniform(0.1, 0.3, B)])
    Z = rng.standard_normal((B, m))
    strides = (n + 37 if t_items else 0, (m + 1 if s_items else 0) if s_items is not None else 0, n + 5 if y_items else 0)
    dense = lambda A, per_item: A if per_item else A[0]
    t_arg, y_arg = dense(T, t_items), dense(Y, y_items)
    s_arg = None if s_items is None else dense(S, s_items)
    inputs = {"t": _strided(T, strides[0]), "s": None if s_items is None else _strided(S, strides[1]),
              "y": _strided(Y, strides[2]), "theta": th.ravel().copy()}
    for z in (None, Z):
        ref_d, ref_mu, ref_info = h.posterior_draws_batched(t_arg, y_arg, th, order=order, s=s_arg, jitter=jitter,
                                                            seed=seed, z=z)
        assert np.all(ref_info == 0)
        ins = dict(inputs, z=None if z is None else Z.ravel().copy())
        for device, with_mu in itertools.product((False, True), (True, False)):
            ctx = ("z" if z is not None else "seed", "device" if device else "host", "mu" if with_mu else "mu = NULL")
            got = _raw_call(h, n, m, order, B, {k: (None if v is None else v.copy()) for k, v in ins.items()}, strides, jitter,
                            seed, with_mu, device)
            for k, v in ins.items():
                assert v is None or np.array_equal(bits(got[k]), bits(v)), (ctx, k, "input modified")
            assert np.array_equal(bits(got["draws"][:B * m]), bits(ref_d.ravel())), ctx
            assert np.all(bits(got["draws"][B * m:]) == F64_SENTINEL), ctx
            assert np.array_equal(got["info"][:B], ref_info) and np.all(got["info"][B:] == I32_SENTINEL), ctx
            if with_mu:
                assert np.array_equal(bits(got["mu"][:B * m]), bits(ref_mu.ravel())), ctx
                assert np.all(bits(got["mu"][B * m:]) == F64_SENTINEL), ctx


# ---- E. the normal stream, read through an identity posterior -------------------------------------------------------------
def _identity_posterior(m):
    """order 0, n = 1, t = [0], s = 100, 200, ..., alpha = rho = 1, jitter 0: every kernel value between two distinct
    points is exp(-5000 k^2) = 0 in float64, so Ks = 0, cov = I, L22 = I, mu = 0 and the draws are the normals."""
    t, s, theta = np.array([0.0]), 100.0 * np.arange(1, m + 1), np.array([1.0, 1.0, 0.5])
    J = P.joint_cov(t, s, theta, 0, 0.0)
    assert np.array_equal(J, np.diag(np.r_[1.25, np.ones(m)]))
    return t, s, np.array([0.3]), theta


@pytest.mark.parametrize("B, Bc", [(11, 3), (11, 2), (4800, 4800), (4800, 4775)])
def test_draws_of_an_identity_posterior_are_the_normal_stream(h, B, Bc):
    m, seed = 127, 2024
    t, s, y, theta = _identity_posterior(m)
    TH = np.tile(theta, (B, 1))
    parts = chunks(B, Bc)
    if B == 11:
        # chunks of 3 and of 2 items of 127 normals start at odd and even offsets with odd and even lengths
        cover = {(b0 * m % 2, bc * m % 2) for c in (3, 2) for b0, bc in chunks(B, c)}
        assert cover == {(0, 0), (0, 1), (1, 0), (1, 1)}
    else:
        # the first chunk is longer than one pass of the grid-stride loop; the second one starts at an odd offset
        npairs, one_pass = normal_pairs(0, Bc * m)
        assert npairs > one_pass
        assert len(parts) == 1 or (parts[1][0] * m) % 2 == 1
    limit = limit_for_chunk(1, m, B, Bc) if Bc < B else BIG_LIMIT
    assert draws_chunk(1, m, B, limit)[0] == Bc
    hd = limited_handle(limit) if Bc < B else h
    try:
        d, mu, info = hd.posterior_draws_batched(t, y, TH, order=0, s=s, jitter=0.0, seed=seed)
    finally:
        if hd is not h:
            hd.close()
    assert np.all(info == 0) and np.all(mu == 0.0)
    ref = philox.normals(seed, B * m + 1)[:B * m].reshape(B, m)
    assert np.max(np.abs(d - ref)) < 1e-13
    assert one_chunk(1, m, B) and one_chunk(1, m, B, z=True)
    d1, _, _ = h.posterior_draws_batched(t, y, TH, order=0, s=s, jitter=0.0, seed=seed)
    assert np.array_equal(bits(d), bits(d1))
    dz, _, _ = h.posterior_draws_batched(t, y, TH, order=0, s=s, jitter=0.0, z=h.normal_fill(seed, B * m).reshape(B, m))
    assert np.array_equal(bits(d), bits(dz))
