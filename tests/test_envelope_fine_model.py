"""NumPy model of the element profile of the SE covariance and of the contraction bounds it gives each GEMM CTA of the
envelope route (left-looking / panel Cholesky and selected inverse of lml_grad_batched).  No GPU: the model is the
reference of the executed-flop counts that tests/test_envelope_fine_gpu.py reads from the device counter.

Profile, per item (gram.cu, solve.cu):
  f_k   first column of row k of the lower triangle whose exp(-d^2 / 2 rho^2) is not exactly zero (NaN counts, the
        diagonal always counts; padding rows keep only their diagonal)
  fb[q] min f_k over the 64-row block q
  er[J] the last row k with f_k <= J * 128 + 127 (the last row of L with a nonzero in tile column J)
  F_I = min(fb[2I], fb[2I+1]) // 128 and E_J = the last tile row I with F_I <= J, exactly as the tile envelope had them

CTA bounds (gemm_tile_body.cuh):
  Cholesky update C(I,J) -= L(I,:) L(J,:)^T, tile rule (look-ahead schedule): skip J < F_I, k from max(F_I, F_J) 128;
  element rule (every other schedule): k from round_down_16(max(min fb over the CTA's rows, min fb over its columns)).
  Selected inverse Z[S,J] = -Z[S,S] Y[S,J] and Z[J,J] = D - Y[S,J]^T Z[S,J]: skip I > E_J, k up to round_up_16(er[J] + 1)
  (Y = L W_JJ: row k of Y is nonzero across the whole tile column J once L has a nonzero anywhere in it).
"""
import numpy as np

TILE = 128
BLK = 64            # the smallest CTA extent (quarter and fine tiles): the granularity of fb
KC = 16             # k-chunk of the GEMM main loop: the granularity of the bounds
EXP_CUT = -708.0    # exp_nonpos (fastexp.cuh) returns exactly 0 for t < -708 and a normal number otherwise
SMS = 148


# ---- profile ---------------------------------------------------------------------------------------------------------
def row_profile(x, rho, nt):
    """f_k for the padded matrix of nt tile rows; t = d * d * nh with nh = -0.5 / (rho * rho), as gram_se_batched."""
    x = np.asarray(x, dtype=np.float64)
    n, npad = x.shape[0], nt * TILE
    nh = -0.5 / (rho * rho)
    f = np.arange(npad)
    for r0 in range(0, n, 512):
        d = x[r0:r0 + 512, None] - x[None, :]
        nz = ~(d * d * nh < EXP_CUT)                 # NaN counts as nonzero
        first = np.argmax(nz, axis=1)                # the diagonal is nonzero: first <= row
        f[r0:r0 + first.shape[0]] = np.minimum(first, np.arange(r0, r0 + first.shape[0]))
    return f


class Profile:
    def __init__(self, x, rho, nt):
        self.nt = nt
        self.f = f = row_profile(x, rho, nt)
        self.fb = f.reshape(-1, BLK).min(axis=1)
        self.F = np.minimum(self.fb.reshape(nt, 2).min(axis=1) // TILE, np.arange(nt))
        self.E = np.array([max(i for i in range(j, nt) if self.F[i] <= j) for j in range(nt)])
        # er[J] = max{k : f_k <= 128 J + 127}: prefix maximum over J of the last row whose f_k falls in tile column J
        last = np.full(nt, -1)
        np.maximum.at(last, f // TILE, np.arange(f.shape[0]))
        self.er = np.maximum.accumulate(last)


# ---- task lists (engine.cu) ------------------------------------------------------------------------------------------
# a task: (ti, tj, k0, k_len, diag, b_tri_first)  -- output tile, contraction start and length, flags that matter here
def chol_panel_tiles(nt, batch):
    return nt if batch >= 64 or nt <= 8 else 8


def chol_launches(nt, pt):
    """Launches of chol_batched outside the look-ahead schedule, in order: per block column the in-panel update, after
    each panel its trailing update."""
    out = []
    for j in range(nt):
        p0 = (j // pt) * pt
        if j > p0:
            out.append([(i, j, p0 * TILE, (j - p0) * TILE, i == j, False) for i in range(j, nt)])
        if (j + 1) % pt == 0 and j + 1 < nt:
            p1 = min(nt, j + 1)
            out.append([(i, jj, p0 * TILE, (p1 - p0) * TILE, i == jj, False) for jj in range(p1, nt) for i in range(jj, nt)])
    return out


def sinv_launches(nt):
    """ENV_BAND launches of sinv_batched: Y, then per block column from nt - 2 down Z[S,J] (NN) and Z[J,J] (TN)."""
    y = [(i, j, j * TILE, TILE, False, True) for j in range(nt) for i in range(j + 1, nt)]
    out = [y] if nt > 1 else []
    for j in range(nt - 2, -1, -1):
        k0, kl = (j + 1) * TILE, (nt - 1 - j) * TILE
        out.append([(i, j, k0, kl, False, False) for i in range(j + 1, nt)])
        out.append([(j, j, k0, kl, False, False)])
    return out


def d_launch_flops(nt):
    """The D = W_JJ^T W_JJ launch (no envelope), half-tile CTAs: the column half n0 = 64 skips the zero half of W_JJ."""
    return nt * 2.0 * TILE * 64 * (TILE + TILE // 2)


# ---- CTAs of a launch (gemm.cu) --------------------------------------------------------------------------------------
def launch_ctas(tasks, batch, cfg=None):
    """(task, TM, TN, m0, n0) per CTA, by the configuration launch_gemm picks: cfg None is the automatic choice
    (quarter tiles below two waves of half-tile CTAs), and the diagonal split sends TF_DIAG tasks to quarter CTAs."""
    c = cfg if cfg else (3 if len(tasks) * batch * 2 < 2 * SMS * 2 else 2)
    diag = [t for t in tasks if t[4]]
    split = c == 2 and batch >= 16 and len(tasks) * batch >= 2048 and diag and len(diag) < len(tasks)
    for t in tasks:
        cc = 3 if (split and t[4]) else c
        tm, tn = (64, 64) if cc == 3 else ((128, 64) if cc == 2 else (128, 128))
        for m0 in range(0, TILE, tm):
            for n0 in range(0, TILE, tn):
                yield t, tm, tn, m0, n0


def cta_k(t, tm, tn, m0, n0):
    """Contraction range of a CTA before the envelope: the triangular-operand and symmetric-quadrant skips."""
    ti, tj, k0, kl, diag, b_tri_first = t
    if tm < TILE and diag and m0 < n0:
        return k0, k0
    if tn < TILE and b_tri_first and n0 >= TILE // 2:
        k0, kl = k0 + TILE // 2, kl - TILE // 2
    return k0, k0 + kl


def chol_cta_flops(P, t, tm, tn, m0, n0, fine):
    ti, tj = t[0], t[1]
    k0, k1 = cta_k(t, tm, tn, m0, n0)
    if fine:
        ka = P.fb[(ti * TILE + m0) // BLK:(ti * TILE + m0 + tm) // BLK].min()
        kb = P.fb[(tj * TILE + n0) // BLK:(tj * TILE + n0 + tn) // BLK].min()
        k0 = max(k0, max(ka, kb) // KC * KC)
    else:
        if tj < P.F[ti]:
            return 0.0
        k0 = max(k0, max(P.F[ti], P.F[tj]) * TILE)
    return 2.0 * tm * tn * max(k1 - k0, 0)


def band_cta_flops(P, t, tm, tn, m0, n0, fine):
    ti, tj = t[0], t[1]
    k0, k1 = cta_k(t, tm, tn, m0, n0)
    if ti > P.E[tj]:
        return 0.0
    k1 = min(k1, -(-(P.er[tj] + 1) // KC) * KC if fine else (P.E[tj] + 1) * TILE)
    return 2.0 * tm * tn * max(k1 - k0, 0)


def chol_flops(profiles, fine=True, cfg=None, pt=None):
    """Executed Cholesky-update flops of one chol_batched call (not the look-ahead schedule) over the items."""
    B, nt = len(profiles), profiles[0].nt
    total = 0.0
    for tasks in chol_launches(nt, pt or chol_panel_tiles(nt, B)):
        for cta in launch_ctas(tasks, B, cfg):
            total += sum(chol_cta_flops(P, *cta, fine) for P in profiles)
    return total


def sinv_flops(profiles, fine=True, cfg=None, with_y=True):
    """Executed flops of the envelope launches of sinv_batched (Y, Z[S,J], Z[J,J])."""
    B, nt = len(profiles), profiles[0].nt
    total = 0.0
    for q, tasks in enumerate(sinv_launches(nt)):
        if q == 0 and not with_y:
            continue
        for cta in launch_ctas(tasks, B, cfg):
            total += sum(band_cta_flops(P, *cta, fine) for P in profiles)
    return total


# ---- tests -----------------------------------------------------------------------------------------------------------
def bench_inputs():
    """bench.py synth_inputs(0): N = 4096, 256 draws."""
    rng = np.random.default_rng(5)
    x = np.sort(rng.uniform(0.0, 0.05 * 4096, size=4096))
    r2 = np.random.default_rng(1000)
    th = np.stack([np.abs(r2.standard_normal(256)) + 0.1, r2.gamma(4.0, 0.25, 256), r2.uniform(0.1, 0.5, 256)], axis=1)
    return x, th


def dense_tile_profile(x, rho, nt):
    """F and E straight from the dense element test, tile by tile (the definition of the tile envelope)."""
    n = x.shape[0]
    t = -0.5 / (rho * rho)
    d = x[:, None] - x[None, :]
    nz = np.eye(nt * TILE, dtype=bool)
    nz[:n, :n] |= ~(d * d * t < EXP_CUT)
    F = np.array([min(i, min(j for j in range(nt) if nz[i * TILE:(i + 1) * TILE, j * TILE:(j + 1) * TILE].any()))
                  for i in range(nt)])
    E = np.array([max(i for i in range(j, nt) if F[i] <= j) for j in range(nt)])
    return F, E


def test_profile_matches_dense_definition():
    """fb gives the tile F and E of the tile envelope exactly, er[J] // 128 = E_J, on sorted, shuffled and NaN inputs."""
    rng = np.random.default_rng(3)
    x = np.sort(rng.uniform(0.0, 90.0, 1900))
    xs = x[rng.permutation(x.shape[0])]
    xn = x.copy()
    xn[1234] = np.nan
    for xx in (x, xs, xn):
        for rho in (0.3, 1.1, 7.0):
            P = Profile(xx, rho, 15)
            F, E = dense_tile_profile(xx, rho, 15)
            assert np.array_equal(P.F, F) and np.array_equal(P.E, E)
            assert np.array_equal(P.er // TILE, P.E)
            assert np.all(P.er >= np.arange(15) * TILE + TILE - 1)
    # NaN row: every later row reaches column 1234, so their profile starts at or before it
    P = Profile(xn, 0.3, 15)
    assert np.all(P.f[1234:1900] <= 1234)


def test_element_bounds_drop_only_zero_products():
    """The element-rule k-range of every CTA lies inside the tile-rule range and starts where a row of either operand
    is nonzero (Cholesky) / ends past the last nonzero row of Y (selected inverse)."""
    rng = np.random.default_rng(4)
    x = rng.uniform(0.0, 60.0, 1500)
    profiles = [Profile(x, rho, 12) for rho in (0.2, 0.9, 3.0)]
    for P in profiles:
        for tasks in chol_launches(12, 12):
            for t, tm, tn, m0, n0 in launch_ctas(tasks, 3, 2):
                assert chol_cta_flops(P, t, tm, tn, m0, n0, True) <= chol_cta_flops(P, t, tm, tn, m0, n0, False)
                rows = np.r_[t[0] * TILE + m0:t[0] * TILE + m0 + tm, t[1] * TILE + n0:t[1] * TILE + n0 + tn]
                k0, k1 = cta_k(t, tm, tn, m0, n0)
                first = max(P.f[rows[:tm]].min(), P.f[rows[tm:]].min())
                kept = max(k1 - max(k0, first), 0)
                assert chol_cta_flops(P, t, tm, tn, m0, n0, True) >= 2.0 * tm * tn * kept
        for tasks in sinv_launches(12):
            for cta in launch_ctas(tasks, 3, 2):
                assert band_cta_flops(P, *cta, True) <= band_cta_flops(P, *cta, False)
                ti, tj = cta[0][0], cta[0][1]
                if ti <= P.E[tj]:
                    k0, k1 = cta_k(*cta)
                    kept = max(min(k1, np.nonzero(P.f <= tj * TILE + TILE - 1)[0].max() + 1) - k0, 0)
                    assert band_cta_flops(P, *cta, True) >= 2.0 * cta[1] * cta[2] * kept


def test_bench_inputs_flop_table():
    """Per step on the bench inputs, in the configurations launch_gemm picks at B = 256 (half-tile CTAs, the diagonal
    Cholesky tiles on quarter CTAs): Cholesky updates 7.28e11 under the tile rule, 6.51e11 (-10.6 %) under the element
    rule; Z[S,J] and Z[J,J] 1.531e12 and 1.444e12 (-5.6 %)."""
    x, th = bench_inputs()
    profiles = [Profile(x, th[b, 1], 32) for b in range(th.shape[0])]
    got = (chol_flops(profiles, False), chol_flops(profiles, True), sinv_flops(profiles, False, with_y=False),
           sinv_flops(profiles, True, with_y=False))
    assert np.allclose(got, (7.2807e11, 6.5061e11, 1.5306e12, 1.4445e12), rtol=1e-4), got
