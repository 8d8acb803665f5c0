"""gpb200_latent_forward_batched / gpb200_latent_backward_batched: the non-centred latent model (f = L z and the reverse
sweep through the Cholesky) for B parameter states in one call.

References: oracle.chol_deriv_ext.latent_adjoint, one call per item, with the bars of test_cholesky_derivatives_gpu.py
(f and zbar within 1e-10 of max |ref|, theta_bar within 1e-9 of the reference's scale = sum |Kbar o dK/dtheta|).  Every
test asserts its own premises: the inputs are dense across tiles (far-tile share and far-tile sum), the items differ
(swapping two items' outputs breaks the bar), and where a schedule or a chunking is the point, the host code picks it
(predicates mirrored from the C code)."""
import functools

import numpy as np
import pytest

from gp_b200 import capi, latent_gp
from oracle import chol_deriv_ext as X
from oracle import gp_oracle as o

pytestmark = pytest.mark.gpu

RTOL = 1e-9
NSM = 148
ALPHA, DIAG_ADD = 1.3, 0.1


# ---- branch predicates, mirrored from the C host code --------------------------------------------------------
def tiles(n):
    return (n + 127) // 128


def gemm_cfg(ntasks, batch, override=0):
    """gemm_pick_cfg (gemm.cu) with the default knobs: 3 = quarter tiles, 2 = half tiles."""
    if override:
        return override
    return 3 if ntasks * batch * 2 < 2 * NSM * 2 else 2


def lookahead(nt, batch):
    """chol_uses_lookahead (engine.cu)."""
    return batch <= 64 and batch * nt <= 256 and nt >= 3


def chol_schedule(n, batch):
    """chol_batched (engine.cu) with the default knobs."""
    nt = tiles(n)
    if lookahead(nt, batch):
        return "lookahead"
    return "left-looking" if (batch >= 64 or nt <= 8) else "panels"


def trtri_level_tasks(nt):
    """tasks per launch of trtri_batched (tasks_trtri / build_nodes, engine.cu)."""
    nodes = []

    def build(lo, hi):
        if hi - lo <= 1:
            return 0
        mid = lo + (hi - lo + 1) // 2
        lvl = max(build(lo, mid), build(mid, hi)) + 1
        nodes.append((lo, mid, hi, lvl))
        return lvl
    top = build(0, nt)
    return [sum((hi - mid) * (mid - lo) for lo, mid, hi, l in nodes if l == lvl) for lvl in range(1, top + 1)]


def fine(ntasks, batch):
    """launch_gemm (gemm.cu): a launch on the dependent chain with few CTAs takes the 16-warp fine tiles."""
    return gemm_cfg(ntasks, batch) == 3 and ntasks * batch * 4 <= NSM


def trsm_tiles_per_cta(ntiles, batch):
    """launch_trsm_tiles_at (panel.cu) with the default knobs."""
    total = ntiles * batch
    if total * 2 <= NSM:
        return 0
    return 4 if total >= NSM * 16 else (2 if total >= NSM * 6 else 1)


def panel_fused(ntiles, batch):
    """launch_potrf_trsm_at (panel.cu): POTRF + TRSM in one launch for small launches."""
    return batch <= NSM and batch * (1 + ntiles) <= NSM


def backward_same_schedule(nt, b1, b2):
    """Every launch of the backward sweep (the tile inverse, the TK_LATENT_G GEMM) makes the same choice for b1 and b2
    items; the other kernels work per item."""
    ks = trtri_level_tasks(nt) + [nt * nt]
    return lookahead(nt, b1) == lookahead(nt, b2) and all(
        gemm_cfg(k, b1) == gemm_cfg(k, b2) and fine(k, b1) == fine(k, b2) for k in ks)


def same_schedule(nt, b1, b2):
    """The forward factorisation and the backward sweep make the same choices for b1 and b2 items (conservative: every
    task count up to nt^2)."""
    la = lambda b: lookahead(nt, b)
    return (la(b1) == la(b2) and (b1 >= 64 or nt <= 8) == (b2 >= 64 or nt <= 8)
            and all(gemm_cfg(k, b1) == gemm_cfg(k, b2) and fine(k, b1) == fine(k, b2) for k in range(1, nt * nt + 1))
            and all(trsm_tiles_per_cta(k, b1) == trsm_tiles_per_cta(k, b2) and panel_fused(k, b1) == panel_fused(k, b2)
                    for k in range(1, nt)))


def _pad256(b):
    return (b + 255) & ~255


def backward_chunk(n, B, nvec, limit):
    """Items per backward chunk under a workspace limit (gpb200_latent_backward_batched, host-pointer mode)."""
    np_ = tiles(n) * 128
    nparts = tiles(n) ** 2 * 4
    per_item = (2 * _pad256(np_ * np_ * 8) + 2 * _pad256(nvec * np_ * 8) + _pad256(nparts * 4 * 8)
                + _pad256(nvec * n * 8) + 64)
    fixed = _pad256(np_ * 8) + _pad256(B * 2 * 8) + 4096
    return min(B, (limit - fixed - 8192) // per_item), fixed, per_item


# ---- inputs and references ----------------------------------------------------------------------------------------
def rho_lat(n):
    """2.5 on [0, 10], 1.5 on [0, 20]: the far tiles of Kbar o dK/dtheta stay above 1e-2 of its largest entry."""
    return 2.5 if n <= 1100 else 1.5


def dense_x(n, seed):
    return np.sort(np.random.default_rng(seed).uniform(0.0, 10.0 if n <= 1100 else 20.0, n))


def item_inputs(n, b, nvec, per_item_x):
    """x, (alpha, rho), z (nvec x n), fbar (nvec x n) of item b: every item has its own theta, z and fbar, and with
    per_item_x its own x."""
    x = dense_x(n, 7000 + n + 131 * b if per_item_x else 6000 + n)
    th = (ALPHA * (1.0 + 0.1 * (b % 4)), rho_lat(n) * (1.0 + 0.05 * (b % 3)))
    rng = np.random.default_rng(9000 + 10 * n + 1000 * b + nvec)
    return x, th, rng.standard_normal((nvec, n)), rng.standard_normal((nvec, n))


def batch_inputs(n, B, nvec, per_item_x):
    items = [item_inputs(n, b, nvec, per_item_x) for b in range(B)]
    x = np.stack([it[0] for it in items]) if per_item_x else items[0][0]
    return (x, np.array([it[1] for it in items]), np.stack([it[2] for it in items]), np.stack([it[3] for it in items]))


@functools.lru_cache(maxsize=None)
def item_ref(n, b, nvec, per_item_x):
    x, (a, r), z, fbar = item_inputs(n, b, nvec, per_item_x)
    return X.latent_adjoint(x, a, r, DIAG_ADD, z, fbar)


def within(got, ref, rtol):
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    return bool(np.max(np.abs(got - ref)) <= rtol * float(np.max(np.abs(ref))))


def theta_within(got, ref, scale, rtol=RTOL):
    return all(abs(got[k] - ref[k]) <= rtol * scale[k] for k in range(2))


def check_premises(n, r, what):
    if tiles(n) < 2:
        return   # one tile: nothing is far from the diagonal
    share = X.far_tile_share(r["L"])
    assert share >= 1e-2, "%s: premise broken, far-tile share of L %.2e < 1e-2" % (what, share)
    for k in range(2):
        share = X.far_tile_share(r["terms"][k])
        assert share >= 1e-2, "%s: premise broken, far-tile share of the adjoint terms %.2e" % (what, share)


def assert_far_sum(n, refs, what):
    """Deleting the far tile pairs from the adjoint would move theta_bar of at least one checked item by far more than
    the bar (the far terms are signed: for a single item they may happen to cancel)."""
    if tiles(n) < 2:
        return
    assert any(all(abs(X.far_tile_sum(r["terms"][k])) >= 1e3 * RTOL * r["scale"][k] for k in range(2)) for r in refs), what


def check_item(n, b, nvec, per_item_x, f, tb, zbar, what):
    r = item_ref(n, b, nvec, per_item_x)
    check_premises(n, r, what)
    assert within(f, r["f"], 1e-10), "%s: f, max err %.3e" % (what, np.max(np.abs(f - r["f"])))
    assert within(zbar, r["zbar"], 1e-10), "%s: zbar, max err %.3e" % (what, np.max(np.abs(zbar - r["zbar"])))
    assert theta_within(tb, r["theta_bar"], r["scale"]), "%s: theta_bar %r, reference %r, scale %r" % (
        what, tb, r["theta_bar"], r["scale"])


def bits(a):
    return np.asarray(a, dtype=np.float64).view(np.uint64).copy()


def same_bits(*pairs):
    for k, (a, b) in enumerate(pairs):
        if not np.array_equal(bits(a), bits(b)):
            d = np.abs(np.asarray(a, dtype=np.float64) - np.asarray(b, dtype=np.float64))
            print("output %d differs: max |diff| %.3e, NaN %d / %d" % (k, np.nanmax(d) if np.isfinite(d).any() else np.nan,
                                                                    int(np.isnan(a).sum()), int(np.isnan(b).sum())))
            return False
    return True


def run(h, n, B, nvec, per_item_x):
    x, th, z, fbar = batch_inputs(n, B, nvec, per_item_x)
    f, info = h.latent_forward_batched(x, th, DIAG_ADD, z)
    tb, zbar = h.latent_backward_batched(fbar)
    return (x, th, z, fbar), (f, info, tb, zbar)


def single_calls(h, x, th, z, fbar, b):
    xb = x[b] if x.ndim == 2 else x
    fs = h.latent_forward(xb, th[b, 0], th[b, 1], DIAG_ADD, z[b])
    tbs, zbs = h.latent_backward(xb, th[b, 0], th[b, 1], DIAG_ADD, z[b], fbar[b])
    return fs, tbs, zbs


# ---- 1, 2. parity per item against the reference and against the single-item calls ----------------------------------
@pytest.mark.parametrize("per_item_x", [False, True], ids=["shared-x", "per-item-x"])
@pytest.mark.parametrize("nvec", [1, 2])
@pytest.mark.parametrize("B", [1, 5, 64])
@pytest.mark.parametrize("n", [100, 300, 1000, 2200])
def test_items_match_reference_and_single_item_calls(handle, n, B, nvec, per_item_x):
    (x, th, z, fbar), (f, info, tb, zbar) = run(handle, n, B, nvec, per_item_x)
    assert f.shape == (B, nvec, n) and zbar.shape == (B, nvec, n) and tb.shape == (B, 2)
    assert np.all(info == 0), info
    # the reference for every item up to n = 1000, for the first, second, middle and last at n = 2200
    checked = list(range(B)) if n <= 1000 else sorted({0, 1, B // 2, B - 1} & set(range(B)))
    for b in checked:
        check_item(n, b, nvec, per_item_x, f[b], tb[b], zbar[b], "n=%d B=%d nvec=%d item %d" % (n, B, nvec, b))
    assert_far_sum(n, [item_ref(n, b, nvec, per_item_x) for b in checked], "far-tile sum premise")
    # premise: the items differ, so a wrong batch index or stride cannot pass
    for i, j in zip(checked, checked[1:]):
        r = item_ref(n, i, nvec, per_item_x)
        assert not within(f[j], r["f"], 1e-10) and not within(zbar[j], r["zbar"], 1e-10), (i, j)
        assert not theta_within(tb[j], r["theta_bar"], r["scale"]), (i, j)
    for b in range(B):
        fs, tbs, zbs = single_calls(handle, x, th, z, fbar, b)
        if B == 1:
            assert same_bits((f[b], fs), (zbar[b], zbs), (tb[b], tbs)), "B = 1 must be bit-identical to the single call"
        else:
            # other batch sizes take other GEMM configurations and Cholesky schedules: the sums are reordered.  theta_bar
            # is a sum of terms that cancel, so its rounding is relative to their size, the reference's scale
            what = "n=%d B=%d item %d vs its single-item call" % (n, B, b)
            assert within(f[b], fs, 1e-12) and within(zbar[b], zbs, 1e-12), what
            if b in checked:
                r = item_ref(n, b, nvec, per_item_x)
                assert theta_within(tb[b], tbs, r["scale"], 1e-12), (what, tb[b] - tbs, r["scale"])


# ---- 3. schedules ----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [0, 1, 2, 3])
def test_every_gemm_configuration(handle, cfg):
    n, B, nvec = 1000, 5, 2
    assert gemm_cfg(tiles(n) ** 2, B, cfg) == (cfg or 2)
    try:
        handle.set_gemm_config(cfg)
        (x, th, z, fbar), (f, info, tb, zbar) = run(handle, n, B, nvec, True)
        assert np.all(info == 0)
        for b in range(B):
            check_item(n, b, nvec, True, f[b], tb[b], zbar[b], "cfg %d item %d" % (cfg, b))
            fs, tbs, zbs = single_calls(handle, x, th, z, fbar, b)
            assert within(f[b], fs, 1e-12) and within(zbar[b], zbs, 1e-12), (cfg, b)
            assert theta_within(tb[b], tbs, item_ref(n, b, nvec, True)["scale"], 1e-12), (cfg, b, tb[b] - tbs)
        assert_far_sum(n, [item_ref(n, b, nvec, True) for b in range(B)], "far-tile sum premise")
    finally:
        handle.set_gemm_config(0)


@pytest.mark.parametrize("B,schedule", [(5, "lookahead"), (16, "panels"), (64, "left-looking")])
def test_every_cholesky_schedule(handle, B, schedule):
    n, nvec = 2200, 1
    assert chol_schedule(n, B) == schedule
    _, (f, info, tb, zbar) = run(handle, n, B, nvec, True)
    assert np.all(info == 0)
    items = sorted({0, B // 2, B - 1})
    for b in items:
        check_item(n, b, nvec, True, f[b], tb[b], zbar[b], "%s B=%d item %d" % (schedule, B, b))
    assert_far_sum(n, [item_ref(n, b, nvec, True) for b in items], "far-tile sum premise")


def test_chunked_backward_is_bit_identical():
    n, B, nvec, chunk = 1000, 160, 1, 80
    nt = tiles(n)
    assert backward_same_schedule(nt, chunk, B)
    _, fixed, per_item = backward_chunk(n, B, nvec, 1 << 62)
    limit = fixed + 8192 + chunk * per_item + per_item // 2
    assert backward_chunk(n, B, nvec, limit)[0] == chunk
    x, th, z, fbar = batch_inputs(n, B, nvec, True)
    h = capi.Handle(0)
    try:
        h.latent_forward_batched(x, th, DIAG_ADD, z)
        c0 = h.launch_count()
        ref = h.latent_backward_batched(fbar)
        whole = h.launch_count() - c0
        h.set_workspace_limit(limit)
        c0 = h.launch_count()
        got = h.latent_backward_batched(fbar)
        assert h.launch_count() - c0 > whole, "premise: the limit must split the backward into chunks"
        assert same_bits((ref[0], got[0]), (ref[1], got[1]))
        f, _ = h.latent_forward_batched(x, th, DIAG_ADD, z)
        check_item(n, B - 1, nvec, True, f[B - 1], got[0][B - 1], got[1][B - 1], "chunked, last item")
    finally:
        h.close()


# ---- 4. the record -----------------------------------------------------------------------------------------------
def test_record_holds_copies_and_survives_repeats_and_single_item_calls():
    import torch
    n, B, nvec = 300, 5, 2
    x, th, z, fbar = batch_inputs(n, B, nvec, True)
    h = capi.Handle(0)
    try:
        f0, _ = h.latent_forward_batched(x, th, DIAG_ADD, z)
        ref = h.latent_backward_batched(fbar)
        assert same_bits((ref[0], h.latent_backward_batched(fbar)[0]), (ref[1], h.latent_backward_batched(fbar)[1])), \
            "a second backward call must repeat the first"
        # the caller overwrites its host buffers between forward and backward
        xh, thh, zh = x.copy(), th.copy(), z.copy()
        h.latent_forward_batched(xh, thh, DIAG_ADD, zh)
        xh[:] = 0.0; thh[:] = 7.0; zh[:] = 3.0
        assert same_bits(*zip(ref, h.latent_backward_batched(fbar)))
        # single-item calls in between touch nothing of the record
        h.latent_forward_batched(x, th, DIAG_ADD, z)
        single_calls(h, x[::-1].copy(), th[::-1].copy(), z, fbar, 2)
        h.latent_forward(x[0], 0.7, 1.1, 0.2, z[0, 0])
        assert same_bits(*zip(ref, h.latent_backward_batched(fbar)))
        # the same in device-pointer mode: the caller's tensors are overwritten after the forward call
        dev = torch.device("cuda", 0)
        h.set_pointer_mode(True)
        xd = torch.tensor(x, device=dev); thd = torch.tensor(th, device=dev); zd = torch.tensor(z, device=dev)
        fd = torch.empty((B, nvec, n), dtype=torch.float64, device=dev); infod = torch.empty(B, dtype=torch.int32, device=dev)
        h.latent_forward_batched_device(n, B, nvec, xd, n, thd, DIAG_ADD, zd, fd, infod)
        xd.fill_(0.0); thd.fill_(-1.0); zd.fill_(5.0)
        fbd = torch.tensor(fbar, device=dev)
        tbd = torch.empty((B, 2), dtype=torch.float64, device=dev); zbd = torch.empty_like(fbd)
        h.latent_backward_batched_device(n, B, nvec, fbd, tbd, zbd)
        torch.cuda.synchronize()
        assert same_bits((fd.cpu().numpy(), f0), (tbd.cpu().numpy(), ref[0]), (zbd.cpu().numpy(), ref[1]))
    finally:
        h.close()


def test_second_forward_replaces_the_record():
    a = batch_inputs(300, 5, 2, True)
    b = batch_inputs(1000, 3, 1, False)
    h, fresh = capi.Handle(0), capi.Handle(0)
    try:
        h.latent_forward_batched(a[0], a[1], DIAG_ADD, a[2])
        h.latent_forward_batched(b[0], b[1], DIAG_ADD, b[2])
        got = h.latent_backward_batched(b[3])
        fresh.latent_forward_batched(b[0], b[1], DIAG_ADD, b[2])
        assert same_bits(*zip(got, fresh.latent_backward_batched(b[3])))
    finally:
        h.close()
        fresh.close()


def raw_backward(h, n, B, nvec):
    fb = np.ones((B, nvec, n)); tb = np.full((B, 2), -3.0); zb = np.full((B, nvec, n), -3.0)
    c0 = h.launch_count()
    rc = h.lib.gpb200_latent_backward_batched(h._h, n, B, nvec, fb.ctypes.data, tb.ctypes.data, zb.ctypes.data)
    untouched = h.launch_count() == c0 and np.all(tb == -3.0) and np.all(zb == -3.0)
    return rc, untouched


def test_backward_without_a_matching_record_is_refused():
    n, B, nvec = 300, 5, 2
    x, th, z, fbar = batch_inputs(n, B, nvec, True)
    h = capi.Handle(0)
    try:
        rc, untouched = raw_backward(h, n, B, nvec)
        assert rc < 0 and untouched, "fresh handle"
        h.latent_forward_batched(x, th, DIAG_ADD, z)
        for args in ((n + 1, B, nvec), (n, B - 1, nvec), (n, B, nvec + 1)):
            rc, untouched = raw_backward(h, *args)
            assert rc < 0 and untouched, args
        assert raw_backward(h, n, B, nvec)[0] == 0, "the record survives a refused call"
        # a failed forward call (bad x_stride) leaves no record
        f = np.empty((B, nvec, n)); info = np.zeros(B, dtype=np.int32)
        zc = np.ascontiguousarray(z); thc = np.ascontiguousarray(th); xc = np.ascontiguousarray(x)
        rc = h.lib.gpb200_latent_forward_batched(h._h, n, B, nvec, xc.ctypes.data, n - 1, thc.ctypes.data, DIAG_ADD,
                                                 zc.ctypes.data, f.ctypes.data, info.ctypes.data)
        assert rc < 0
        rc, untouched = raw_backward(h, n, B, nvec)
        assert rc < 0 and untouched, "after a failed forward call"
        with pytest.raises(capi.GpB200Error):
            h.latent_backward_batched(fbar)
    finally:
        h.close()


# ---- 5. failed items -------------------------------------------------------------------------------------------
def pivot(x, alpha, rho, diag_add):
    """1-based index of the first pivot of cov_exp_quad(x, alpha, rho) + diag_add I that is not > 0 (NaN included), 0
    when it factors: a column-by-column Cholesky (dpotrf's NaN handling differs between LAPACK builds)."""
    K = o.add_diag(alpha * alpha * np.exp(-0.5 * (x[:, None] - x[None, :]) ** 2 / (rho * rho)), diag_add)
    n = K.shape[0]
    L = np.zeros_like(K)
    for j in range(n):
        d = K[j, j] - L[j, :j] @ L[j, :j]
        if not d > 0:
            return j + 1
        L[j, j] = np.sqrt(d)
        L[j + 1:, j] = (K[j + 1:, j] - L[j + 1:, :j] @ L[j, :j]) / L[j, j]
    return 0


def test_failed_items_report_the_pivot_and_leave_the_others_alone():
    """Two items fail: one with a NaN amplitude (every entry of K is NaN: pivot 1), one whose first two points coincide
    with no diagonal term (alpha = 1, diag_add = 0: the second pivot is exactly 0).  (A NaN inside x does not make the
    SE covariance fail: the Gram kernel, here as in the single-item call, maps the point to one uncorrelated with the
    others.)  The other points are 3 apart at length-scales near 1, so their covariances factor without a diagonal
    term."""
    n, B, nvec = 300, 4, 2
    bad_alpha, bad_dup = 1, 2
    keep = [0, 3]
    assert same_schedule(tiles(n), B, len(keep))
    rng = np.random.default_rng(11)
    x = 3.0 * np.arange(n) + 0.2 * rng.uniform(size=(B, n))
    th = np.stack([1.0 + 0.2 * rng.uniform(size=B), 0.9 + 0.3 * rng.uniform(size=B)], axis=1)
    z = rng.standard_normal((B, nvec, n)); fbar = rng.standard_normal((B, nvec, n))
    th[bad_alpha, 0] = np.nan
    th[bad_dup, 0] = 1.0
    x[bad_dup, 1] = x[bad_dup, 0]
    h = capi.Handle(0)
    try:
        f, info = h.latent_forward_batched(x, th, 0.0, z)
        tb, zbar = h.latent_backward_batched(fbar)
        for b in (bad_alpha, bad_dup):
            assert info[b] == pivot(x[b], th[b, 0], th[b, 1], 0.0) > 0, (b, info[b])
            assert np.all(np.isnan(f[b])) and np.all(np.isnan(zbar[b])) and np.all(np.isnan(tb[b])), b
        assert info[bad_alpha] == 1 and info[bad_dup] == 2
        assert np.all(info[keep] == 0) and np.all(np.isfinite(tb[keep]))
        f2, info2 = h.latent_forward_batched(x[keep], th[keep], 0.0, z[keep])
        tb2, zbar2 = h.latent_backward_batched(fbar[keep])
        assert np.all(info2 == 0)
        assert same_bits((f[keep], f2), (tb[keep], tb2), (zbar[keep], zbar2))
    finally:
        h.close()


# ---- 6. device-pointer mode ------------------------------------------------------------------------------------
def test_device_mode_is_bit_identical_and_respects_strides_and_guards():
    import torch
    n, B, nvec = 300, 3, 2
    x, th, z, fbar = batch_inputs(n, B, nvec, True)
    h = capi.Handle(0)
    try:
        ref_f, ref_info = h.latent_forward_batched(x, th, DIAG_ADD, z)
        ref_tb, ref_zbar = h.latent_backward_batched(fbar)
        dev = torch.device("cuda", 0)
        xs, g = n + 37, 64
        xbuf = torch.full((B * xs + g,), float("nan"), dtype=torch.float64, device=dev)
        for b in range(B):
            xbuf[b * xs:b * xs + n] = torch.tensor(x[b])
        thd = torch.tensor(th, device=dev); zd = torch.tensor(z, device=dev); fbd = torch.tensor(fbar, device=dev)
        inputs = [t.clone() for t in (xbuf, thd, zd, fbd)]
        fb = torch.full((B * nvec * n + 2 * g,), 12345.0, dtype=torch.float64, device=dev)
        tbb = torch.full((2 * B + 2 * g,), 12345.0, dtype=torch.float64, device=dev)
        zbb = torch.full((B * nvec * n + 2 * g,), 12345.0, dtype=torch.float64, device=dev)
        ib = torch.full((B + 2 * g,), -7, dtype=torch.int32, device=dev)
        stream = torch.cuda.Stream(device=dev)
        h.set_pointer_mode(True)
        h.set_stream(stream.cuda_stream)
        with torch.cuda.stream(stream):
            h.latent_forward_batched_device(n, B, nvec, xbuf, xs, thd, DIAG_ADD, zd, fb[g:g + B * nvec * n], ib[g:g + B])
            h.latent_backward_batched_device(n, B, nvec, fbd, tbb[g:g + 2 * B], zbb[g:g + B * nvec * n])
        stream.synchronize()
        for buf, fill in ((fb, 12345.0), (tbb, 12345.0), (zbb, 12345.0), (ib, -7)):
            assert torch.all(buf[:g] == fill) and torch.all(buf[-g:] == fill), "write outside the window"
        for a, b in zip(inputs, (xbuf, thd, zd, fbd)):
            assert torch.equal(torch.nan_to_num(a, nan=-1.0), torch.nan_to_num(b, nan=-1.0)), "an input was written"
        got = [fb[g:-g].cpu().numpy().reshape(B, nvec, n), tbb[g:-g].cpu().numpy().reshape(B, 2),
               zbb[g:-g].cpu().numpy().reshape(B, nvec, n)]
        assert same_bits((got[0], ref_f), (got[1], ref_tb), (got[2], ref_zbar))
        assert np.array_equal(ib[g:-g].cpu().numpy(), ref_info)
    finally:
        h.close()


def test_device_loop_runs_without_a_host_round_trip():
    """forward -> fbar = (y - f) / sigma^2 in torch -> backward on the caller's stream.  Behind a long device sleep the
    stream is still busy when the loop has been enqueued: none of the calls waited for the device."""
    import torch
    n, B, nvec, sigma = 1000, 8, 1, 0.3
    x, th, z, _ = batch_inputs(n, B, nvec, False)
    dev = torch.device("cuda", 0)
    y = torch.tensor(np.sin(x), device=dev)
    xd = torch.tensor(x, device=dev); thd = torch.tensor(th, device=dev); zd = torch.tensor(z, device=dev)
    f = torch.empty((B, nvec, n), dtype=torch.float64, device=dev); info = torch.empty(B, dtype=torch.int32, device=dev)
    tb = torch.empty((B, 2), dtype=torch.float64, device=dev); zbar = torch.empty_like(f)
    h = capi.Handle(0)
    try:
        stream = torch.cuda.Stream(device=dev)
        h.set_pointer_mode(True)
        h.set_stream(stream.cuda_stream)

        def loop():
            h.latent_forward_batched_device(n, B, nvec, xd, 0, thd, DIAG_ADD, zd, f, info)
            fbar = (y - f) / sigma ** 2
            h.latent_backward_batched_device(n, B, nvec, fbar, tb, zbar)
            return fbar
        with torch.cuda.stream(stream):
            loop()   # warm-up: grows the record and the workspace, builds the task lists
        stream.synchronize()
        with torch.cuda.stream(stream):
            torch.cuda._sleep(2_000_000_000)
            fbar = loop()
            busy = not stream.query()
        stream.synchronize()
        assert busy, "a call synchronised with the device"
    finally:
        h.close()
    # the same states in host mode, backward from torch's fbar
    h = capi.Handle(0)
    try:
        ref_f, _ = h.latent_forward_batched(x, th, DIAG_ADD, z)
        ref_tb, ref_zbar = h.latent_backward_batched(fbar.cpu().numpy())
        assert same_bits((f.cpu().numpy(), ref_f), (tb.cpu().numpy(), ref_tb), (zbar.cpu().numpy(), ref_zbar))
    finally:
        h.close()


# ---- 7. the Python mirror --------------------------------------------------------------------------------------
def test_exact_gp_log_prob_batched_rows_match_the_single_state_function(handle):
    rng = np.random.default_rng(17)
    n, B = 200, 4
    x = np.arange(n) * 0.8 + 0.05 * rng.standard_normal(n)
    y = np.sin(x) + 0.1 * rng.standard_normal(n)
    z = rng.standard_normal((B, n))
    l = np.array([0.9, 1.1, 0.7, 1.4]); sigma = np.array([0.3, 0.25, 0.4, 0.35]); alpha = np.array([1.0, 1.3, 0.8, 1.1])
    lp, g = latent_gp.exact_gp_log_prob_batched(x, y, l, sigma, z, alpha=alpha, jitter=1e-6, handle=handle)
    for b in range(B):
        lps, gs = latent_gp.exact_gp_log_prob(x, y, l[b], sigma[b], z[b], alpha=alpha[b], jitter=1e-6, handle=handle)
        assert abs(lp[b] - lps) <= 1e-12 * abs(lps), b
        for k in ("l", "sigma", "alpha"):
            assert abs(g[k][b] - gs[k]) <= 1e-12 * abs(gs[k]), (b, k, g[k][b], gs[k])
        assert within(g["z"][b], gs["z"], 1e-12) and within(g["f"][b], gs["f"], 1e-12), b
    # one state against central differences of the oracle's lp (exact_gp.stan: alpha = 1, jitter 1e-10)
    lp1, g1 = latent_gp.exact_gp_log_prob_batched(x, y, l, sigma, z, handle=handle)
    rlp, rg = o.exact_gp_lp_grad(x, y, l[1], sigma[1], z[1])
    assert abs(lp1[1] - rlp) <= 1e-9 * abs(rlp)
    hh = 1e-6
    fd = (o.exact_gp_lp_grad(x, y, l[1] + hh, sigma[1], z[1])[0] - o.exact_gp_lp_grad(x, y, l[1] - hh, sigma[1], z[1])[0]) / (2 * hh)
    assert abs(g1["l"][1] - fd) <= 1e-6 * max(1.0, abs(fd)), (g1["l"][1], fd)
    assert abs(g1["l"][1] - rg["l"]) <= 1e-8 * abs(rg["l"])


# ---- 8. bad arguments ------------------------------------------------------------------------------------------
def test_bad_arguments_launch_nothing(handle):
    n, B, nvec = 300, 2, 1
    x = np.zeros(n); th = np.ones((B, 2)); z = np.zeros((B, n)); f = np.empty((B, n)); info = np.zeros(B, dtype=np.int32)
    p = lambda a: a.ctypes.data
    fwd = dict(n=n, B=B, nvec=nvec, x=p(x), xs=0, th=p(th), z=p(z), f=p(f), info=p(info))
    cases = [dict(n=0), dict(B=0), dict(nvec=0), dict(xs=n - 1), dict(x=None), dict(th=None), dict(z=None), dict(f=None),
             dict(info=None)]
    lib = handle.lib
    for c in cases:
        a = dict(fwd, **c)
        c0 = handle.launch_count()
        rc = lib.gpb200_latent_forward_batched(handle._h, a["n"], a["B"], a["nvec"], a["x"], a["xs"], a["th"], DIAG_ADD,
                                               a["z"], a["f"], a["info"])
        assert rc < 0 and handle.launch_count() == c0, c
    tb = np.empty((B, 2)); zb = np.empty((B, n))
    for c in [dict(n=0), dict(B=0), dict(nvec=0), dict(fb=None), dict(tb=None), dict(zb=None)]:
        a = dict(dict(n=n, B=B, nvec=nvec, fb=p(z), tb=p(tb), zb=p(zb)), **c)
        c0 = handle.launch_count()
        rc = lib.gpb200_latent_backward_batched(handle._h, a["n"], a["B"], a["nvec"], a["fb"], a["tb"], a["zb"])
        assert rc < 0 and handle.launch_count() == c0, c
