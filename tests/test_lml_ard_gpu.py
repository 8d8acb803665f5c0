"""gpb200_lml_grad_ard_batched on the GPU: the batched LML + gradient of the ARD squared-exponential covariance
(QQard) against the float64 reference of tests/support/ard_oracle.py, against the one-dimensional SE route, across
schedules and GEMM configurations, in device-pointer mode, and on failing items and bad arguments."""
import os
import sys

import numpy as np
import pytest

from gp_b200 import capi
sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "support"))
import ard_oracle  # noqa: E402

NSM = 148
PW = 10  # doubles per trace partial record of the ARD epilogue (epi_partial_width)


# ---- branch predicates, mirrored from the C host code --------------------------------------------------------
def tiles(n):
    return (n + 127) // 128


def lauum_tasks(nt):
    """tasks_lauum (engine.cu): one task per lower tile."""
    return nt * (nt + 1) // 2


def gemm_cfg(ntasks, batch):
    """gemm_pick_cfg (gemm.cu) with the default knobs: 3 = quarter tiles, 2 = half tiles."""
    return 3 if ntasks * batch * 2 < 2 * NSM * 2 else 2


def diag_split(ntasks, batch):
    """diag_split_applies (gemm.cu)."""
    return gemm_cfg(ntasks, batch) == 2 and batch >= 16 and ntasks * batch >= 2048


def uses_graph(n, B, chunk=None):
    """lml_core replays the evaluation as one CUDA graph (api_gp.cu); the ARD kind never takes the one-CTA kernel."""
    nt = tiles(n)
    return (chunk is None or chunk == B) and nt <= 64 and B * nt * nt <= 4096


def _pad256(b):
    return (b + 255) & ~255


def ard_chunk(n, D, B, limit, x_per_item=False, y_per_item=False):
    """Items per chunk under a workspace limit: the arithmetic of lml_core (api_gp.cu) for the ARD kind."""
    np_ = tiles(n) * 128
    nt = np_ // 128
    nparts = lauum_tasks(nt) * 4
    ctas = nt * B
    zks = 1 if (ctas >= 2 * NSM or nt < 4) else min(nt, (2 * NSM + ctas - 1) // ctas)
    per_item = (_pad256(np_ * np_ * 8) * 2 + 3 * _pad256(np_ * 8) + _pad256(nparts * PW * 8)
                + (_pad256(zks * np_ * 8) if zks > 1 else 0) + 64)
    xl = n * D
    fixed = (_pad256(B * (xl if x_per_item else 0) * 8 + xl * 8) + _pad256(B * (n if y_per_item else 0) * 8 + n * 8)
             + 2 * _pad256(B * (D + 2) * 8) + _pad256(B * 8) + _pad256(B * 4) + 4096)
    return min(B, (limit - fixed - 8192) // per_item), fixed, per_item


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a.view(np.uint32)


def _item(X, y, b):
    return (X[b] if X.ndim == 3 else X), (y[b] if y.ndim == 2 else y)


def check_items(lml, grad, info, X, y, th, items, jitter=0.0, rtol=1e-9):
    D = th.shape[1] - 2
    for b in items:
        Xb, yb = _item(X, y, b)
        rv, rg = ard_oracle.lml_grad_ard(Xb, yb, th[b, 0], th[b, 1:D + 1], th[b, D + 1], jitter)
        assert info[b] == 0, (b, info[b])
        assert abs(lml[b] - rv) <= rtol * max(abs(rv), 1.0), (b, lml[b], rv)
        scale = np.max(np.abs(rg))
        for k in range(D + 2):  # per gradient component, relative to the item's gradient scale
            assert abs(grad[b, k] - rg[k]) <= rtol * max(abs(rg[k]), scale, 1e-300), (b, k, grad[b, k], rg[k])


@pytest.fixture(scope="module")
def h():
    hd = capi.Handle(0)
    yield hd
    hd.close()


def handle_with(**env):
    """A handle created under the given GPB200_* environment knobs (read by gpb200_create)."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update({k: str(v) for k, v in env.items()})
    try:
        return capi.Handle(0)
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


# ---- 1. parity with the reference ------------------------------------------------------------------------------
SMALL = [(D, n, per) for D in (1, 2, 3, 5, 8) for n, per in ((1, False), (7, True), (100, False), (129, True), (515, False))]


@pytest.mark.gpu
@pytest.mark.parametrize("D,n,per_item", SMALL)
def test_parity_small_and_tile_edges(h, D, n, per_item):
    X, y, th = ard_oracle.synth_ard(n, D, 4, seed=100 * D + n, per_item=per_item)
    lml, grad, info = h.lml_grad_ard_batched(X, y, th)
    check_items(lml, grad, info, X, y, th, range(4))


@pytest.mark.gpu
@pytest.mark.parametrize("D,n,B,per_item", [(5, 1000, 64, True), (2, 1000, 64, False), (3, 2100, 1, False),
                                             (1, 2100, 4, True)])
def test_parity_large(h, D, n, B, per_item):
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=7 * D + B, per_item=per_item)
    lml, grad, info = h.lml_grad_ard_batched(X, y, th)
    check_items(lml, grad, info, X, y, th, sorted({0, B // 3, B // 2, B - 1}))


@pytest.mark.gpu
def test_parity_diag_split_batch(h):
    n, D, B = 2100, 8, 300
    assert diag_split(lauum_tasks(tiles(n)), B)  # premise: the LAUUM launch takes the diagonal split
    X, _, th = ard_oracle.synth_ard(n, D, B, seed=21)
    _, y, _ = ard_oracle.synth_ard(n, D, B, seed=22, per_item=True)  # shared X, per-item y (B, n)
    lml, grad, info = h.lml_grad_ard_batched(X, y, th)
    assert np.all(info == 0)
    check_items(lml, grad, info, X, y, th, [0, 1, 149, 298, 299])


# ---- 2. D = 1 is the SE model ------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("envelope", [0, 1])
@pytest.mark.parametrize("n,B", [(300, 8), (2100, 8)])
def test_one_dimension_matches_the_se_route(envelope, n, B):
    hd = handle_with(GPB200_ENVELOPE=envelope)
    try:
        from oracle import gp_oracle as o
        x, y = o.synth_xy(n, 3)
        th = o.synth_theta(B, 4)
        l0, g0, i0 = hd.lml_grad_batched(x, y, th, jitter=1e-8)
        l1, g1, i1 = hd.lml_grad_ard_batched(x[:, None], y, th, jitter=1e-8)
        assert np.all(i0 == 0) and np.all(i1 == 0)
        for b in range(B):
            assert abs(l1[b] - l0[b]) <= 1e-12 * abs(l0[b])
            scale = np.max(np.abs(g0[b]))
            for k in range(3):
                assert abs(g1[b, k] - g0[b, k]) <= 1e-12 * max(abs(g0[b, k]), scale), (b, k, g1[b, k], g0[b, k])
    finally:
        hd.close()


# ---- 3. permutation and constant columns -------------------------------------------------------------------------
@pytest.mark.gpu
def test_permuting_columns_permutes_the_gradient(h):
    n, D, B = 515, 5, 6
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=31, per_item=True)
    perm = np.array([3, 0, 4, 1, 2])
    l0, g0, _ = h.lml_grad_ard_batched(X, y, th)
    thp = th.copy()
    thp[:, 1:D + 1] = th[:, 1:D + 1][:, perm]
    l1, g1, _ = h.lml_grad_ard_batched(X[:, :, perm], y, thp)
    np.testing.assert_allclose(l1, l0, rtol=1e-13)
    gp = g0.copy()
    gp[:, 1:D + 1] = g0[:, 1:D + 1][:, perm]
    for b in range(B):
        np.testing.assert_allclose(g1[b], gp[b], rtol=1e-13, atol=1e-13 * np.max(np.abs(gp[b])))


@pytest.mark.gpu
def test_constant_column_has_zero_gradient_and_drops_out(h):
    n, D, B = 700, 3, 5
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=41)
    X[:, 1] = 0.37
    l3, g3, _ = h.lml_grad_ard_batched(X, y, th)
    assert np.all(g3[:, 2] == 0.0)
    l2, g2, _ = h.lml_grad_ard_batched(X[:, [0, 2]], y, th[:, [0, 1, 3, 4]])
    np.testing.assert_allclose(l3, l2, rtol=1e-12)
    for b in range(B):
        np.testing.assert_allclose(g3[b, [0, 1, 3, 4]], g2[b], rtol=1e-12, atol=1e-12 * np.max(np.abs(g2[b])))


# ---- 4. schedules, configurations, graphs, chunks ------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("knob", ["cfg1", "cfg2", "cfg3", "GPB200_DIAG_SPLIT", "GPB200_LOOKAHEAD", "GPB200_NO_GRAPH"])
def test_every_schedule_agrees_with_the_reference(knob):
    hd = handle_with(**({knob: 1 if knob == "GPB200_NO_GRAPH" else 0} if knob.startswith("GPB200") else {}))
    try:
        if knob.startswith("cfg"):
            hd.set_gemm_config(int(knob[3]))
        for n, D, B in ((515, 3, 4), (1300, 8, 24)):
            X, y, th = ard_oracle.synth_ard(n, D, B, seed=n + D, per_item=True)
            lml, grad, info = hd.lml_grad_ard_batched(X, y, th)
            check_items(lml, grad, info, X, y, th, [0, B // 2, B - 1])
    finally:
        hd.close()


def trsm_tiles_per_cta(ntiles, batch):
    """launch_trsm_tiles_at (panel.cu) with the default knobs: 0 = a latency form (row-split kernel), else the
    tiles per CTA of the batched kernels."""
    total = ntiles * batch
    if total * 2 <= NSM:
        return 0
    return 4 if total >= NSM * 16 else (2 if total >= NSM * 6 else 1)


def panel_fused(ntiles, batch):
    """launch_potrf_trsm_at (panel.cu): POTRF + TRSM in one launch for small launches."""
    return batch <= NSM and batch * (1 + ntiles) <= NSM


def same_schedule(nt, b1, b2):
    """Every launch of the dense route picks the same kernel and configuration for batches b1 and b2 (the predicates
    above; POTRF and the tile inverse do not depend on the batch)."""
    la = lambda b: b <= 64 and b * nt <= 256 and nt >= 3
    return (la(b1) == la(b2) and (b1 >= 64 or nt <= 8) == (b2 >= 64 or nt <= 8)
            and all(gemm_cfg(k, b1) == gemm_cfg(k, b2) and diag_split(k, b1) == diag_split(k, b2)
                    for k in range(1, lauum_tasks(nt) + 1))
            and all(trsm_tiles_per_cta(k, b1) == trsm_tiles_per_cta(k, b2) and panel_fused(k, b1) == panel_fused(k, b2)
                    for k in range(1, nt)))


def chunk_limit(n, D, B, chunk):
    _, fixed, per_item = ard_chunk(n, D, B, 1 << 62, x_per_item=True, y_per_item=True)
    limit = fixed + 8192 + chunk * per_item + per_item // 2
    assert ard_chunk(n, D, B, limit, True, True)[0] == chunk
    return limit


@pytest.mark.gpu
def test_graph_replay_is_bit_identical_to_the_eager_call(h):
    n, D, B = 515, 4, 128
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=51, per_item=True)
    assert uses_graph(n, B)
    eager = handle_with(GPB200_NO_GRAPH=1)
    try:
        ref = eager.lml_grad_ard_batched(X, y, th)
    finally:
        eager.close()
    r0 = h.graph_replays()
    got = h.lml_grad_ard_batched(X, y, th)
    got2 = h.lml_grad_ard_batched(X, y, th)
    assert h.graph_replays() >= r0 + 2
    for a, b in zip(ref, got):
        assert np.array_equal(_bits(a), _bits(b))
    for a, b in zip(ref, got2):
        assert np.array_equal(_bits(a), _bits(b))


@pytest.mark.gpu
def test_chunking_is_bit_identical_when_the_chunks_take_the_same_schedule(h):
    # chunks of 2400 items against the 4800-item call: every launch (GEMM configuration, diagonal split, TRSM form,
    # fused panel, look-ahead) makes the same choice, so the chunks must reproduce the unchunked bits
    n, D, B, chunk = 200, 4, 4800, 2400
    nt = tiles(n)
    assert same_schedule(nt, chunk, B) and not uses_graph(n, B)
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=52, per_item=True)
    ref = h.lml_grad_ard_batched(X, y, th)
    hc = capi.Handle(0)
    try:
        hc.set_workspace_limit(chunk_limit(n, D, B, chunk))
        chunked = hc.lml_grad_ard_batched(X, y, th)
    finally:
        hc.close()
    assert np.all(ref[2] == 0)
    for a, b in zip(ref, chunked):
        assert np.array_equal(_bits(a), _bits(b))
    check_items(*chunked, X, y, th, [0, chunk - 1, chunk, B - 1])


@pytest.mark.gpu
def test_chunks_with_another_schedule_agree_to_rounding(h):
    # 64-item chunks of a 128-item call: the small chunks take the fused POTRF + TRSM launch and other TRSM forms
    n, D, B, chunk = 515, 4, 128, 64
    assert not same_schedule(tiles(n), chunk, B)
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=51, per_item=True)
    ref = h.lml_grad_ard_batched(X, y, th)
    hc = capi.Handle(0)
    try:
        hc.set_workspace_limit(chunk_limit(n, D, B, chunk))
        chunked = hc.lml_grad_ard_batched(X, y, th)
    finally:
        hc.close()
    assert np.array_equal(ref[2], chunked[2]) and np.all(ref[2] == 0)
    np.testing.assert_allclose(chunked[0], ref[0], rtol=1e-12, atol=0)
    for b in range(B):
        scale = np.max(np.abs(ref[1][b]))
        assert np.max(np.abs(chunked[1][b] - ref[1][b])) <= 1e-10 * scale, b
    check_items(*chunked, X, y, th, [0, chunk - 1, chunk, B - 1])


# ---- 5. LML only -------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("n,B", [(300, 4), (1000, 40)])
def test_lml_only_matches_the_gradient_call(h, n, B):
    X, y, th = ard_oracle.synth_ard(n, 3, B, seed=61)
    l1, _, _ = h.lml_grad_ard_batched(X, y, th)
    l0, _, i0 = h.lml_grad_ard_batched(X, y, th, want_grad=False)
    assert np.all(i0 == 0)
    np.testing.assert_allclose(l0, l1, rtol=1e-12)


# ---- 6. failing items ------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("want_grad", [True, False])
def test_failed_items_report_the_pivot_and_leave_neighbours_alone(h, want_grad):
    n, D, B = 300, 3, 6
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=71, per_item=True)
    bad_sing, bad_nan = 1, 4
    X[bad_sing, 1] = X[bad_sing, 0]            # duplicate rows, no noise, no jitter: exactly singular
    th[bad_sing, 0] = 1.0
    th[bad_sing, D + 1] = 0.0
    X[bad_nan, 5, 2] = np.nan
    lml, grad, info = h.lml_grad_ard_batched(X, y, th, want_grad=want_grad)
    for b in (bad_sing, bad_nan):
        assert info[b] == ard_oracle.pivot(X[b], th[b, 0], th[b, 1:D + 1], th[b, D + 1]) > 0, (b, info[b])
    keep = [b for b in range(B) if b not in (bad_sing, bad_nan)]
    l2, g2, i2 = h.lml_grad_ard_batched(X[keep], y[keep], th[keep], want_grad=want_grad)
    assert np.all(info[keep] == 0) and np.all(i2 == 0)
    assert np.array_equal(_bits(lml[keep]), _bits(l2))
    if want_grad:
        assert np.array_equal(_bits(grad[keep]), _bits(g2))


# ---- 7. device-pointer mode --------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_device_mode_is_bit_identical_and_respects_strides_and_guards(h):
    import torch
    n, D, B = 515, 3, 5
    X, y, th = ard_oracle.synth_ard(n, D, B, seed=81, per_item=True)
    ref = h.lml_grad_ard_batched(X, y, th)
    xs, ys, guard = n * D + 37, n + 11, 64
    Xh = np.full(B * xs + guard, np.nan)
    yh = np.full(B * ys + guard, np.nan)
    for b in range(B):
        Xh[b * xs:b * xs + n * D] = X[b].T.reshape(-1)  # column-major n x D
        yh[b * ys:b * ys + n] = y[b]
    dev = torch.device("cuda", 0)
    dX = torch.from_numpy(Xh).to(dev)
    dy = torch.from_numpy(yh).to(dev)
    dth = torch.from_numpy(th).to(dev)
    sentinel = -7.25
    dl = torch.full((B + guard,), sentinel, dtype=torch.float64, device=dev)
    dg = torch.full((B * (D + 2) + guard,), sentinel, dtype=torch.float64, device=dev)
    di = torch.full((B + guard,), -3, dtype=torch.int32, device=dev)
    stream = torch.cuda.Stream(device=dev)
    with torch.cuda.stream(stream):
        h.set_stream(stream.cuda_stream)
        h.set_pointer_mode(True)
        try:
            h.lml_grad_ard_batched_device(n, D, B, dX, xs, dy, ys, dth, 0.0, True, dl, dg, di)
        finally:
            h.set_pointer_mode(False)
        stream.synchronize()  # only the caller's stream
        lml, grad, info = dl.cpu().numpy(), dg.cpu().numpy(), di.cpu().numpy()
    h.set_stream(torch.cuda.current_stream().cuda_stream)
    assert np.array_equal(_bits(lml[:B]), _bits(ref[0]))
    assert np.array_equal(_bits(grad[:B * (D + 2)].reshape(B, D + 2)), _bits(ref[1]))
    assert np.array_equal(info[:B], ref[2])
    assert np.all(lml[B:] == sentinel) and np.all(grad[B * (D + 2):] == sentinel) and np.all(info[B:] == -3)
    assert np.array_equal(_bits(dX.cpu().numpy()), _bits(Xh)) and np.array_equal(_bits(dy.cpu().numpy()), _bits(yh))


# ---- 8. bad arguments ----------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_bad_arguments_return_negative_and_launch_nothing(h):
    lib = h.lib
    n, D, B = 50, 2, 3
    X = np.zeros(n * D * B); y = np.zeros(n * B); th = np.ones((B, D + 2))
    lml = np.empty(B); grad = np.empty((B, D + 2)); info = np.zeros(B, dtype=np.int32)
    p = capi._ptr

    def call(n_=n, D_=D, B_=B, xs=0, ys=0):
        return lib.gpb200_lml_grad_ard_batched(h._h, n_, D_, B_, p(X), xs, p(y), ys, p(th), 0.0, 1, p(lml), p(grad), p(info))

    before = h.launch_count()
    for kw in ({"n_": 0}, {"n_": -3}, {"B_": -1}, {"D_": 0}, {"D_": 9}, {"xs": n * D - 1}, {"ys": n - 1}):
        rc = call(**kw)
        assert rc < 0, kw
        assert lib.gpb200_last_error(h._h), kw
    assert h.launch_count() == before
    assert call(B_=0) == 0 and h.launch_count() == before


# ---- 9. the GPU gradient is the derivative of the GPU LML ------------------------------------------------------------
@pytest.mark.gpu
def test_gradient_matches_central_differences_of_the_gpu_lml(h):
    n, D = 2048, 3
    X, y, th = ard_oracle.synth_ard(n, D, 1, seed=91)
    _, g, _ = h.lml_grad_ard_batched(X, y, th)
    rows = []
    steps = []
    for k in range(D + 2):
        hk = 1e-5 * th[0, k]
        for s in (1.0, -1.0):
            t = th[0].copy()
            t[k] += s * hk
            rows.append(t)
        steps.append(hk)
    lp, _, info = h.lml_grad_ard_batched(X, y, np.array(rows), want_grad=False)
    assert np.all(info == 0)
    for k in range(D + 2):
        fd = (lp[2 * k] - lp[2 * k + 1]) / (2 * steps[k])
        assert abs(fd - g[0, k]) <= 1e-5 * max(abs(g[0, k]), 1.0), (k, fd, g[0, k])
