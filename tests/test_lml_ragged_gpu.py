"""gpb200_lml_grad_ragged: B GPs of different sizes in one call (per-group GPs, multiple_players.stan:59-63).

Every item is checked against the oracle or against the uniform entry point at its own size; the sizes cross the
one-CTA path (n <= 128), the tile boundaries, the dense route, the envelope route (nt >= 16) and the selected inverse
(B_k * nt >= 256)."""
import os

import numpy as np
import pytest

from gp_b200 import capi
from oracle import gp_oracle as o

pytestmark = pytest.mark.gpu

CROSS = [1, 2, 7, 127, 128, 129, 255, 256, 257, 1000, 2177]   # + the Westbrook series (1438)


def relerr(a, b):
    return float(np.max(np.abs(np.asarray(a) - np.asarray(b))) / max(np.max(np.abs(np.asarray(b))), 1e-300))


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def groups(sizes, seed):
    xs, ys = [], []
    for g, n in enumerate(sizes):
        x, y = o.synth_xy(n, seed + g)
        xs.append(x); ys.append(y)
    return xs, ys, o.synth_theta(len(sizes), seed)


def westbrook_xy(westbrook):
    x, y = westbrook["x"], westbrook["y"] - westbrook["y"].mean()
    order = np.argsort(x, kind="stable")
    return x[order], y[order]


@pytest.fixture(scope="module")
def crossing(westbrook):
    xs, ys, th = groups(CROSS, 11)
    wx, wy = westbrook_xy(westbrook)
    xs.insert(10, wx); ys.insert(10, wy)
    th = np.insert(th, 10, [0.5, 0.2, 0.45], axis=0)
    return xs, ys, th


def test_oracle_parity_across_every_boundary(handle, crossing):
    xs, ys, th = crossing
    jitter = 1e-6   # the Westbrook series repeats inputs (test_westbrook_real_inputs)
    lml, grad, info = handle.lml_grad_ragged(xs, ys, th, jitter)
    assert np.all(info == 0)
    for b in range(len(xs)):
        rv, rg = o.lml_grad_lapack(xs[b], ys[b], *th[b], jitter=jitter)
        assert abs(lml[b] - rv) <= 1e-9 * abs(rv), (b, len(xs[b]), lml[b], rv)
        for k in range(3):
            assert abs(grad[b, k] - rg[k]) <= 1e-9 * abs(rg[k]), (b, k, grad[b], rg)


def test_selected_inverse_bucket_against_oracle(handle):
    # 16 items of nt = 17 (B_k * nt = 272 >= 256): the envelope route with the selected inverse, beside a small bucket
    sizes = [2049 + 7 * g for g in range(16)] + [60, 300]
    xs, ys, th = groups(sizes, 5)
    lml, grad, info = handle.lml_grad_ragged(xs, ys, th)
    assert np.all(info == 0)
    for b in (0, 7, 15, 16, 17):
        rv, rg = o.lml_grad_lapack(xs[b], ys[b], *th[b])
        assert abs(lml[b] - rv) <= 1e-9 * abs(rv), b
        assert relerr(grad[b], rg) < 1e-9, (b, grad[b], rg)
    # and the uniform call of each size
    for b in range(16):
        l1, g1, _ = handle.lml_grad_batched(xs[b], ys[b], th[b:b + 1])
        assert abs(lml[b] - l1[0]) <= 1e-12 * abs(l1[0]) and relerr(grad[b], g1[0]) < 1e-11, b


def test_equivalent_to_uniform_call_per_item(handle, crossing):
    xs, ys, th = crossing
    lml, grad, info = handle.lml_grad_ragged(xs, ys, th, 1e-6)
    for b in range(len(xs)):
        l1, g1, i1 = handle.lml_grad_batched(xs[b], ys[b], th[b:b + 1], 1e-6)
        assert info[b] == i1[0] == 0
        assert abs(lml[b] - l1[0]) <= 1e-12 * abs(l1[0]), (b, lml[b], l1[0])
        assert relerr(grad[b], g1[0]) < 1e-11, (b, grad[b], g1[0])


@pytest.mark.parametrize("n,B", [(100, 9), (1024, 32), (2100, 4)])
def test_equal_sizes_match_the_uniform_call(handle, n, B):
    xs, ys, th = groups([n] * B, 3)
    lml, grad, info = handle.lml_grad_ragged(xs, ys, th)
    l1, g1, i1 = handle.lml_grad_batched(np.stack(xs), np.stack(ys), th)
    assert np.array_equal(info, i1)
    assert np.all(np.abs(lml - l1) <= 1e-13 * np.abs(l1))
    assert relerr(grad, g1) < 1e-13


def test_permuting_items_permutes_outputs_bit_for_bit(handle):
    sizes = [300, 90, 1500, 300, 129, 2177, 64, 1000]
    xs, ys, th = groups(sizes, 21)
    ref = handle.lml_grad_ragged(xs, ys, th)
    perm = np.random.default_rng(4).permutation(len(sizes))
    got = handle.lml_grad_ragged([xs[p] for p in perm], [ys[p] for p in perm], th[perm])
    for r, g in zip(ref, got):
        assert np.array_equal(bits(r[perm]), bits(g))


def test_lml_only_matches_the_gradient_call(handle, crossing):
    # without the gradient z = L^-1 y comes from a substitution instead of the explicit inverse (as in
    # gpb200_lml_grad_batched), so the two agree to rounding, and each agrees with the uniform LML-only call
    xs, ys, th = crossing
    l1, _, i1 = handle.lml_grad_ragged(xs, ys, th, 1e-6)
    l0, _, i0 = handle.lml_grad_ragged(xs, ys, th, 1e-6, want_grad=False)
    assert np.array_equal(i0, i1) and np.all(i0 == 0)
    assert np.all(np.abs(l0 - l1) <= 1e-12 * np.abs(l1))
    for b in range(len(xs)):
        u0, _, _ = handle.lml_grad_batched(xs[b], ys[b], th[b:b + 1], 1e-6, want_grad=False)
        assert abs(l0[b] - u0[0]) <= 1e-12 * abs(u0[0]), b


def test_non_positive_definite_item_is_isolated(handle):
    sizes = [50, 400, 300, 2177, 90]
    xs, ys, th = groups(sizes, 8)
    ok = handle.lml_grad_ragged(xs, ys, th)
    assert np.all(ok[2] == 0)
    bad = 2
    xs[bad] = xs[bad].copy(); xs[bad][41] = xs[bad][40]   # two equal inputs, no noise, no jitter: singular
    th = th.copy(); th[bad, 2] = 0.0
    lml, grad, info = handle.lml_grad_ragged(xs, ys, th)
    _, _, i1 = handle.lml_grad_batched(xs[bad], ys[bad], th[bad:bad + 1])
    assert i1[0] > 0 and info[bad] == i1[0]
    for b in range(len(sizes)):
        if b == bad:
            continue
        assert info[b] == 0 and np.isfinite(lml[b]) and np.all(np.isfinite(grad[b]))
        assert np.array_equal(bits(lml[b:b + 1]), bits(ok[0][b:b + 1])) and np.array_equal(bits(grad[b]), bits(ok[1][b]))


def test_device_pointer_mode_is_bit_identical_and_writes_only_its_outputs(crossing):
    import torch
    xs, ys, th = crossing
    B = len(xs)
    h = capi.Handle(0)
    try:
        host = h.lml_grad_ragged(xs, ys, th, 1e-6)
        offsets = np.zeros(B + 1, dtype=np.int64)
        offsets[1:] = np.cumsum([len(v) for v in xs])
        dev = torch.device("cuda", 0)
        x = torch.from_numpy(np.concatenate(xs)).to(dev)
        y = torch.from_numpy(np.concatenate(ys)).to(dev)
        t = torch.from_numpy(np.ascontiguousarray(th)).to(dev)
        x0, y0, t0 = x.clone(), y.clone(), t.clone()
        G = 16   # guard bands around every output
        lml = torch.full((B + 2 * G,), 7.25, dtype=torch.float64, device=dev)
        grad = torch.full((3 * B + 2 * G,), -3.5, dtype=torch.float64, device=dev)
        info = torch.full((B + 2 * G,), 12345, dtype=torch.int32, device=dev)
        stream = torch.cuda.Stream(dev)
        stream.wait_stream(torch.cuda.current_stream(dev))   # the inputs and guard fills come first
        h.set_pointer_mode(True)
        h.set_stream(stream.cuda_stream)
        h.lml_grad_ragged_device(B, offsets, x, y, t, 1e-6, True, lml[G:], grad[G:], info[G:])
        stream.synchronize()
        h.set_pointer_mode(False)
        L, Gr, I = lml.cpu().numpy(), grad.cpu().numpy(), info.cpu().numpy()
        assert np.all(L[:G] == 7.25) and np.all(L[G + B:] == 7.25)
        assert np.all(Gr[:G] == -3.5) and np.all(Gr[G + 3 * B:] == -3.5)
        assert np.all(I[:G] == 12345) and np.all(I[G + B:] == 12345)
        assert np.array_equal(bits(L[G:G + B]), bits(host[0]))
        assert np.array_equal(bits(Gr[G:G + 3 * B].reshape(B, 3)), bits(host[1]))
        assert np.array_equal(I[G:G + B], host[2])
        assert torch.equal(x, x0) and torch.equal(y, y0) and torch.equal(t, t0)
    finally:
        h.close()


def test_workspace_chunking_and_dense_route(handle, crossing):
    # six items of nt = 8 beside two smaller buckets; the limit holds about two of them at a time
    sizes = [1000, 900, 1024, 897, 1000, 950, 300, 50]
    cx, cy, cth = groups(sizes, 31)
    ref = handle.lml_grad_ragged(cx, cy, cth)
    h = capi.Handle(0)
    try:
        h.set_workspace_limit(int(2.5 * 2 * 1024 * 1024 * 8) + (1 << 20))
        chunked = h.lml_grad_ragged(cx, cy, cth)
        launches = h.launch_count()
        h.set_workspace_limit(0)
        h.lml_grad_ragged(cx, cy, cth)
        assert launches > h.launch_count() - launches   # the chunked call really took more launches
    finally:
        h.close()
    # chunks may take other GEMM and Cholesky schedules than the whole bucket: equal to rounding
    assert np.array_equal(chunked[2], ref[2]) and np.all(ref[2] == 0)
    assert np.all(np.abs(chunked[0] - ref[0]) <= 1e-12 * np.abs(ref[0])) and relerr(chunked[1], ref[1]) < 1e-11
    xs, ys, th = crossing
    ref = handle.lml_grad_ragged(xs, ys, th, 1e-6)
    old = os.environ.get("GPB200_ENVELOPE")
    os.environ["GPB200_ENVELOPE"] = "0"
    try:
        hd = capi.Handle(0)
    finally:
        if old is None:
            del os.environ["GPB200_ENVELOPE"]
        else:
            os.environ["GPB200_ENVELOPE"] = old
    try:
        dense = hd.lml_grad_ragged(xs, ys, th, 1e-6)
    finally:
        hd.close()
    assert np.array_equal(dense[2], ref[2])
    assert np.all(np.abs(dense[0] - ref[0]) <= 1e-12 * np.abs(ref[0])) and relerr(dense[1], ref[1]) < 1e-11


def test_more_groups_than_a_grid_dimension_holds(handle):
    # 70 000 tiny groups (B above 65535) in one call: every launch indexes the groups in gridDim.x or in chunks
    rng = np.random.default_rng(17)
    sizes = rng.integers(1, 24, size=70000)
    xs, ys = [], []
    for g, n in enumerate(sizes):
        x = np.sort(rng.uniform(0.0, 0.05 * n + 1.0, size=n))
        xs.append(x); ys.append(np.sin(x) + 0.3 * rng.standard_normal(n))
    th = o.synth_theta(len(sizes), 18)
    lml, grad, info = handle.lml_grad_ragged(xs, ys, th)
    assert np.all(info == 0) and np.all(np.isfinite(lml)) and np.all(np.isfinite(grad))
    for b in (0, 1, 65534, 65535, 65536, 69999) + tuple(rng.integers(0, 70000, 6)):
        rv, rg = o.lml_grad_lapack(xs[b], ys[b], *th[b])
        assert abs(lml[b] - rv) <= 1e-9 * abs(rv), b
        assert np.all(np.abs(grad[b] - rg) <= 1e-9 * np.abs(rg)), (b, grad[b], rg)


def test_bad_arguments_return_negative_codes_and_write_nothing(handle):
    lib = handle.lib
    x = np.linspace(0.0, 5.0, 20); y = np.sin(x); th = np.tile([1.0, 0.5, 0.3], (3, 1))
    cases = [
        (-1, [0, 5, 10, 20], "B must be >= 0"),
        (3, [1, 5, 10, 20], "offsets[0]"),
        (3, [0, 10, 5, 20], "non-decreasing"),
        (3, [0, 5, 5, 20], "n_b >= 1"),
        (1, [0, 70000], "65407"),
    ]
    for B, off, word in cases:
        off = np.asarray(off, dtype=np.int64)
        xx = np.zeros(max(int(off[-1]), 20)); xx[:20] = x
        yy = np.zeros_like(xx); yy[:20] = y
        lml = np.full(3, 9.0); grad = np.full(9, 9.0); info = np.full(3, 9, dtype=np.int32)
        rc = lib.gpb200_lml_grad_ragged(handle._h, B, off.ctypes.data, xx.ctypes.data, yy.ctypes.data, th.ctypes.data,
                                        0.0, 1, lml.ctypes.data, grad.ctypes.data, info.ctypes.data)
        assert rc < 0, (B, off)
        msg = lib.gpb200_last_error(handle._h).decode()
        assert "lml_grad_ragged" in msg and word in msg, msg
        assert np.all(lml == 9.0) and np.all(grad == 9.0) and np.all(info == 9)
    assert lib.gpb200_lml_grad_ragged(handle._h, 0, None, None, None, None, 0.0, 1, None, None, None) == 0
    assert lib.gpb200_lml_grad_ragged(handle._h, 1, None, None, None, None, 0.0, 1, None, None, None) < 0
