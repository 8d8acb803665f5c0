"""The envelope route of lml_grad_batched at batch sizes where the throughput TRSM kernels solve several row tiles per
CTA, and the dispatch order of its GEMM launches (widest-band items first).

The batched TRSM solves only the tiles (I, J) with F_I <= J; every other tile is exactly zero and stays as the Gram
wrote it, so the factor is bit-identical to the dense route of a GPB200_ENVELOPE=0 handle.  The GEMM launches take the
items by descending bandwidth; each item's arithmetic does not depend on where it is dispatched, so a batch permuted
into that order gives bit-identical results item by item."""
import numpy as np
import pytest

from gp_b200 import capi
from test_envelope_gpu import TILE, bench_like, lml_parity, routes, tile_profile

pytestmark = pytest.mark.gpu

N = 2048
B = 160   # 15 row tiles below the first diagonal tile x 160 items >= 148 * 16: the pipelined TRSM takes several row
          # tiles per CTA (two with the envelope, four on the dense route; panel.cu)


def handle_with(monkeypatch, **env):
    for k, v in env.items():
        monkeypatch.setenv(k, v)
    h = capi.Handle(0)
    for k in env:
        monkeypatch.delenv(k)
    return h


def shuffled(x, y, seed):
    """128-point blocks in a random order, shuffled inside each block: F is not monotone."""
    rng = np.random.default_rng(seed)
    blocks = [np.arange(s, min(s + TILE, x.shape[0])) for s in range(0, x.shape[0], TILE)]
    p = np.concatenate([rng.permutation(blocks[i]) for i in rng.permutation(len(blocks))])
    return x[p], y[p]


def bandwidth(x, rho):
    F, _ = tile_profile(x, rho)
    return int(np.max(np.arange(F.shape[0]) - F))


def dead_trsm_tiles(x, rho):
    """TRSM tiles (I > J) outside the envelope: F_I > J."""
    F, _ = tile_profile(x, rho)
    return sum(int(F[i] > j) for i in range(F.shape[0]) for j in range(i))


def dead_between_live(x, rho):
    """Tiles outside the envelope with a live tile further down the same block column (F not monotone)."""
    F, _ = tile_profile(x, rho)
    nt = F.shape[0]
    return sum(int(F[i] > j and np.any(F[i + 1:] <= j)) for j in range(nt) for i in range(j + 1, nt))


@pytest.mark.parametrize("pipelined", ["1", "0"])
@pytest.mark.parametrize("order", ["sorted", "shuffled"])
def test_lml_bit_identical_to_dense_route(monkeypatch, order, pipelined):
    x, y, th = bench_like(N, B, 21)
    if order == "shuffled":
        x, y = shuffled(x, y, 22)
        assert sum(dead_between_live(x, th[b, 1]) for b in range(0, B, 16)) > 0
    assert routes(N, B)[0]
    assert sum(dead_trsm_tiles(x, th[b, 1]) for b in range(0, B, 16)) > 0
    h = handle_with(monkeypatch, GPB200_TRSM_PIPELINED=pipelined)
    h0 = handle_with(monkeypatch, GPB200_TRSM_PIPELINED=pipelined, GPB200_ENVELOPE="0")
    try:
        l1, _, i1 = h.lml_grad_batched(x, y, th, want_grad=False)
        l0, _, i0 = h0.lml_grad_batched(x, y, th, want_grad=False)
    finally:
        h.close()
        h0.close()
    assert np.all(i0 == 0)
    assert np.array_equal(i1, i0)
    assert np.array_equal(l1.view(np.int64), l0.view(np.int64))


def mixed_batch(Bm=32, n=2000):
    x, y, th = bench_like(n, Bm, 23)
    th[:, 1] = np.geomspace(0.02, 60.0, Bm)   # bandwidth from one tile to the whole matrix, ascending in the item index
    return x, y, th


def test_dispatch_order_does_not_change_results(handle):
    x, y, th = mixed_batch()
    Bm = th.shape[0]
    assert routes(x.shape[0], Bm) == (True, True)
    bw = np.array([bandwidth(x, th[b, 1]) for b in range(Bm)])
    p = np.argsort(-bw, kind="stable")       # the order the GEMM launches take: descending bandwidth, ties by index
    assert not np.array_equal(p, np.arange(Bm))
    l1, g1, i1 = handle.lml_grad_batched(x, y, th)
    l2, g2, i2 = handle.lml_grad_batched(x, y, th[p])   # already in dispatch order
    inv = np.argsort(p)
    assert np.all(i1 == 0)
    assert np.array_equal(i2[inv], i1)
    assert np.array_equal(l2[inv].view(np.int64), l1.view(np.int64))
    assert np.array_equal(g2[inv].view(np.int64), g1.view(np.int64))
    lml_parity(l1, g1, x, y, th, [0, Bm // 2, Bm - 1])


def test_failed_item_late_pivot(handle, monkeypatch):
    """A negative jitter makes K + jitter I indefinite wherever points crowd.  Item 5 has its first 1829 points far
    apart (K is diagonal there) and a dense cluster after them: its first non-positive pivot falls in tile column 14
    of 16.  Item 9 (no noise, long length scale) fails at once.  The other items keep sigma^2 + jitter > 0."""
    jitter = -0.05
    x1, y, th = bench_like(N, B, 24)
    th[:, 2] = np.random.default_rng(25).uniform(0.3, 0.5, B)
    x = np.tile(x1, (B, 1))
    late = 14 * TILE + 37
    x[5, :late] = np.arange(late) * 50.0
    x[5, late:] = 1e6 + (x1[late:] - x1[late])
    th[5] = (1.0, 1.0, 0.1)
    th[9] = (30.0, 40.0, 0.0)
    h0 = handle_with(monkeypatch, GPB200_ENVELOPE="0")
    try:
        lml0, grad0, info0 = h0.lml_grad_batched(x, y, th, jitter)
    finally:
        h0.close()
    lml, grad, info = handle.lml_grad_batched(x, y, th, jitter)
    assert (info0[5] - 1) // TILE == 14 and info0[9] != 0
    assert np.array_equal(info, info0)
    ok = [b for b in range(B) if b not in (5, 9)]
    assert np.all(info[ok] == 0)
    assert np.all(np.abs(lml[ok] - lml0[ok]) <= 1e-12 * np.abs(lml0[ok]))
    for b in ok:
        assert np.max(np.abs(grad[b] - grad0[b])) <= 1e-10 * np.max(np.abs(grad0[b])), b


def test_chunked_call_matches_unchunked(handle):
    x, y, th = mixed_batch(Bm=48)
    Bm, n = th.shape[0], x.shape[0]
    np_ = (n + TILE - 1) // TILE * TILE
    h = capi.Handle(0)
    try:
        h.set_workspace_limit(int(11.5 * 2 * np_ * np_ * 8))   # about eleven items per chunk: five chunks
        lml, grad, info = h.lml_grad_batched(x, y, th)
    finally:
        h.close()
    lml1, grad1, info1 = handle.lml_grad_batched(x, y, th)
    assert np.all(info1 == 0)
    assert np.array_equal(info, info1)
    assert np.all(np.abs(lml - lml1) <= 1e-12 * np.abs(lml1))
    for b in range(Bm):
        assert np.max(np.abs(grad[b] - grad1[b])) <= 1e-10 * np.max(np.abs(grad1[b])), b
