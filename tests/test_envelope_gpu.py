"""The tile envelope of the SE path of lml_grad_batched: envelope Cholesky (both passes) and the selected inverse
(the gradient when B * nt >= 256).

Every test asserts its premise: the batch takes the route it targets (envelope from 16 tile rows on, selected inverse
when B * nt >= 256, as in api_gp.cu) and the executed DMMA flops are below the dense count.  The dense route of a handle created with
GPB200_ENVELOPE=0 is the reference of the bit-identity checks."""
import numpy as np
import pytest

from gp_b200 import capi
from oracle import gp_oracle as o

pytestmark = pytest.mark.gpu
TILE = 128
SINV_MIN_BATCH = 16   # with nt >= 16 tile rows: B * nt >= 256, the selected-inverse route


def routes(n, B):
    """(envelope, selected inverse) as lml_core picks them (default handle)."""
    nt = (n + TILE - 1) // TILE
    env = 16 <= nt <= 512
    return env, env and B * nt >= 256
EXP_MIN = -708.3964185322641   # log(2^-1022): exp_nonpos flushes below this to exactly zero


def tile_profile(x, rho):
    """F (first tile column of each tile row with a nonzero exp(-d^2/2rho^2)) and E (last tile row I with F_I <= J)."""
    n = x.shape[0]
    nt = (n + TILE - 1) // TILE
    t = -0.5 * (x[:, None] - x[None, :]) ** 2 / rho ** 2
    nz = ~(t < EXP_MIN)   # NaN counts as nonzero
    F = np.empty(nt, dtype=int)
    for i in range(nt):
        row = nz[i * TILE:(i + 1) * TILE]
        F[i] = min(i, min(j for j in range(nt) if row[:, j * TILE:(j + 1) * TILE].any()))
    E = np.array([max(i for i in range(j, nt) if F[i] <= j) for j in range(nt)])
    return F, E


def chol_flops(F, with_env=True):
    """Flops of the Cholesky updates, 2 * 128^3 per (tile, k-tile) product, under the ENV_CHOL rule."""
    nt = F.shape[0]
    c = 0
    for i in range(nt):
        for j in range(i + 1):
            if with_env and j < F[i]:
                continue
            c += j - (max(F[i], F[j]) if with_env else 0)
    return 2.0 * TILE ** 3 * c


def lml_parity(lml, grad, x, y, th, items):
    for b in items:
        xb = x[b] if x.ndim == 2 else x
        yb = y[b] if y.ndim == 2 else y
        rv, rg = o.lml_grad_lapack(xb, yb, *th[b])
        assert abs(lml[b] - rv) / abs(rv) < 1e-9, b
        assert np.max(np.abs(grad[b] - rg)) / np.max(np.abs(rg)) < 1e-9, b


def bench_like(n, B, seed):
    rng = np.random.default_rng(seed)
    x = np.sort(rng.uniform(0.0, 0.05 * n, size=n))
    y = np.sin(x) + 0.5 * np.sin(3.1 * x) + 0.3 * rng.standard_normal(n)
    th = np.stack([np.abs(rng.standard_normal(B)) + 0.1, rng.gamma(4.0, 0.25, B), rng.uniform(0.1, 0.5, B)], axis=1)
    return x, y, th


def case(name):
    rng = np.random.default_rng(11)
    B = SINV_MIN_BATCH
    if name == "bench4096":
        x, y, th = bench_like(4096, B, 3)
    elif name == "ragged2100":
        x, y, th = bench_like(2100, B, 4)
    elif name == "shuffled":
        # 128-point blocks in a random order, shuffled inside each block: F is not monotone, most tiles stay zero
        x, y, th = bench_like(2100, B, 5)
        blocks = [np.arange(s, min(s + TILE, x.shape[0])) for s in range(0, x.shape[0], TILE)]
        p = np.concatenate([rng.permutation(blocks[i]) for i in rng.permutation(len(blocks))])
        x, y = x[p], y[p]
    elif name == "clustered":
        n = 2000
        centers = np.array([0.0, 40.0, 41.0, 90.0, 200.0])
        x = np.sort(np.concatenate([c + rng.uniform(0, 6.0, n // 5) for c in centers]))
        y = np.sin(x) + 0.3 * rng.standard_normal(n)
        _, _, th = bench_like(n, B, 6)
    elif name == "repeated":
        n = 2000
        x = np.sort(np.round(rng.uniform(0, 80.0, n), 1))
        y = np.sin(x) + 0.3 * rng.standard_normal(n)
        _, _, th = bench_like(n, B, 7)
    elif name == "tiny_alpha":
        x, y, th = bench_like(2000, B, 8)
        th[0, 0] = 1e-160   # alpha^2 e underflows to zero where e does not
    elif name == "mixed":
        x, y, th = bench_like(2000, B, 9)
        th[:, 1] = np.geomspace(0.02, 60.0, B)   # one tile of bandwidth up to fully dense
    return x, y, th


CASES = ["bench4096", "ragged2100", "shuffled", "clustered", "repeated", "tiny_alpha", "mixed"]


@pytest.mark.parametrize("name", CASES)
def test_parity_against_oracle(handle, name):
    x, y, th = case(name)
    B = th.shape[0]
    assert routes(x.shape[0], B) == (True, True)
    profs = [tile_profile(x, th[b, 1]) for b in range(B)]
    nt = profs[0][0].shape[0]
    # one uncounted call first: the first call of a small shape also runs the sequence that a CUDA graph then records
    handle.lml_grad_batched(x, y, th, want_grad=False)
    handle.lib.gpb200_set_flop_counting(handle._h, 1)
    lml, grad, info = handle.lml_grad_batched(x, y, th, want_grad=False)
    flops = handle.lib.gpb200_executed_gemm_flops(handle._h)
    handle.lib.gpb200_set_flop_counting(handle._h, 0)
    assert flops < B * chol_flops(np.zeros(nt, dtype=int), with_env=False)
    lml_g, grad, info_g = handle.lml_grad_batched(x, y, th)
    assert np.all(info == 0) and np.all(info_g == 0)
    assert np.all(np.abs(lml - lml_g) <= 1e-12 * np.abs(lml))
    if name == "mixed":
        bw = [int(np.max(np.arange(nt) - F)) for F, _ in profs]
        assert min(bw) <= 1 and max(bw) == nt - 1
    if name == "shuffled":
        assert any(np.any(np.diff(F) < 0) for F, _ in profs)
    items = [0, B // 2, B - 1] if x.shape[0] > 3000 else list(range(0, B, 3)) + [B - 1]
    lml_parity(lml_g, grad, x, y, th, items)


@pytest.fixture
def dense_handle(monkeypatch):
    monkeypatch.setenv("GPB200_ENVELOPE", "0")
    h = capi.Handle(0)
    yield h
    h.close()


@pytest.mark.parametrize("name", ["bench4096", "shuffled", "mixed"])
def test_against_dense_route(handle, dense_handle, name):
    x, y, th = case(name)
    l1, _, i1 = handle.lml_grad_batched(x, y, th, want_grad=False)
    l0, _, i0 = dense_handle.lml_grad_batched(x, y, th, want_grad=False)
    assert np.array_equal(i1, i0)
    assert np.array_equal(l1.view(np.int64), l0.view(np.int64))   # envelope Cholesky: bit-identical
    l1, g1, i1 = handle.lml_grad_batched(x, y, th)
    l0, g0, i0 = dense_handle.lml_grad_batched(x, y, th)
    assert np.array_equal(i1, i0)
    assert np.all(np.abs(l1 - l0) <= 1e-12 * np.abs(l0))
    for b in range(th.shape[0]):
        assert np.max(np.abs(g1[b] - g0[b])) <= 1e-10 * np.max(np.abs(g0[b])), b


def test_failed_items_leave_neighbours_alone(handle, dense_handle):
    x, y, th = case("ragged2100")
    th = th.copy()
    th[3, 2] = 0.0
    th[3, 0] = 30.0
    th[3, 1] = 40.0          # no noise, long length scale: numerically singular
    th[7, 1] = np.nan        # a NaN item
    lml, grad, info = handle.lml_grad_batched(x, y, th)
    lml0, grad0, info0 = dense_handle.lml_grad_batched(x, y, th)
    assert info[3] != 0
    assert np.array_equal(info, info0)
    ok = [b for b in range(th.shape[0]) if b not in (3, 7)]
    assert np.all(np.abs(lml[ok] - lml0[ok]) <= 1e-12 * np.abs(lml0[ok]))
    lml_parity(lml, grad, x, y, th, [2, 4, 8])


def test_chunked_batches(handle):
    x, y, th = case("clustered")
    n = x.shape[0]
    np_ = (n + TILE - 1) // TILE * TILE
    h = capi.Handle(0)
    try:
        h.set_workspace_limit(int(5.5 * 2 * np_ * np_ * 8))   # a few items per chunk
        lml, grad, info = h.lml_grad_batched(x, y, th)
    finally:
        h.close()
    lml1, grad1, info1 = handle.lml_grad_batched(x, y, th)
    assert np.array_equal(info, info1)
    assert np.all(np.abs(lml - lml1) <= 1e-12 * np.abs(lml1))
    for b in range(th.shape[0]):
        assert np.max(np.abs(grad[b] - grad1[b])) <= 1e-10 * np.max(np.abs(grad1[b])), b


def test_device_pointer_mode(handle):
    torch = pytest.importorskip("torch")
    x, y, th = case("shuffled")
    B, n = th.shape[0], x.shape[0]
    lml, grad, info = handle.lml_grad_batched(x, y, th)
    h = capi.Handle(0)
    try:
        dev = torch.device("cuda", 0)
        h.set_stream(torch.cuda.current_stream(dev).cuda_stream)
        h.set_pointer_mode(True)
        dx, dy, dth = (torch.from_numpy(np.ascontiguousarray(a)).to(dev) for a in (x, y, th))
        dl = torch.empty(B, dtype=torch.float64, device=dev)
        dg = torch.empty(B, 3, dtype=torch.float64, device=dev)
        di = torch.zeros(B, dtype=torch.int32, device=dev)
        h.lml_grad_batched_device(n, B, dx, 0, dy, 0, dth, 0.0, True, dl, dg, di)
        torch.cuda.current_stream(dev).synchronize()
        assert np.array_equal(di.cpu().numpy(), info)
        assert np.array_equal(dl.cpu().numpy().view(np.int64), lml.view(np.int64))
        assert np.array_equal(dg.cpu().numpy().view(np.int64), grad.view(np.int64))
    finally:
        h.close()


def test_graph_replay_matches_eager(handle, monkeypatch):
    x, y, th = bench_like(2000, SINV_MIN_BATCH, 12)   # B * nt^2 = 4096: the sequence is replayed as a CUDA graph
    assert routes(2000, SINV_MIN_BATCH) == (True, True)
    r0 = handle.graph_replays()
    out = [handle.lml_grad_batched(x, y, th) for _ in range(3)]
    assert handle.graph_replays() - r0 == 3
    monkeypatch.setenv("GPB200_NO_GRAPH", "1")
    h = capi.Handle(0)
    try:
        eager = h.lml_grad_batched(x, y, th)
    finally:
        h.close()
    for got in out:
        for a, b in zip(got, eager):
            assert np.array_equal(np.asarray(a).view(np.uint8), np.asarray(b).view(np.uint8))


def test_flop_counter_matches_profile(monkeypatch):
    """LML-only, two items (the look-ahead schedule), half-tile configuration (no CTA-level skipping besides the
    envelope): executed flops = 2 * 128^3 per kept (tile, k-tile) product of the numpy profile.  Eager launches: a
    CUDA graph replays the counter it was recorded with."""
    x, y, th = bench_like(2000, 2, 13)
    assert routes(2000, 2) == (True, False)
    monkeypatch.setenv("GPB200_NO_GRAPH", "1")
    h = capi.Handle(0)
    try:
        h.set_gemm_config(2)
        h.lib.gpb200_set_flop_counting(h._h, 1)
        _, _, info = h.lml_grad_batched(x, y, th, want_grad=False)
        got = h.lib.gpb200_executed_gemm_flops(h._h)
    finally:
        h.close()
    assert np.all(info == 0)
    want = sum(chol_flops(tile_profile(x, th[b, 1])[0]) for b in range(2))
    dense = 2 * chol_flops(np.zeros(16, dtype=int), with_env=False)
    assert want < dense
    assert got == want
