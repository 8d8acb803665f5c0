"""Executed DMMA flops of the envelope route against the NumPy model of tests/test_envelope_fine_model.py: every GEMM CTA
of the Cholesky (panel and pure left-looking schedules) contracts from the first nonzero column of its own rows, and the
selected inverse ends its contraction at the last nonzero row of Y[S,J].  The counts must agree exactly, on sorted,
shuffled (non-monotone profile) and NaN inputs.  Half-tile configuration, eager launches (a CUDA graph replays the
counter it was recorded with)."""
import numpy as np
import pytest

from gp_b200 import capi
from test_envelope_fine_model import Profile, chol_flops, d_launch_flops, sinv_flops
from test_envelope_gpu import bench_like, routes

pytestmark = pytest.mark.gpu
N = 2048
NT = N // 128


def inputs(name, B):
    x, y, th = bench_like(N, B, 31)
    if name == "shuffled":
        # 128-point blocks in a random order, sorted inside: F is not monotone, and the rows of a tile keep a profile
        # that changes inside the tile
        p = np.random.default_rng(32).permutation(NT)
        x, y = (a.reshape(NT, 128)[p].ravel() for a in (x, y))
    elif name == "nan":
        x = np.tile(x, (B, 1))
        x[3, 777] = np.nan   # item 3: every row below 777 reaches column 777
    return x, y, th


def executed(monkeypatch, x, y, th, want_grad):
    monkeypatch.setenv("GPB200_NO_GRAPH", "1")
    h = capi.Handle(0)
    try:
        h.set_gemm_config(2)
        h.lib.gpb200_set_flop_counting(h._h, 1)
        _, _, info = h.lml_grad_batched(x, y, th, want_grad=want_grad)
        return h.lib.gpb200_executed_gemm_flops(h._h), info
    finally:
        h.close()


@pytest.mark.parametrize("B", [32, 64])   # 32: 8-tile panels with trailing updates; 64: pure left-looking
@pytest.mark.parametrize("name", ["sorted", "shuffled", "nan"])
def test_executed_flops_match_model(monkeypatch, name, B):
    x, y, th = inputs(name, B)
    assert routes(N, B) == (True, True)
    profiles = [Profile(x[b] if x.ndim == 2 else x, th[b, 1], NT) for b in range(B)]
    if name == "shuffled":
        assert any(np.any(np.diff(P.F) < 0) for P in profiles)
    chol = chol_flops(profiles, fine=True, cfg=2)
    assert chol < chol_flops(profiles, fine=False, cfg=2)
    got, info = executed(monkeypatch, x, y, th, want_grad=False)
    assert got == chol
    assert np.all(info[np.arange(B) != 3] == 0) if name == "nan" else np.all(info == 0)
    band = sinv_flops(profiles, fine=True, cfg=2)
    if name != "shuffled":   # a shuffled tile's last rows reach the columns of the tile before it: little to trim
        assert band < sinv_flops(profiles, fine=False, cfg=2)
    got, _ = executed(monkeypatch, x, y, th, want_grad=True)
    assert got == chol + band + B * d_launch_flops(NT)
