"""Contract checks of the C ABI (include/gpb200.h) that the parity tests do not reach: explicit leading dimensions
and strides, device-pointer mode and stream ordering, the LML-only batched substitution and the
derivative-observation LML + gradient on half tiles and under the diagonal split.

The entry points are called through the raw symbols (h.lib.gpb200_*), because the capi wrappers always pass
dense leading dimensions.  Device buffers are torch CUDA tensors.

Vector accesses to caller memory.  In device mode the kernels read and write the caller's arrays directly, so
an odd leading dimension or stride must never meet a 16-byte access.  The kernels that touch caller memory in
that mode -- pack_kernel / unpack_kernel (solve.cu), gram_outer_kernel, gram_ard_kernel, gram_deriv_kernel and
approx_basis_kernel (gram.cu), add_mean_transpose_kernel and normal_fill_kernel (rng.cu), lml_small_kernel
(small.cu), hermite_kernel / hermite_matvec_kernel (solve.cu), trmv_lower_n_kernel reading the right-hand side
of gp_condition, kernel_eval_kernel -- all use scalar accesses, except gram_outer_kernel, whose paired store
falls back to scalar stores unless ldk is even and K is 16-byte aligned (gram.cu:57).  So every entry point
accepts any leading dimension >= the row count, and the odd ones below run in device mode as well.
"""
import ctypes as C

import numpy as np
import pytest
import scipy.linalg as sla

from gp_b200 import capi
from oracle import gp_oracle as o
from oracle import philox

torch = pytest.importorskip("torch")

pytestmark = pytest.mark.gpu

F64_SENTINEL = np.uint64(0x7FF8DEADBEEF5A5A)   # a quiet NaN whose payload no kernel produces
I32_SENTINEL = np.int32(-1515870811)           # 0xA5A5A5A5
NSM = 148


def relerr(a, b):
    a = np.asarray(a, dtype=np.float64); b = np.asarray(b, dtype=np.float64)
    return float(np.max(np.abs(a - b)) / max(np.max(np.abs(b)), 1e-300))


def assert_lml_close(got, ref, rtol=1e-9, ctx=None):
    assert abs(got - ref) <= rtol * abs(ref), (ctx, got, ref)


def assert_grad_close(got, ref, rtol=1e-9, ctx=None):
    """Each component against its own magnitude.  A component below 1e-6 of the largest one is the difference of
    terms of the size of the largest (the trace and quadratic-form sums cancel), so its rounding error scales with
    the largest component: there, and only there, the norm-wise bound applies."""
    got = np.asarray(got, dtype=np.float64); ref = np.asarray(ref, dtype=np.float64)
    scale = float(np.max(np.abs(ref)))
    for k in range(ref.shape[0]):
        bound = rtol * (abs(ref[k]) if abs(ref[k]) >= 1e-6 * scale else scale)
        assert abs(got[k] - ref[k]) <= bound, (ctx, k, got, ref)


# ---- branch predicates, mirrored from the C host code --------------------------------------------------------
def small_in_place(n):
    """lml_small_applies (small.cu:335) with the default knob: the one-CTA kernel, which in device mode reads and
    writes the caller's arrays in place (api_gp.cu:33-38)."""
    return n <= 128


def gemm_cfg(ntasks, batch):
    """gemm_pick_cfg (gemm.cu:480-484) with the default knobs: 3 = quarter tiles, 2 = half tiles."""
    return 3 if ntasks * batch * 2 < 2 * NSM * 2 else 2


def diag_split(ntasks, batch):
    """diag_split_applies (gemm.cu:528-530)."""
    return gemm_cfg(ntasks, batch) == 2 and batch >= 16 and ntasks * batch >= 2048


def lauum_tasks(nt):
    """tasks_lauum (engine.cu:151-162): one task per lower tile."""
    return nt * (nt + 1) // 2


def tiles(n):
    return (n + 127) // 128


def uses_trsv_blocked(bc):
    """LML-only chunk of the batched path: trsv_blocked from 32 items on, trsv_sweep below (api_gp.cu:105-106)."""
    return bc >= 32


def uses_graph(n, B, chunk=None):
    """lml_core replays the evaluation as one CUDA graph (api_gp.cu:121)."""
    nt = tiles(n)
    return not small_in_place(n) and (chunk is None or chunk == B) and nt <= 64 and B * nt * nt <= 4096


def uses_lookahead(n, B):
    """chol_uses_lookahead (engine.cu:196-200) with the default knobs."""
    nt = tiles(n)
    return B <= 64 and B * nt <= 256 and nt >= 3


def _pad256(b):
    return (b + 255) & ~255


def lml_chunk(n_grid, B, limit, nblocks=1, deriv=False, x_per_item=False, y_per_item=False):
    """Items per chunk under a workspace limit: the arithmetic of lml_core (api_gp.cu:20-53)."""
    n = n_grid * nblocks
    ts, pw = (2 + nblocks, 8) if deriv else (3, 4)
    np_ = tiles(n) * 128
    nt = np_ // 128
    nparts = lauum_tasks(nt) * 4
    ctas = nt * B
    zks = 1 if (ctas >= 2 * NSM or nt < 4) else min(nt, (2 * NSM + ctas - 1) // ctas)
    per_item = (_pad256(np_ * np_ * 8) * 2 + 3 * _pad256(np_ * 8) + _pad256(nparts * pw * 8)
                + (_pad256(zks * np_ * 8) if zks > 1 else 0) + 64)
    fixed = (_pad256(B * (n_grid if x_per_item else 0) * 8 + n_grid * 8) + _pad256(B * (n if y_per_item else 0) * 8 + n * 8)
             + 2 * _pad256(B * ts * 8) + _pad256(B * 8) + _pad256(B * 4) + 4096)
    return min(B, (limit - fixed - 8192) // per_item), fixed, per_item


def limit_for_chunk(n_grid, B, chunk, **kw):
    _, fixed, per_item = lml_chunk(n_grid, B, 1 << 62, **kw)
    limit = fixed + 8192 + chunk * per_item + per_item // 2
    assert lml_chunk(n_grid, B, limit, **kw)[0] == chunk
    return limit


@pytest.fixture(scope="module")
def h():
    hd = capi.Handle(0)
    yield hd
    hd.close()


class device_mode:
    """Device-pointer mode with the handle bound to a stream (default: torch's current stream); restores host
    mode and the default stream on exit."""

    def __init__(self, hd, stream=None):
        self.hd, self.stream = hd, stream

    def __enter__(self):
        s = self.stream if self.stream is not None else torch.cuda.current_stream()
        self.hd.set_stream(s.cuda_stream)
        self.hd.set_pointer_mode(True)
        return self.hd

    def __exit__(self, *exc):
        self.hd.set_pointer_mode(False)
        self.hd.set_stream(torch.cuda.current_stream().cuda_stream)
        return False


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64) if a.dtype == np.float64 else a.view(np.uint32)


# ---- A. leading dimensions, guard bands, host and device mode ----------------------------------------------
class Arg:
    """One array argument.  role: 'in', 'out' or 'inout'; data: (rows, cols) window (1-D = one column); has_ld: the
    entry point takes a leading dimension (or a stride) for it; host: a host array in either pointer mode."""

    def __init__(self, role, data, has_ld=False, host=False):
        d = np.asarray(data)
        self.role, self.has_ld, self.host = role, has_ld, host
        self.data = d.reshape(-1, 1) if d.ndim == 1 else d
        self.dtype = self.data.dtype

    def ld(self, pad):
        rows = self.data.shape[0]
        return max(rows, 1) + (pad if self.has_ld else 0)

    def build(self, pad):
        rows, cols = self.data.shape
        ld = self.ld(pad)
        size = ld * cols + max(ld, 8)   # one trailing guard column (at least 8 elements)
        if self.role == "in":
            full = np.full(size, np.nan) if self.dtype == np.float64 else np.full(size, I32_SENTINEL, np.int32)
        elif self.dtype == np.float64:
            full = np.full(size, F64_SENTINEL, np.uint64).view(np.float64)
        else:
            full = np.full(size, I32_SENTINEL, np.int32)
        if self.role != "out":
            self.window(full, ld)[...] = self.data
        return full, ld

    def window(self, full, ld):
        rows, cols = self.data.shape
        return full[:ld * cols].reshape(cols, ld).T[:rows]

    def gaps(self, full, ld):
        mask = np.ones(full.shape[0], bool)
        self.window(mask, ld)[...] = False
        return full[mask]


def _run(hd, args, call, pad, device):
    bufs, lds = {}, {}
    for k, a in args.items():
        bufs[k], lds[k] = a.build(pad)
    orig = {k: v.copy() for k, v in bufs.items()}
    if not device:
        rc = call(hd, {k: v.ctypes.data for k, v in bufs.items()}, lds)
        return rc, bufs, lds, orig
    tens = {k: (v if args[k].host else torch.from_numpy(v).cuda()) for k, v in bufs.items()}
    ptrs = {k: (t.ctypes.data if args[k].host else t.data_ptr()) for k, t in tens.items()}
    with device_mode(hd):
        rc = call(hd, ptrs, lds)
    torch.cuda.current_stream().synchronize()
    return rc, {k: (t if args[k].host else t.cpu().numpy()) for k, t in tens.items()}, lds, orig


def check_layouts(hd, args, call, pads=(1, 37), expect_rc=0):
    """Runs `call` dense in host mode (the reference), then with ld = rows + pad in host mode and dense and padded in
    device mode, and checks (i) every output window bit-identical to the reference, (ii) every output gap and guard
    element still the sentinel, (iii) every input buffer unchanged, gaps included; (iv) device mode is bit-identical
    to host mode because both are compared with the same reference.  Returns the reference output windows."""
    rc, ref, ref_lds, _ = _run(hd, args, call, 0, False)
    assert rc == expect_rc, (rc, hd.lib.gpb200_last_error(hd._h))
    ref_win = {k: a.window(ref[k], ref_lds[k]).copy() for k, a in args.items()}
    for device in (False, True):
        for pad in ((0,) + tuple(pads)) if device else tuple(pads):
            rc, got, lds, orig = _run(hd, args, call, pad, device)
            ctx = ("device" if device else "host", pad)
            assert rc == expect_rc, (ctx, rc, hd.lib.gpb200_last_error(hd._h))
            for k, a in args.items():
                g, ld = got[k], lds[k]
                if a.role == "in":
                    assert np.array_equal(_bits(g), _bits(orig[k])), (ctx, k, "input modified")
                    continue
                assert np.array_equal(_bits(a.window(g, ld)), _bits(ref_win[k])), (ctx, k, "window differs from dense host")
                sent = F64_SENTINEL if a.dtype == np.float64 else np.uint32(np.int64(I32_SENTINEL) & 0xFFFFFFFF)
                assert np.all(_bits(a.gaps(g, ld)) == sent), (ctx, k, "gap or guard element written")
    return {k: (w[:, 0] if w.shape[1] == 1 else w) for k, w in ref_win.items() if args[k].role != "in"}


def _spd(n, seed, diag=0.09):
    x, _ = o.synth_xy(n, seed)
    return o.gram_se(x, 1.1, 0.8, diag)


def _lower_nan_upper(L):
    """A factor with NaN in its strict upper triangle: the entry points take the lower triangle only."""
    M = np.tril(L).copy()
    M[np.triu_indices(L.shape[0], 1)] = np.nan
    return M


def case_gram_outer(n, m=None):
    m = n + 2 if m is None else m
    rng = np.random.default_rng(n)
    x = np.sort(rng.uniform(-2, 2, n)); y = np.sort(rng.uniform(-2, 2, m))
    args = {"x": Arg("in", x), "y": Arg("in", y), "K": Arg("out", np.zeros((n, m)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_gram_outer(hd._h, capi.KINDS["RT"], n, m, p["x"], p["y"], 1.7, 0.6, p["K"], ld["K"])
    return args, call, lambda r: relerr(r["K"], 1.7 * o.outer_kernel("RT", x, y, 0.6)) < 1e-13


def case_gram_ard(n, m=None):
    m = n + 2 if m is None else m
    rng = np.random.default_rng(n)
    X = rng.standard_normal((n, 3)); Y = rng.standard_normal((m, 3)); rho = np.array([0.5, 1.0, 2.0])
    args = {"X": Arg("in", X, True), "Y": Arg("in", Y, True), "rho": Arg("in", rho), "K": Arg("out", np.zeros((n, m)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_gram_ard(hd._h, n, m, 3, p["X"], ld["X"], p["Y"], ld["Y"], 1.3, p["rho"], p["K"], ld["K"])
    return args, call, lambda r: relerr(r["K"], o.rk_QQard(X, Y, (1.3, rho))) < 1e-13


def case_gram_se(n, m=None):
    x, _ = o.synth_xy(n, 11)
    args = {"x": Arg("in", x), "K": Arg("out", np.zeros((n, n)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_gram_se(hd._h, n, p["x"], 1.3, 0.7, 0.09, p["K"], ld["K"])
    return args, call, lambda r: relerr(r["K"], o.gram_se(x, 1.3, 0.7, 0.09)) < 1e-14


def case_gram_deriv(n, m=None):
    t = np.linspace(0, 0.1 * n + 1, n); noise = np.array([0.1, 0.2, 0.3])
    args = {"t": Arg("in", t), "noise": Arg("in", noise), "K": Arg("out", np.zeros((3 * n, 3 * n)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_gram_deriv(hd._h, n, p["t"], 1.2, 0.9, 3, p["noise"], 1e-6, 0, p["K"], ld["K"])
    return args, call, lambda r: relerr(r["K"], o.gram_deriv(t, 1.2, 0.9, noise, 1e-6, 3)) < 1e-13


def case_approx_L_basis(n, m=None):
    x = np.linspace(-1, 1, n); M = 7
    args = {"x": Arg("in", x), "out": Arg("out", np.zeros((n, M)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_approx_L_basis(hd._h, n, M, 0.25, p["x"], 1.3, 0.4, p["out"], ld["out"])
    return args, call, lambda r: relerr(r["out"], o.approx_L_basis(M, 0.25, x, 1.3, 0.4)) < 1e-12


def case_potrf(n, m=None):
    K = _spd(n, 3)
    args = {"A": Arg("inout", K, True)}
    call = lambda hd, p, ld: hd.lib.gpb200_potrf(hd._h, n, p["A"], ld["A"])

    def oracle(r):
        return relerr(r["A"], o.cholesky_decompose(K)) < 1e-9 and np.all(np.triu(r["A"], 1) == 0.0)
    return args, call, oracle


def _solve_case(n, nrhs, both):
    K = _spd(n, 7, 0.04)
    L = o.cholesky_decompose(K)
    B = np.random.default_rng(n).standard_normal((n, nrhs))
    args = {"L": Arg("in", _lower_nan_upper(L), True), "B": Arg("inout", B, True)}
    f = "gpb200_potrs" if both else "gpb200_trsm_lower"
    call = lambda hd, p, ld: getattr(hd.lib, f)(hd._h, n, nrhs, p["L"], ld["L"], p["B"], ld["B"])
    ref = (lambda: sla.cho_solve((L, True), B)) if both else (lambda: sla.solve_triangular(L, B, lower=True))
    return args, call, lambda r: relerr(r["B"], ref()) < (1e-8 if both else 1e-9)


def case_trsm_lower(n, m=None):
    return _solve_case(n, 5 if m is None else m, False)


def case_potrs(n, m=None):
    return _solve_case(n, 5 if m is None else m, True)


def _trmv_case(n, trans):
    L = o.cholesky_decompose(_spd(n, 5))
    z = np.random.default_rng(n).standard_normal(n)
    args = {"L": Arg("in", _lower_nan_upper(L), True), "z": Arg("in", z), "f": Arg("out", np.zeros(n))}
    fn = "gpb200_trmv_lower_t" if trans else "gpb200_trmv_lower"
    call = lambda hd, p, ld: getattr(hd.lib, fn)(hd._h, n, p["L"], ld["L"], p["z"], p["f"])
    return args, call, lambda r: relerr(r["f"], (L.T if trans else L) @ z) < 1e-12


def case_trmv_lower(n, m=None):
    return _trmv_case(n, False)


def case_trmv_lower_t(n, m=None):
    return _trmv_case(n, True)


def case_mvn_chol_lpdf(n, m=None):
    L = o.cholesky_decompose(_spd(n, 9))
    _, y = o.synth_xy(n, 9)
    mu = 0.1 * np.random.default_rng(n).standard_normal(n)
    args = {"y": Arg("in", y), "mu": Arg("in", mu), "L": Arg("in", _lower_nan_upper(L), True), "lp": Arg("out", np.zeros(1))}
    call = lambda hd, p, ld: hd.lib.gpb200_mvn_chol_lpdf(hd._h, n, p["y"], p["mu"], p["L"], ld["L"], 0, p["lp"])

    def oracle(r):
        ref = o.multi_normal_cholesky_lpdf(y, mu, L)
        return abs(r["lp"][0] - ref) <= 1e-9 * abs(ref)
    return args, call, oracle


def case_gp_condition(n, m=None):
    m = n // 2 + 2 if m is None else m
    t = np.linspace(0, 0.05 * n + 1, n); ts = np.linspace(0.01, 0.05 * n + 0.9, m)
    K = 1.2 * o.outer_kernel("QQ", t, t, 0.7); Ks = 1.2 * o.outer_kernel("QQ", ts, t, 0.7)
    Kss = 1.2 * o.outer_kernel("QQ", ts, ts, 0.7)
    y = np.sin(t)
    args = {"K": Arg("in", K, True), "Ks": Arg("in", Ks, True), "Kss": Arg("in", Kss, True), "y": Arg("in", y),
            "mu": Arg("out", np.zeros(m)), "cov": Arg("out", np.zeros((m, m)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_gp_condition(hd._h, n, m, p["K"], ld["K"], p["Ks"], ld["Ks"], p["Kss"], ld["Kss"],
                                                        p["y"], 0.04, 1e-8, p["mu"], p["cov"], ld["cov"])

    def oracle(r):
        rmu, rcov = o.gp_condition(K, Ks, Kss, y, 0.04, 1e-8)
        return relerr(r["mu"], rmu) < 1e-8 and relerr(r["cov"], rcov) < 1e-8
    return args, call, oracle


def case_cond_mvn(n, m=None):
    ng, nd = n, (n // 3 + 1 if m is None else m)
    N = ng + nd
    S = _spd(N, 13, 0.05)
    mean = 0.1 * np.arange(N); xg = np.sin(np.arange(ng))
    args = {"mean": Arg("in", mean), "S": Arg("in", S, True), "xg": Arg("in", xg),
            "cm": Arg("out", np.zeros(nd)), "cv": Arg("out", np.zeros((nd, nd)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_cond_mvn(hd._h, ng, nd, p["mean"], p["S"], ld["S"], p["xg"], p["cm"], p["cv"], ld["cv"])

    def oracle(r):
        rm, rv = o.condMVN(mean, S, list(range(ng, N)), list(range(ng)), xg)
        return relerr(r["cm"], rm) < 1e-8 and relerr(r["cv"], rv) < 1e-8
    return args, call, oracle


def case_mvrnorm(n, m=None):
    mdim, nd = n, (n // 2 + 1 if m is None else m)
    S = _spd(mdim, 17, 0.05)
    mu = np.linspace(-1, 1, mdim)
    args = {"mu": Arg("in", mu), "S": Arg("in", S, True), "out": Arg("out", np.zeros((nd, mdim)), True)}
    call = lambda hd, p, ld: hd.lib.gpb200_mvrnorm(hd._h, nd, mdim, p["mu"], p["S"], ld["S"], 1e-9, 99, p["out"], ld["out"])

    def oracle(r):   # test_host_mirror_gpu.py::test_mvrnorm_is_mean_plus_chol_times_the_stream checks the draws the same way
        Z = philox.normals(99, mdim * nd).reshape(nd, mdim)
        L = o.cholesky_decompose(o.add_diag(S, 1e-9))
        out = r["out"].reshape(nd, mdim)
        return relerr(out, mu[None, :] + Z @ L.T) < 1e-10
    return args, call, oracle


def case_rbf_cov_chol(n, m=None):
    x = np.arange(n) * 1.0 + 0.1 * np.sin(np.arange(n))
    args = {"x": Arg("in", x), "L": Arg("out", np.zeros(n * n)), "dL": Arg("out", np.zeros(n * n))}
    call = lambda hd, p, ld: hd.lib.gpb200_rbf_cov_chol(hd._h, n, p["x"], 0.7, p["L"], p["dL"])

    def oracle(r):
        Lr, dLr = o.rbf_cov_chol(x, 0.7)
        return relerr(r["L"].reshape(n, n, order="F"), Lr) < 1e-9 and relerr(r["dL"].reshape(n, n, order="F"), dLr) < 1e-8
    return args, call, oracle


def case_rbf_cov_chol_batched(n, m=None):
    x = np.arange(n) * 1.0 + 0.1 * np.sin(np.arange(n))
    ls = np.array([0.5, 0.6, 0.7]); P = 3
    args = {"x": Arg("in", x), "ls": Arg("in", ls, host=True), "L": Arg("out", np.zeros(P * n * n)),
            "dL": Arg("out", np.zeros(P * n * n)), "info": Arg("out", np.zeros(P, np.int32), host=True)}
    call = lambda hd, p, ld: hd.lib.gpb200_rbf_cov_chol_batched(hd._h, n, p["x"], P, p["ls"], p["L"], p["dL"], p["info"])

    def oracle(r):
        ok = np.all(r["info"] == 0)
        for q in range(P):
            Lr, dLr = o.rbf_cov_chol(x, ls[q])
            ok &= relerr(r["L"][q * n * n:(q + 1) * n * n].reshape(n, n, order="F"), Lr) < 1e-9
            ok &= relerr(r["dL"][q * n * n:(q + 1) * n * n].reshape(n, n, order="F"), dLr) < 1e-8
        return ok
    return args, call, oracle


def _latent_inputs(n):
    x = 0.5 * np.arange(n) + 0.05 * np.sin(np.arange(n))   # well conditioned with rho = 0.8 and diag_add = 0.05
    rng = np.random.default_rng(n)
    return x, rng.standard_normal(2 * n), rng.standard_normal(2 * n)


def case_latent_forward(n, m=None):
    x, z, _ = _latent_inputs(n)
    args = {"x": Arg("in", x), "z": Arg("in", z), "f": Arg("out", np.zeros(2 * n))}
    call = lambda hd, p, ld: hd.lib.gpb200_latent_forward(hd._h, n, p["x"], 1.1, 0.8, 0.05, 2, p["z"], p["f"])

    def oracle(r):
        L = o.cholesky_decompose(o.gram_se(x, 1.1, 0.8, 0.05))
        return relerr(r["f"].reshape(2, n), z.reshape(2, n) @ L.T) < 1e-10
    return args, call, oracle


def case_latent_backward(n, m=None):
    x, z, fbar = _latent_inputs(n)
    args = {"x": Arg("in", x), "z": Arg("in", z), "fbar": Arg("in", fbar), "tb": Arg("out", np.zeros(2)),
            "zbar": Arg("out", np.zeros(2 * n))}
    call = lambda hd, p, ld: hd.lib.gpb200_latent_backward(hd._h, n, p["x"], 1.1, 0.8, 0.05, 2, p["z"], p["fbar"], p["tb"], p["zbar"])

    def oracle(r):   # theta_bar: test_host_mirror_gpu.py::test_reverse_mode_cholesky_adjoint_matches_oracle_and_forward_mode
        L = o.cholesky_decompose(o.gram_se(x, 1.1, 0.8, 0.05))
        return relerr(r["zbar"].reshape(2, n), fbar.reshape(2, n) @ L) < 1e-10 and np.all(np.isfinite(r["tb"]))
    return args, call, oracle


def _tables(n):
    x = np.arange(n) * 1.0 + 0.1 * np.sin(np.arange(n))
    lp = np.array([0.5, 0.6, 0.7])
    Ls, dLs = zip(*[o.rbf_cov_chol(x, l) for l in lp])
    return lp, Ls, dLs


def case_approx_L(n, m=None):
    lp, Ls, dLs = _tables(n)
    args = {"lp": Arg("in", lp, host=True), "out": Arg("out", np.zeros(n * n))}
    for q in range(3):
        args["L%d" % q] = Arg("in", Ls[q].ravel(order="F"))
        args["D%d" % q] = Arg("in", dLs[q].ravel(order="F"))

    def call(hd, p, ld):
        pa = (C.c_void_p * 3)(*[p["L%d" % q] for q in range(3)])
        pb = (C.c_void_p * 3)(*[p["D%d" % q] for q in range(3)])
        return hd.lib.gpb200_approx_L(hd._h, n, 0.66, 3, p["lp"], pa, pb, p["out"])
    return args, call, lambda r: relerr(r["out"].reshape(n, n, order="F"), o.approx_L(0.66, lp, Ls, dLs)) < 1e-13


def case_approx_Lz(n, m=None):
    lp, Ls, dLs = _tables(n)
    z = np.cos(np.arange(n))
    args = {"lp": Arg("in", lp, host=True), "z": Arg("in", z), "vz": Arg("out", np.zeros(n)), "dvz": Arg("out", np.zeros(n))}
    for q in range(3):
        args["L%d" % q] = Arg("in", Ls[q].ravel(order="F"))
        args["D%d" % q] = Arg("in", dLs[q].ravel(order="F"))

    def call(hd, p, ld):
        pa = (C.c_void_p * 3)(*[p["L%d" % q] for q in range(3)])
        pb = (C.c_void_p * 3)(*[p["D%d" % q] for q in range(3)])
        return hd.lib.gpb200_approx_Lz(hd._h, n, 0.63, 3, p["lp"], pa, pb, p["z"], p["vz"], p["dvz"])

    def oracle(r):
        rv, rd = o.approx_Lz(0.63, lp, Ls, dLs, z)
        return relerr(r["vz"], rv) < 1e-12 and relerr(r["dvz"], rd) < 1e-12
    return args, call, oracle


def case_kernel_eval(n, m=None):
    rng = np.random.default_rng(n)
    tj = rng.uniform(-2, 2, n); tk = rng.uniform(-2, 2, n)
    args = {"tj": Arg("in", tj), "tk": Arg("in", tk), "out": Arg("out", np.zeros(n))}
    call = lambda hd, p, ld: hd.lib.gpb200_kernel_eval(hd._h, capi.KINDS["TT"], n, p["tj"], p["tk"], 1.44, 0.8, p["out"])
    return args, call, lambda r: relerr(r["out"], 1.44 * o.dk_TT(tj, tk, 0.8)) < 1e-13


def case_normal_fill(n, m=None):
    args = {"out": Arg("out", np.zeros(n))}
    call = lambda hd, p, ld: hd.lib.gpb200_normal_fill(hd._h, 1234, 6, n, p["out"])
    # the integer stream bit for bit: test_host_mirror_gpu.py::test_device_normals_match_the_restated_stream
    return args, call, lambda r: relerr(r["out"], philox.normals(1234, n, offset=6)) < 1e-14


def case_lml_grad_batched(n, m=None):
    B = 3
    rng = np.random.default_rng(n)
    X = np.sort(rng.uniform(0, 0.05 * n + 1, (n, B)), axis=0)
    Y = np.sin(X) + 0.3 * rng.standard_normal((n, B))
    th = o.synth_theta(B, n)
    args = {"x": Arg("in", X, True), "y": Arg("in", Y, True), "th": Arg("in", th.ravel()),
            "lml": Arg("out", np.zeros(B)), "grad": Arg("out", np.zeros(3 * B)), "info": Arg("out", np.zeros(B, np.int32))}
    call = lambda hd, p, ld: hd.lib.gpb200_lml_grad_batched(hd._h, n, B, p["x"], ld["x"], p["y"], ld["y"], p["th"], 0.0, 1,
                                                            p["lml"], p["grad"], p["info"])

    def oracle(r):
        assert np.all(r["info"] == 0)
        for b in range(B):
            rv, rg = o.lml_grad(X[:, b], Y[:, b], *th[b])
            assert_lml_close(r["lml"][b], rv, ctx=b)
            assert_grad_close(r["grad"][3 * b:3 * b + 3], rg, ctx=b)
        return True
    return args, call, oracle


def case_lml_grad_deriv_batched(n, m=None):
    B, nb = 3, 2
    rng = np.random.default_rng(n + 1)
    T = np.sort(rng.uniform(0, 0.12 * n + 1, (n, B)), axis=0)
    Y = np.concatenate([np.sin(T), np.cos(T)], axis=0) + 0.2 * rng.standard_normal((2 * n, B))
    th = np.column_stack([rng.uniform(0.7, 1.5, B), rng.uniform(0.8, 1.6, B), rng.uniform(0.1, 0.4, B), rng.uniform(0.1, 0.4, B)])
    args = {"t": Arg("in", T, True), "y": Arg("in", Y, True), "th": Arg("in", th.ravel()),
            "lml": Arg("out", np.zeros(B)), "grad": Arg("out", np.zeros(4 * B)), "info": Arg("out", np.zeros(B, np.int32))}
    call = lambda hd, p, ld: hd.lib.gpb200_lml_grad_deriv_batched(hd._h, n, 0, nb, B, p["t"], ld["t"], p["y"], ld["y"], p["th"],
                                                                  1e-8, 1, p["lml"], p["grad"], p["info"])

    def oracle(r):
        assert np.all(r["info"] == 0)
        for b in range(B):
            rv, rg = o.lml_grad_deriv(T[:, b], Y[:, b], th[b, 0], th[b, 1], th[b, 2:], 1e-8, nb, 0)
            assert_lml_close(r["lml"][b], rv, ctx=b)
            assert_grad_close(r["grad"][4 * b:4 * b + 4], rg, ctx=b)
        return True
    return args, call, oracle


CASES = {k[5:]: v for k, v in globals().items() if k.startswith("case_")}
# the batched LML entry points take strides >= n + 3 (one more than the others' smallest padding)
STRIDE_PADS = {"lml_grad_batched": (3, 37), "lml_grad_deriv_batched": (3, 37)}


@pytest.mark.parametrize("n", [1, 127, 129, 300])
@pytest.mark.parametrize("entry", sorted(CASES))
def test_leading_dimensions_guards_and_pointer_modes(h, entry, n):
    args, call, oracle = CASES[entry](n)
    ref = check_layouts(h, args, call, pads=STRIDE_PADS.get(entry, (1, 37)))
    assert oracle(ref), entry


# automatic GEMM configuration of each entry point's main product (task lists of api_core.cu:365-379,
# api_sample.cu:25-35, api_gp.cu:405-419): 2200 = 18 tiles, 18 x 18 tasks of one item
@pytest.mark.parametrize("entry", ["trsm_lower", "potrs", "mvrnorm", "gp_condition"])
def test_leading_dimensions_on_half_tiles(h, entry):
    n = 2200
    assert gemm_cfg(tiles(n) * tiles(n), 1) == 2
    args, call, oracle = CASES[entry](n, n)
    ref = check_layouts(h, args, call, pads=(1,))
    assert oracle(ref), entry


# ---- B. device mode: the in-place small path and stream ordering ---------------------------------------------
def _strided(rows_by_item, stride):
    """(B, n) items laid out with `stride` doubles between items (0 = the first item shared)."""
    B, n = rows_by_item.shape
    if stride == 0:
        return rows_by_item[0].copy()
    buf = np.full(B * stride, np.nan)
    buf.reshape(B, stride)[:, :n] = rows_by_item
    return buf


def _lml_raw(hd, n, B, x, xs, y, ys, th, want_grad, device, jitter=0.0, stream=None):
    """One gpb200_lml_grad_batched call on host or device buffers; returns numpy (lml, grad, info)."""
    th = np.ascontiguousarray(th, dtype=np.float64)
    if not device:
        lml = np.empty(B); grad = np.empty(3 * B); info = np.zeros(B, np.int32)
        rc = hd.lib.gpb200_lml_grad_batched(hd._h, n, B, x.ctypes.data, xs, y.ctypes.data, ys, th.ctypes.data, jitter,
                                            want_grad, lml.ctypes.data, grad.ctypes.data, info.ctypes.data)
        assert rc == 0, hd.lib.gpb200_last_error(hd._h)
        return lml, grad.reshape(B, 3), info
    dx, dy, dth = (torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (x, y, th))
    lml = torch.empty(B, dtype=torch.float64, device="cuda"); grad = torch.empty(3 * B, dtype=torch.float64, device="cuda")
    info = torch.empty(B, dtype=torch.int32, device="cuda")
    with device_mode(hd, stream):
        rc = hd.lib.gpb200_lml_grad_batched(hd._h, n, B, dx.data_ptr(), xs, dy.data_ptr(), ys, dth.data_ptr(), jitter,
                                            want_grad, lml.data_ptr(), grad.data_ptr(), info.data_ptr())
    assert rc == 0, hd.lib.gpb200_last_error(hd._h)
    torch.cuda.synchronize()
    return lml.cpu().numpy(), grad.cpu().numpy().reshape(B, 3), info.cpu().numpy()


def _sample(B, k=16):
    return sorted(set(np.linspace(0, B - 1, min(B, k)).astype(int).tolist()))


@pytest.mark.parametrize("stride_kind", ["shared", "dense", "padded"])
@pytest.mark.parametrize("n", [1, 33, 128])
def test_small_path_in_place_device_mode(h, n, stride_kind):
    """n <= 128 in device mode: one launch reads x, y, theta and writes lml, grad, info in the caller's arrays."""
    assert small_in_place(n)
    stride = {"shared": 0, "dense": n, "padded": n + 3}[stride_kind]
    for B in (1, 5, 4096):
        rng = np.random.default_rng(n * 7 + B)
        X = np.sort(rng.uniform(0, 0.05 * n + 1, (B, n)), axis=1)
        Y = np.sin(X) + 0.3 * rng.standard_normal((B, n))
        th = o.synth_theta(B, n + B)
        x, y = _strided(X, stride), _strided(Y, stride)
        for want_grad in (0, 1):
            hl, hg, hi = _lml_raw(h, n, B, x, stride, y, stride, th, want_grad, False)
            dl, dg, di = _lml_raw(h, n, B, x, stride, y, stride, th, want_grad, True)
            assert np.array_equal(_bits(hl), _bits(dl)) and np.array_equal(hi, di), (B, want_grad)
            if want_grad:
                assert np.array_equal(_bits(hg), _bits(dg)), B
            assert np.all(di == 0)
            for b in (_sample(B) if B > 5 else range(B)):
                xb, yb = (X[b], Y[b]) if stride else (X[0], Y[0])
                rv, rg = o.lml_grad(xb, yb, *th[b])
                assert_lml_close(dl[b], rv, ctx=(B, want_grad, b))
                if want_grad:
                    assert_grad_close(dg[b], rg, ctx=(B, b))


@pytest.mark.parametrize("n", [100, 300])
def test_lml_grad_device_mode_returns_info(h, n):
    """gpb200_lml_grad in device mode: lml and grad are device pointers, the status (through the handle's info
    slot) is the return value."""
    x, y = o.synth_xy(n, 5)
    th = np.array([1.1, 0.9, 0.3])
    hv, hg = h.lml_grad(x, y, th)
    dx, dy, dth = (torch.from_numpy(a).cuda() for a in (x, y, th))
    lml = torch.empty(1, dtype=torch.float64, device="cuda"); grad = torch.empty(3, dtype=torch.float64, device="cuda")
    with device_mode(h):
        rc = h.lib.gpb200_lml_grad(h._h, n, dx.data_ptr(), dy.data_ptr(), dth.data_ptr(), 0.0, lml.data_ptr(), grad.data_ptr())
        assert rc == 0
        torch.cuda.current_stream().synchronize()
        assert lml.item() == hv and np.array_equal(grad.cpu().numpy(), hg)
        rv, rg = o.lml_grad(x, y, *th)
        assert_lml_close(hv, rv); assert_grad_close(hg, rg)
        xd = torch.from_numpy(np.repeat(np.linspace(0, 1, n // 2), 2)).cuda()   # duplicated inputs, no noise: singular
        th0 = torch.tensor([1.0, 0.5, 0.0], dtype=torch.float64, device="cuda")
        rc = h.lib.gpb200_lml_grad(h._h, n, xd.data_ptr(), dy.data_ptr(), th0.data_ptr(), 0.0, lml.data_ptr(), grad.data_ptr())
    assert rc > 0


def _to_host_on(stream, *tensors):
    """Copies enqueued on `stream` into pinned host memory."""
    outs = []
    with torch.cuda.stream(stream):
        for t in tensors:
            hbuf = torch.empty(t.shape, dtype=t.dtype, pin_memory=True)
            hbuf.copy_(t, non_blocking=True)
            outs.append(hbuf)
    return outs


def _upload_on(stream, a):
    """A device copy of the host array `a`, enqueued on `stream` (pinned staging: no host synchronisation)."""
    with torch.cuda.stream(stream):
        return torch.from_numpy(np.ascontiguousarray(a)).pin_memory().to("cuda", non_blocking=True)


def _lml_on_stream(hd, s, n, B, seed, bind=True):
    """LML + gradient in device mode with the inputs produced on s right before the call; returns the inputs and
    the device outputs, which the caller reads on a stream of its choice.  bind=False: the handle is already in
    device mode on s."""
    x, y = o.synth_xy(n, seed)
    th = o.synth_theta(B, seed)
    src = _upload_on(s, np.concatenate([x, y, th.ravel()]))
    with torch.cuda.stream(s):
        dx = torch.empty(n, dtype=torch.float64, device="cuda"); dy = torch.empty_like(dx)
        dth = torch.empty(3 * B, dtype=torch.float64, device="cuda")
        lml = torch.empty(B, dtype=torch.float64, device="cuda"); grad = torch.empty(3 * B, dtype=torch.float64, device="cuda")
        info = torch.empty(B, dtype=torch.int32, device="cuda")
        dx.copy_(src[:n]); dy.copy_(src[n:2 * n]); dth.copy_(src[2 * n:])
        call = lambda: hd.lib.gpb200_lml_grad_batched(hd._h, n, B, dx.data_ptr(), 0, dy.data_ptr(), 0, dth.data_ptr(), 0.0, 1,
                                                      lml.data_ptr(), grad.data_ptr(), info.data_ptr())
        if bind:
            with device_mode(hd, s):
                rc = call()
        else:
            rc = call()
        assert rc == 0, hd.lib.gpb200_last_error(hd._h)
    return (x, y, th), (lml, grad, info)


def _check_lml_items(inputs, outs, items=None):
    (x, y, th), (lml, grad, info) = inputs, [t.numpy() for t in outs]
    B = th.shape[0]
    assert np.all(info == 0)
    ref = o.lml_grad if x.shape[0] <= 1024 else o.lml_grad_lapack
    for b in (range(B) if items is None else items):
        rv, rg = ref(x, y, *th[b])
        assert_lml_close(lml[b], rv, ctx=b)
        assert_grad_close(grad.reshape(B, 3)[b], rg, ctx=b)
    return lml, grad


@pytest.mark.parametrize("n,B,schedule", [(300, 3, "graph"), (2048, 1, "lookahead_graph"), (4096, 5, "lookahead_eager"),
                                          (1024, 80, "tiled"), (100, 7, "small")])
def test_results_are_ready_after_synchronising_the_callers_stream(h, n, B, schedule):
    expect = {"graph": (True, None), "lookahead_graph": (True, True), "lookahead_eager": (False, True), "tiled": (False, False),
              "small": (False, False)}[schedule]
    assert uses_graph(n, B) == expect[0]
    if expect[1] is not None:
        assert uses_lookahead(n, B) == expect[1]
    if schedule == "small":
        assert small_in_place(n)
    s = torch.cuda.Stream()
    inputs, outs = _lml_on_stream(h, s, n, B, 31)
    outs = _to_host_on(s, *outs)
    if schedule == "graph":   # the second call replays the graph the first one captured
        before = h.graph_replays()
        inputs2, outs2 = _lml_on_stream(h, s, n, B, 32)
        outs2 = _to_host_on(s, *outs2)
    s.synchronize()
    items = None if B <= 8 else _sample(B, 8)
    lml, grad = _check_lml_items(inputs, outs, items)
    if schedule == "graph":
        assert h.graph_replays() == before + 1
        _check_lml_items(inputs2, outs2)
    if schedule == "tiled":   # every item: bit-identical to the host-mode call (same schedule)
        x, y, th = inputs
        hl, hg, _ = h.lml_grad_batched(x, y, th)
        assert np.array_equal(hl, lml) and np.array_equal(hg.ravel(), grad)


def test_potrf_and_gp_condition_on_the_callers_stream(h):
    n, m = 300, 200
    K = _spd(n, 3)
    args, _, _ = case_gp_condition(n, m)
    Kc, Ks, Kss = (args[k].data for k in ("K", "Ks", "Kss"))
    y = args["y"].data[:, 0]
    s = torch.cuda.Stream()
    # column-major device copies (a row-major tensor of A^T); K, Kc and Kss are symmetric
    dA, dK, dKs, dKss, dy = (_upload_on(s, a) for a in (K, Kc, Ks.T, Kss, y))
    with torch.cuda.stream(s):
        mu = torch.empty(m, dtype=torch.float64, device="cuda"); cov = torch.empty((m, m), dtype=torch.float64, device="cuda")
        with device_mode(h, s):
            assert h.lib.gpb200_potrf(h._h, n, dA.data_ptr(), n) == 0
            assert h.lib.gpb200_gp_condition(h._h, n, m, dK.data_ptr(), n, dKs.data_ptr(), m, dKss.data_ptr(), m, dy.data_ptr(),
                                             0.04, 1e-8, mu.data_ptr(), cov.data_ptr(), m) == 0
    A, hm, hc = _to_host_on(s, dA, mu, cov)
    s.synchronize()
    assert relerr(A.numpy().T, o.cholesky_decompose(K)) < 1e-9
    rmu, rcov = o.gp_condition(Kc, Ks, Kss, y, 0.04, 1e-8)
    assert relerr(hm.numpy(), rmu) < 1e-8 and relerr(hc.numpy().T, rcov) < 1e-8


def test_set_stream_orders_the_new_stream_after_the_old_one(h):
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    with device_mode(h, s1):
        big_in, big_out = _lml_on_stream(h, s1, 4096, 5, 41, bind=False)     # eager look-ahead: still running below
        h.set_stream(s2.cuda_stream)                                          # the edge under test
        small_in, small_out = _lml_on_stream(h, s2, 1000, 3, 42, bind=False)  # reuses the same workspace
    big_out = _to_host_on(s2, *big_out)
    small_out = _to_host_on(s2, *small_out)
    s2.synchronize()
    _check_lml_items(small_in, small_out)
    _check_lml_items(big_in, big_out)


def test_workspace_growth_without_host_synchronisation(h):
    """Device-mode calls of growing size on one stream: each one frees and reallocates the workspace and drops the
    cached graphs (engine.cu:13-31); the caller synchronises once, at the end."""
    h2 = capi.Handle(0)
    try:
        s = torch.cuda.Stream()
        pending = []
        with device_mode(h2, s):
            for n, B in ((300, 3), (1000, 4), (2000, 2), (300, 3)):
                inputs, outs = _lml_on_stream(h2, s, n, B, n + B, bind=False)
                pending.append((inputs, _to_host_on(s, *outs)))
            K = _spd(2500, 2, 0.2)
            dA = _upload_on(s, K)
            assert h2.lib.gpb200_potrf(h2._h, 2500, dA.data_ptr(), 2500) == 0
        (A,) = _to_host_on(s, dA)
        s.synchronize()
        for inputs, outs in pending:
            _check_lml_items(inputs, outs)
        assert relerr(A.numpy().T, o.cholesky_decompose(K)) < 1e-9
    finally:
        h2.close()


def test_chunking_in_device_mode_with_strided_items(h):
    n, B, stride = 300, 200, 303
    rng = np.random.default_rng(9)
    X = np.sort(rng.uniform(0, 15, (B, n)), axis=1)
    Y = np.sin(X) + 0.3 * rng.standard_normal((B, n))
    th = o.synth_theta(B, 9)
    x, y = _strided(X, stride), _strided(Y, stride)
    limit = limit_for_chunk(n, B, 80, x_per_item=True, y_per_item=True)
    ref = _lml_raw(h, n, B, x, stride, y, stride, th, 1, True)
    try:
        h.set_workspace_limit(limit)
        dev = _lml_raw(h, n, B, x, stride, y, stride, th, 1, True)
        host = _lml_raw(h, n, B, x, stride, y, stride, th, 1, False)
    finally:
        h.set_workspace_limit(0)
    for a, b in zip(dev, host):   # same chunks, same schedule
        assert np.array_equal(_bits(a), _bits(b))
    # chunks of 80 and 40 take other GEMM configurations than the 200-item batch: equal to rounding
    assert np.array_equal(dev[2], ref[2]) and np.all(dev[2] == 0)
    assert np.allclose(dev[0], ref[0], rtol=1e-12, atol=0) and relerr(dev[1], ref[1]) < 1e-10
    for b in _sample(B, 6):
        rv, rg = o.lml_grad(X[b], Y[b], *th[b])
        assert_lml_close(dev[0][b], rv, ctx=b); assert_grad_close(dev[1][b], rg, ctx=b)


# ---- C. LML-only batches: the blocked forward substitution -------------------------------------------------
def _se_batch(n, B, per_item, seed):
    rng = np.random.default_rng(seed)
    if per_item:
        X = np.sort(rng.uniform(0, 0.05 * n, (B, n)), axis=1)
        Y = np.sin(X) + 0.5 * np.sin(3.1 * X) + 0.3 * rng.standard_normal((B, n))
        return X, Y, X, Y
    x, y = o.synth_xy(n, seed)
    return x, y, np.broadcast_to(x, (B, n)), np.broadcast_to(y, (B, n))


@pytest.mark.parametrize("per_item", [False, True])
@pytest.mark.parametrize("n,B", [(129, 32), (300, 33), (1000, 64), (2100, 40)])
def test_lml_only_batches_take_the_blocked_substitution(h, n, B, per_item):
    assert uses_trsv_blocked(B)
    x, y, X, Y = _se_batch(n, B, per_item, n + B)
    th = o.synth_theta(B, n)
    lml, _, info = h.lml_grad_batched(x, y, th, want_grad=False)
    lml2, _, info2 = h.lml_grad_batched(x, y, th)
    assert np.all(info == 0) and np.array_equal(info, info2)
    for b in range(B):
        assert_lml_close(lml[b], o.lml(X[b], Y[b], *th[b]), ctx=b)
        assert abs(lml[b] - lml2[b]) <= 1e-12 * abs(lml2[b]), b


def test_lml_only_chunks_take_both_substitution_kernels(h):
    n, B = 300, 40
    x, y = o.synth_xy(n, 4)
    th = o.synth_theta(B, 4)
    limit = limit_for_chunk(n, B, 32)
    assert uses_trsv_blocked(32) and not uses_trsv_blocked(B - 32)
    lml2, _, _ = h.lml_grad_batched(x, y, th)
    try:
        h.set_workspace_limit(limit)
        lml, _, info = h.lml_grad_batched(x, y, th, want_grad=False)
    finally:
        h.set_workspace_limit(0)
    assert np.all(info == 0)
    for b in range(B):
        assert_lml_close(lml[b], o.lml(x, y, *th[b]), ctx=b)
        assert abs(lml[b] - lml2[b]) <= 1e-12 * abs(lml2[b]), b


def test_lml_only_batch_reports_a_singular_item_and_keeps_its_neighbours(h):
    n, B, bad = 300, 33, 7
    _, _, X, Y = _se_batch(n, B, True, 3)
    X = X.copy()
    X[bad] = np.repeat(np.linspace(0, 10, n // 2), 2)   # duplicated inputs and sigma = 0: singular
    th = o.synth_theta(B, 3)
    th[bad, 2] = 0.0
    assert uses_trsv_blocked(B)
    lml, _, info = h.lml_grad_batched(X, Y, th, want_grad=False)
    assert info[bad] > 0
    for b in range(B):
        if b != bad:
            assert info[b] == 0
            assert_lml_close(lml[b], o.lml(X[b], Y[b], *th[b]), ctx=b)


def _deriv_batch(ng, order0, nblocks, B, per_item, seed):
    rng = np.random.default_rng(seed)
    T = np.sort(rng.uniform(0, 0.12 * ng, (B if per_item else 1, ng)), axis=1)
    truth = lambda t: [np.sin(t), np.cos(t), -np.sin(t)][order0:order0 + nblocks]
    Y = np.stack([np.concatenate(truth(t)) for t in T]) + 0.2 * rng.standard_normal((T.shape[0], ng * nblocks))
    th = np.column_stack([rng.uniform(0.7, 1.5, B), rng.uniform(0.8, 1.6, B)] + [rng.uniform(0.1, 0.4, B) for _ in range(nblocks)])
    t, y = (T, Y) if per_item else (T[0], Y[0])
    return t, y, np.broadcast_to(T, (B, ng)), np.broadcast_to(Y, (B, ng * nblocks)), th


@pytest.mark.parametrize("ng,order0,nblocks,B", [(100, 0, 3, 40), (129, 1, 2, 32)])
def test_lml_only_derivative_batches(h, ng, order0, nblocks, B):
    assert uses_trsv_blocked(B)
    t, y, T, Y, th = _deriv_batch(ng, order0, nblocks, B, False, ng)
    lml, _, info = h.lml_grad_deriv_batched(t, y, th, 1e-8, order0=order0, nblocks=nblocks, want_grad=False)
    lml2, _, _ = h.lml_grad_deriv_batched(t, y, th, 1e-8, order0=order0, nblocks=nblocks)
    assert np.all(info == 0)
    for b in range(B):
        rv, _ = o.lml_grad_deriv(T[b], Y[b], th[b, 0], th[b, 1], th[b, 2:], 1e-8, nblocks, order0)
        assert_lml_close(lml[b], rv, ctx=b)
        assert abs(lml[b] - lml2[b]) <= 1e-12 * abs(lml2[b]), b


# ---- D. derivative-observation LML + gradient on half tiles and under the diagonal split ----------------------
@pytest.mark.parametrize("ng,order0,nblocks,B,per_item", [
    (70, 1, 2, 120, False),    # 140 x 140: half tiles, no split
    (100, 0, 3, 400, False),   # 300: split
    (100, 0, 3, 400, True),    # the same with per-item grids and observations
    (300, 0, 3, 64, False),    # 900: split, block boundaries 300 and 600 inside (diagonal) tiles
    (512, 0, 3, 32, False),    # C2 shape, 1536: split, block boundaries on tile edges
])
def test_derivative_lml_grad_on_half_tiles_and_diagonal_split(h, monkeypatch, ng, order0, nblocks, B, per_item):
    ntasks = lauum_tasks(tiles(ng * nblocks))
    assert gemm_cfg(ntasks, B) == 2
    split = diag_split(ntasks, B)
    assert split == (B != 120)
    t, y, T, Y, th = _deriv_batch(ng, order0, nblocks, B, per_item, ng + B)
    lml, grad, info = h.lml_grad_deriv_batched(t, y, th, 1e-8, order0=order0, nblocks=nblocks)
    assert np.all(info == 0)
    for b in range(B):
        rv, rg = o.lml_grad_deriv(T[b], Y[b], th[b, 0], th[b, 1], th[b, 2:], 1e-8, nblocks, order0)
        assert_lml_close(lml[b], rv, ctx=b)
        assert_grad_close(grad[b], rg, ctx=b)
    monkeypatch.setenv("GPB200_DIAG_SPLIT", "0")
    h2 = capi.Handle(0)
    try:
        lml2, grad2, info2 = h2.lml_grad_deriv_batched(t, y, th, 1e-8, order0=order0, nblocks=nblocks)
    finally:
        h2.close()
    # the split changes the summation order of the trace partials only
    assert np.array_equal(info, info2)
    assert np.all(np.abs(lml - lml2) <= 1e-12 * np.abs(lml2))
    for b in range(B):
        assert relerr(grad[b], grad2[b]) < 1e-10, b
