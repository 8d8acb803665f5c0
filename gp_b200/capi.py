"""ctypes binding of libgpb200.so (the C ABI declared in include/gpb200.h).

This is the only way Python reaches the GPU code.  There is no CPU fallback: if the shared library
is missing, or no sm_100 GPU is present, the calls raise.  NumPy arrays go through the host-pointer
mode of the ABI (exactly what R's .Call shim does); torch CUDA tensors go through the
device-pointer mode (used by bench.py for the HBM-resident measurement).
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("GPB200_LIB", os.path.join(_HERE, "lib", "libgpb200.so"))

KINDS = {"QQ": 0, "QR": 1, "RQ": 2, "RR": 3, "QT": 4, "TQ": 5, "RT": 6, "TR": 7, "TT": 8, "RR_QUIRK": 9}

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int)
_h = C.c_void_p
_ll = C.c_longlong

# name -> (restype, argtypes); mirrors include/gpb200.h one to one
SIGNATURES = {
    "gpb200_create": (C.c_int, [C.POINTER(_h), C.c_int]),
    "gpb200_destroy": (C.c_int, [_h]),
    "gpb200_set_stream": (C.c_int, [_h, C.c_void_p]),
    "gpb200_set_stream_unordered": (C.c_int, [_h, C.c_void_p]),
    "gpb200_set_pointer_mode": (C.c_int, [_h, C.c_int]),
    "gpb200_synchronize": (C.c_int, [_h]),
    "gpb200_last_error": (C.c_char_p, [_h]),
    "gpb200_launch_count": (_ll, [_h]),
    "gpb200_version": (C.c_int, []),
    "gpb200_set_workspace_limit": (C.c_int, [_h, _ll]),
    "gpb200_graph_replays": (_ll, [_h]),
    "gpb200_set_chol_panel_tiles": (C.c_int, [_h, C.c_int]),
    "gpb200_set_gemm_config": (C.c_int, [_h, C.c_int]),
    "gpb200_set_profiling": (C.c_int, [_h, C.c_int]),
    "gpb200_get_profile": (C.c_int, [_h, C.c_void_p, C.c_void_p]),
    "gpb200_set_flop_counting": (C.c_int, [_h, C.c_int]),
    "gpb200_executed_gemm_flops": (C.c_double, [_h]),
    "gpb200_debug_bench_panel": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]),
    "gpb200_debug_panel_trace": (C.c_int, [_h, C.c_void_p]),
    "gpb200_kernel_eval": (C.c_int, [_h, C.c_int, _ll, C.c_void_p, C.c_void_p, C.c_double, C.c_double, C.c_void_p]),
    "gpb200_gram_outer": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_double, C.c_double,
                                    C.c_void_p, C.c_int]),
    "gpb200_gram_ard": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_double,
                                  C.c_void_p, C.c_void_p, C.c_int]),
    "gpb200_gram_se": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_void_p, C.c_int]),
    "gpb200_gram_deriv": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_double,
                                    C.c_int, C.c_void_p, C.c_int]),
    "gpb200_approx_L_basis": (C.c_int, [_h, C.c_int, C.c_int, C.c_double, C.c_void_p, C.c_double, C.c_double, C.c_void_p,
                                        C.c_int]),
    "gpb200_potrf": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_int]),
    "gpb200_trsm_lower": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "gpb200_potrs": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int]),
    "gpb200_trmv_lower": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "gpb200_trmv_lower_t": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]),
    "gpb200_mvn_chol_lpdf": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "gpb200_lml_grad": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "gpb200_lml_grad_batched": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p, _ll, C.c_void_p,
                                          C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_lml_grad_deriv_batched": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p, _ll,
                                                C.c_void_p, C.c_double, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_rbf_cov_chol": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "gpb200_rbf_cov_chol_batched": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p,
                                              C.c_void_p]),
    "gpb200_se_chol_tangent": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_int,
                                         C.c_void_p, C.c_void_p]),
    "gpb200_latent_forward": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_void_p, C.c_void_p]),
    "gpb200_latent_backward": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_void_p,
                                         C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_approx_L": (C.c_int, [_h, C.c_int, C.c_double, C.c_int, C.c_void_p, C.POINTER(C.c_void_p),
                                  C.POINTER(C.c_void_p), C.c_void_p]),
    "gpb200_approx_Lz": (C.c_int, [_h, C.c_int, C.c_double, C.c_int, C.c_void_p, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_void_p), C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_gp_condition": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_void_p,
                                      C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_void_p, C.c_void_p, C.c_int]),
    "gpb200_cond_mvn": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                  C.c_void_p, C.c_int]),
    "gpb200_normal_fill": (C.c_int, [_h, C.c_ulonglong, C.c_ulonglong, _ll, C.c_void_p]),
    "gpb200_mvrnorm": (C.c_int, [_h, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_ulonglong,
                                 C.c_void_p, C.c_int]),
    "gpb200_posterior_draws_batched": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p, _ll,
                                                 C.c_void_p, _ll, C.c_void_p, C.c_double, C.c_void_p, C.c_ulonglong,
                                                 C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_mg_gram_panel": (C.c_int, [_h, C.c_int, C.c_void_p, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                                       C.c_void_p, _ll]),
    "gpb200_mg_panel_factor": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p]),
    "gpb200_mg_panel_factor_col": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_int, C.c_void_p]),
    "gpb200_mg_panel_update": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_int, C.c_int, C.c_void_p,
                                         _ll]),
    "gpb200_mg_panel_update_cols": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_int, C.c_int, C.c_void_p,
                                              _ll, C.c_int, C.c_int]),
    "gpb200_mg_panel_trsv": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p]),
    "gpb200_mg_comm_id": (C.c_int, [_h, C.c_void_p]),
    "gpb200_mg_comm_init": (C.c_int, [_h, C.c_void_p, C.c_int, C.c_int]),
    "gpb200_mg_comm_destroy": (C.c_int, [_h]),
    "gpb200_mg_bcast": (C.c_int, [_h, C.c_void_p, _ll, C.c_int, C.POINTER(_ll)]),
    "gpb200_mg_wait": (C.c_int, [_h, _ll]),
    "gpb200_mg_allreduce": (C.c_int, [_h, C.c_void_p, _ll, C.c_int, C.c_int]),
    "gpb200_mg_panel_to_square": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p]),
    "gpb200_mg_my_columns": (_ll, [C.c_int, C.c_int, C.c_int, C.c_int]),
    "gpb200_mg_inverse_rows": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_mg_solve_partials": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_mg_trace_partials": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                           C.c_void_p, C.c_void_p]),
    "gpb200_mg_quadform_partials": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "gpb200_mg_panel_logdiag": (C.c_int, [_h, C.c_int, C.c_int, C.c_int, C.c_void_p, _ll, C.c_void_p]),
}

_lib = None


class GpB200Error(RuntimeError):
    pass


class NotPositiveDefiniteError(GpB200Error):
    """Raised where Stan Math's cholesky_decompose throws std::domain_error; .info is the 1-based
    index of the first non-positive pivot."""

    def __init__(self, where, info):
        super().__init__("%s: matrix is not positive definite (first non-positive pivot at %d)" % (where, info))
        self.info = info


def load():
    """Load libgpb200.so and bind every symbol of include/gpb200.h.  Raises if it is missing."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise GpB200Error("libgpb200.so not built (%s); run `python -c 'import __graft_entry__ as g; g.build()'`. "
                              "There is no CPU fallback." % LIB_PATH)
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(lib, name)  # AttributeError if the symbol is missing
            f.restype = res
            f.argtypes = args
        _lib = lib
    return _lib


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    return a.data_ptr()  # torch tensor


def _f(a):
    """float64 column-major (Fortran) copy/view of a host array."""
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


class Handle:
    """One handle per GPU (include/gpb200.h: gpb200_create)."""

    def __init__(self, device: int = 0):
        self.lib = load()
        self._h = _h()
        rc = self.lib.gpb200_create(C.byref(self._h), int(device))
        if rc != 0:
            raise GpB200Error("gpb200_create(device=%d) failed with %d: no usable sm_100 GPU (there is no CPU "
                              "fallback)" % (device, rc))
        self.device = device
        self.device_pointers = False

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self.lib.gpb200_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing -------------------------------------------------------------------------------
    def _check(self, rc, where, allow_info=False):
        if rc < 0:
            msg = self.lib.gpb200_last_error(self._h)
            raise GpB200Error("%s failed (%d): %s" % (where, rc, msg.decode() if msg else ""))
        if rc > 0 and not allow_info:
            raise NotPositiveDefiniteError(where, rc)
        return rc

    def set_stream(self, cuda_stream_ptr, ordered=True):
        """ordered=False: no edge from the old stream to the new one (the caller orders with its own events)"""
        f = self.lib.gpb200_set_stream if ordered else self.lib.gpb200_set_stream_unordered
        self._check(f(self._h, C.c_void_p(cuda_stream_ptr)), "set_stream")

    def set_pointer_mode(self, device: bool):
        self._check(self.lib.gpb200_set_pointer_mode(self._h, int(bool(device))), "set_pointer_mode")
        self.device_pointers = bool(device)

    def set_workspace_limit(self, nbytes: int):
        self._check(self.lib.gpb200_set_workspace_limit(self._h, int(nbytes)), "set_workspace_limit")

    def synchronize(self):
        self._check(self.lib.gpb200_synchronize(self._h), "synchronize")

    def launch_count(self) -> int:
        return int(self.lib.gpb200_launch_count(self._h))

    PROFILE_CLASSES = ("gemm", "potrf_tile", "trsm_tile", "gram", "solve", "other")

    def graph_replays(self) -> int:
        return int(self.lib.gpb200_graph_replays(self._h))

    def set_chol_panel_tiles(self, tiles: int):
        self._check(self.lib.gpb200_set_chol_panel_tiles(self._h, int(tiles)), "set_chol_panel_tiles")

    def set_gemm_config(self, cfg: int):
        self._check(self.lib.gpb200_set_gemm_config(self._h, int(cfg)), "set_gemm_config")

    def set_profiling(self, on: bool):
        self._check(self.lib.gpb200_set_profiling(self._h, int(bool(on))), "set_profiling")

    def debug_bench_panel(self, what, nt, batch, reps=5):
        """Mean device time (ms) of one panel kernel launch: what 0 POTRF tile, 1 TRSM tiles, 2 tile inverses."""
        ms = np.zeros(1)
        self._check(self.lib.gpb200_debug_bench_panel(self._h, int(what), int(nt), int(batch), int(reps), _ptr(ms)),
                    "debug_bench_panel")
        return float(ms[0])

    def get_profile(self):
        ms = np.zeros(6); cnt = np.zeros(6, dtype=np.int64)
        self._check(self.lib.gpb200_get_profile(self._h, _ptr(ms), _ptr(cnt)), "get_profile")
        return {k: (float(ms[i]), int(cnt[i])) for i, k in enumerate(self.PROFILE_CLASSES)}

    # -- a9 -------------------------------------------------------------------------------------
    def kernel_eval(self, kind, tj, tk, l, amp2=1.0):
        tj = np.asarray(tj, dtype=np.float64)
        tk = np.asarray(tk, dtype=np.float64)
        tj, tk = np.broadcast_arrays(tj, tk)
        shape = tj.shape
        a = np.ascontiguousarray(tj).ravel()
        b = np.ascontiguousarray(tk).ravel()
        out = np.empty(a.shape[0])
        self._check(self.lib.gpb200_kernel_eval(self._h, KINDS[kind] if isinstance(kind, str) else kind, a.shape[0],
                                                _ptr(a), _ptr(b), amp2, l, _ptr(out)), "kernel_eval")
        return out.reshape(shape)

    def gram_outer(self, kind, x, y, l, amp2=1.0):
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        y = np.ascontiguousarray(y, dtype=np.float64).ravel()
        n, m = x.shape[0], y.shape[0]
        K = np.empty((n, m), order="F")
        self._check(self.lib.gpb200_gram_outer(self._h, KINDS[kind] if isinstance(kind, str) else kind, n, m, _ptr(x),
                                               _ptr(y), amp2, l, _ptr(K), max(n, 1)), "gram_outer")
        return K

    def gram_ard(self, X, Y, alpha, rho):
        X = _f(np.atleast_2d(X)); Y = _f(np.atleast_2d(Y))
        n, D = X.shape
        m = Y.shape[0]
        rho = np.ascontiguousarray(np.broadcast_to(np.asarray(rho, dtype=np.float64), (D,)))
        K = np.empty((n, m), order="F")
        self._check(self.lib.gpb200_gram_ard(self._h, n, m, D, _ptr(X), max(n, 1), _ptr(Y), max(m, 1), alpha, _ptr(rho),
                                             _ptr(K), max(n, 1)), "gram_ard")
        return K

    def gram_se(self, x, alpha, rho, diag_add=0.0):
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        n = x.shape[0]
        K = np.empty((n, n), order="F")
        self._check(self.lib.gpb200_gram_se(self._h, n, _ptr(x), alpha, rho, diag_add, _ptr(K), max(n, 1)), "gram_se")
        return K

    def gram_deriv(self, t, alpha, rho, noise, jitter=0.0, nblocks=3, quirk=False):
        t = np.ascontiguousarray(t, dtype=np.float64).ravel()
        n = t.shape[0]
        noise = np.ascontiguousarray(np.asarray(noise, dtype=np.float64).ravel()[:nblocks])
        N = n * nblocks
        K = np.empty((N, N), order="F")
        self._check(self.lib.gpb200_gram_deriv(self._h, n, _ptr(t), alpha, rho, nblocks, _ptr(noise), jitter,
                                               int(quirk), _ptr(K), max(N, 1)), "gram_deriv")
        return K

    def approx_L_basis(self, M, scale, x, sigma, l):
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        n = x.shape[0]
        out = np.empty((n, M), order="F")
        self._check(self.lib.gpb200_approx_L_basis(self._h, n, int(M), scale, _ptr(x), sigma, l, _ptr(out), max(n, 1)),
                    "approx_L_basis")
        return out

    # -- a6-a8 ----------------------------------------------------------------------------------
    def potrf(self, A, raise_on_info=True):
        A = np.array(A, dtype=np.float64, order="F", copy=True)
        n = A.shape[0]
        rc = self._check(self.lib.gpb200_potrf(self._h, n, _ptr(A), max(n, 1)), "potrf", allow_info=not raise_on_info)
        return A if raise_on_info else (A, rc)

    def trsm_lower(self, L, B):
        L = _f(L); B = np.array(B, dtype=np.float64, order="F", copy=True)
        vec = B.ndim == 1
        B2 = B.reshape(-1, 1, order="F") if vec else B
        n, nrhs = B2.shape
        self._check(self.lib.gpb200_trsm_lower(self._h, n, nrhs, _ptr(L), max(n, 1), _ptr(B2), max(n, 1)), "trsm_lower")
        return B2.ravel(order="F") if vec else B2

    def potrs(self, L, B):
        L = _f(L); B = np.array(B, dtype=np.float64, order="F", copy=True)
        vec = B.ndim == 1
        B2 = B.reshape(-1, 1, order="F") if vec else B
        n, nrhs = B2.shape
        self._check(self.lib.gpb200_potrs(self._h, n, nrhs, _ptr(L), max(n, 1), _ptr(B2), max(n, 1)), "potrs")
        return B2.ravel(order="F") if vec else B2

    def trmv_lower(self, L, z):
        L = _f(L); z = np.ascontiguousarray(z, dtype=np.float64)
        n = z.shape[0]
        f = np.empty(n)
        self._check(self.lib.gpb200_trmv_lower(self._h, n, _ptr(L), max(n, 1), _ptr(z), _ptr(f)), "trmv_lower")
        return f

    def trmv_lower_t(self, L, z):
        L = _f(L); z = np.ascontiguousarray(z, dtype=np.float64)
        n = z.shape[0]
        f = np.empty(n)
        self._check(self.lib.gpb200_trmv_lower_t(self._h, n, _ptr(L), max(n, 1), _ptr(z), _ptr(f)), "trmv_lower_t")
        return f

    def mvn_chol_lpdf(self, y, mu, L, drop_constants=False):
        L = _f(L); y = np.ascontiguousarray(y, dtype=np.float64)
        n = y.shape[0]
        mu_a = None if mu is None else np.ascontiguousarray(np.broadcast_to(np.asarray(mu, dtype=np.float64), (n,)))
        lp = C.c_double()
        self._check(self.lib.gpb200_mvn_chol_lpdf(self._h, n, _ptr(y), _ptr(mu_a), _ptr(L), max(n, 1),
                                                  int(drop_constants), C.addressof(lp)), "mvn_chol_lpdf")
        return lp.value

    # -- CS-A -----------------------------------------------------------------------------------
    def lml_grad(self, x, y, theta, jitter=0.0, want_grad=True):
        x = np.ascontiguousarray(x, dtype=np.float64); y = np.ascontiguousarray(y, dtype=np.float64)
        th = np.ascontiguousarray(theta, dtype=np.float64)
        lml = C.c_double()
        g = np.empty(3)
        self._check(self.lib.gpb200_lml_grad(self._h, x.shape[0], _ptr(x), _ptr(y), _ptr(th), jitter,
                                             C.addressof(lml), _ptr(g) if want_grad else None), "lml_grad")
        return (lml.value, g) if want_grad else lml.value

    def lml_grad_batched(self, x, y, theta, jitter=0.0, want_grad=True):
        """x, y: (n,) shared or (B, n) per item; theta (B, 3).  Returns lml[B], grad[B,3], info[B]."""
        th = np.ascontiguousarray(theta, dtype=np.float64)
        B = th.shape[0]
        x = np.ascontiguousarray(x, dtype=np.float64); y = np.ascontiguousarray(y, dtype=np.float64)
        n = x.shape[-1]
        xs = n if x.ndim == 2 else 0
        ys = n if y.ndim == 2 else 0
        lml = np.empty(B); grad = np.empty((B, 3)); info = np.zeros(B, dtype=np.int32)
        self._check(self.lib.gpb200_lml_grad_batched(self._h, n, B, _ptr(x), xs, _ptr(y), ys, _ptr(th), jitter,
                                                     int(want_grad), _ptr(lml), _ptr(grad), _ptr(info)),
                    "lml_grad_batched")
        return lml, grad, info

    def lml_grad_batched_device(self, n, B, x, x_stride, y, y_stride, theta, jitter, want_grad, lml, grad, info):
        """Device-pointer variant: every array argument is a torch CUDA tensor (float64 / int32); the
        handle must be in device-pointer mode.  Asynchronous on the handle's stream."""
        assert self.device_pointers
        self._check(self.lib.gpb200_lml_grad_batched(self._h, n, B, _ptr(x), x_stride, _ptr(y), y_stride, _ptr(theta),
                                                     jitter, int(want_grad), _ptr(lml), _ptr(grad), _ptr(info)),
                    "lml_grad_batched")

    def lml_grad_deriv_batched(self, t, y, theta, jitter=0.0, order0=0, nblocks=None, want_grad=True):
        """GP observed through derivative orders order0 .. order0+nblocks-1 on the grid t.
        t: (n,) shared or (B, n); y: (n*nblocks,) or (B, n*nblocks), blocks stacked by order;
        theta: (B, 2+nblocks) = (alpha, rho, noise[nblocks]).  Returns lml[B], grad[B, 2+nblocks], info[B]."""
        th = np.ascontiguousarray(theta, dtype=np.float64)
        B = th.shape[0]
        if nblocks is None:
            nblocks = th.shape[1] - 2
        if th.ndim != 2 or th.shape[1] != 2 + nblocks:
            raise ValueError("theta must be (B, 2 + nblocks)")
        t = np.ascontiguousarray(t, dtype=np.float64); y = np.ascontiguousarray(y, dtype=np.float64)
        n = t.shape[-1]
        if y.shape[-1] != n * nblocks:
            raise ValueError("y must hold n * nblocks stacked observations")
        t_s = n if t.ndim == 2 else 0
        y_s = n * nblocks if y.ndim == 2 else 0
        lml = np.empty(B); grad = np.empty((B, 2 + nblocks)); info = np.zeros(B, dtype=np.int32)
        self._check(self.lib.gpb200_lml_grad_deriv_batched(self._h, n, order0, nblocks, B, _ptr(t), t_s, _ptr(y), y_s,
                                                           _ptr(th), jitter, int(want_grad), _ptr(lml), _ptr(grad),
                                                           _ptr(info)), "lml_grad_deriv_batched")
        return lml, grad, info

    # -- a1-a3 / f-1 ----------------------------------------------------------------------------
    def rbf_cov_chol(self, x1, l):
        x1 = np.ascontiguousarray(x1, dtype=np.float64).ravel()
        n = x1.shape[0]
        L = np.empty((n, n), order="F"); dL = np.empty((n, n), order="F")
        self._check(self.lib.gpb200_rbf_cov_chol(self._h, n, _ptr(x1), l, _ptr(L), _ptr(dL)), "rbf_cov_chol")
        return L, dL

    def rbf_cov_chol_batched(self, x1, ls):
        """Tables for approx_L: returns (Ls, dLdls) as arrays of shape (P, n, n) [each slice column-major]."""
        x1 = np.ascontiguousarray(x1, dtype=np.float64).ravel()
        ls = np.ascontiguousarray(ls, dtype=np.float64).ravel()
        n, P = x1.shape[0], ls.shape[0]
        L = np.empty((P, n, n)); dL = np.empty((P, n, n)); info = np.zeros(P, dtype=np.int32)
        self._check(self.lib.gpb200_rbf_cov_chol_batched(self._h, n, _ptr(x1), P, _ptr(ls), _ptr(L), _ptr(dL),
                                                         _ptr(info)), "rbf_cov_chol_batched")
        if np.any(info > 0):
            raise NotPositiveDefiniteError("rbf_cov_chol_batched", int(info[info > 0][0]))
        # each slice was written column-major: expose as Fortran-ordered matrices
        return [L[q].T.copy(order="F") for q in range(P)], [dL[q].T.copy(order="F") for q in range(P)]

    def se_chol_tangent(self, x, alpha, rho, diag_add, wrt):
        """L = chol(cov_exp_quad(x, alpha, rho) + diag_add I) and dL/d(alpha if wrt == 0 else rho)."""
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        n = x.shape[0]
        L = np.empty((n, n), order="F"); dL = np.empty((n, n), order="F")
        self._check(self.lib.gpb200_se_chol_tangent(self._h, n, _ptr(x), alpha, rho, diag_add, int(wrt), _ptr(L),
                                                    _ptr(dL)), "se_chol_tangent")
        return L, dL

    def latent_forward(self, x, alpha, rho, diag_add, z):
        """f = L z (z: (n,) or (nvec, n)) with L = chol(cov_exp_quad(x, alpha, rho) + diag_add I); L stays on the device."""
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        z2 = np.ascontiguousarray(np.atleast_2d(np.asarray(z, dtype=np.float64)))
        n, nvec = x.shape[0], z2.shape[0]
        f = np.empty((nvec, n))
        self._check(self.lib.gpb200_latent_forward(self._h, n, _ptr(x), alpha, rho, diag_add, nvec, _ptr(z2), _ptr(f)), "latent_forward")
        return f[0] if np.ndim(z) == 1 else f

    def latent_backward(self, x, alpha, rho, diag_add, z, fbar):
        """Reverse sweep through f = L z and the Cholesky: returns ((d/dalpha, d/drho), zbar)."""
        x = np.ascontiguousarray(x, dtype=np.float64).ravel()
        z2 = np.ascontiguousarray(np.atleast_2d(np.asarray(z, dtype=np.float64)))
        fb = np.ascontiguousarray(np.atleast_2d(np.asarray(fbar, dtype=np.float64)))
        n, nvec = x.shape[0], z2.shape[0]
        tb = np.empty(2); zbar = np.empty((nvec, n))
        self._check(self.lib.gpb200_latent_backward(self._h, n, _ptr(x), alpha, rho, diag_add, nvec, _ptr(z2), _ptr(fb), _ptr(tb),
                                                    _ptr(zbar)), "latent_backward")
        return tb, (zbar[0] if np.ndim(z) == 1 else zbar)

    def _tables(self, Ls, dLdls):
        Ls = [_f(a) for a in Ls]; dLs = [_f(a) for a in dLdls]
        P = len(Ls)
        pa = (C.c_void_p * P)(*[a.ctypes.data for a in Ls])
        pb = (C.c_void_p * P)(*[a.ctypes.data for a in dLs])
        return Ls, dLs, pa, pb, P

    def approx_L(self, l, lp, Ls, dLdls):
        Ls, dLs, pa, pb, P = self._tables(Ls, dLdls)
        lp = np.ascontiguousarray(lp, dtype=np.float64)
        n = Ls[0].shape[0]
        out = np.empty((n, n), order="F")
        self._check(self.lib.gpb200_approx_L(self._h, n, l, P, _ptr(lp), pa, pb, _ptr(out)), "approx_L")
        return out

    def approx_Lz(self, l, lp, Ls, dLdls, z):
        Ls, dLs, pa, pb, P = self._tables(Ls, dLdls)
        lp = np.ascontiguousarray(lp, dtype=np.float64)
        z = np.ascontiguousarray(z, dtype=np.float64)
        n = Ls[0].shape[0]
        vz = np.empty(n); dvz = np.empty(n)
        self._check(self.lib.gpb200_approx_Lz(self._h, n, l, P, _ptr(lp), pa, pb, _ptr(z), _ptr(vz), _ptr(dvz)),
                    "approx_Lz")
        return vz, dvz

    # -- a10 ------------------------------------------------------------------------------------
    def gp_condition(self, K, Ks, Kss, y, noise_var, jitter=0.0):
        K = _f(K); Ks = _f(Ks); Kss = _f(Kss); y = np.ascontiguousarray(y, dtype=np.float64)
        n = K.shape[0]; m = Ks.shape[0]
        mu = np.empty(m); cov = np.empty((m, m), order="F")
        self._check(self.lib.gpb200_gp_condition(self._h, n, m, _ptr(K), n, _ptr(Ks), m, _ptr(Kss), m, _ptr(y),
                                                 noise_var, jitter, _ptr(mu), _ptr(cov), m), "gp_condition")
        return mu, cov

    def cond_mvn(self, mean, sigma, ng, x_given):
        sigma = _f(sigma)
        N = sigma.shape[0]
        nd = N - ng
        mean_a = None if mean is None else np.ascontiguousarray(mean, dtype=np.float64)
        xg = np.ascontiguousarray(x_given, dtype=np.float64)
        cm = np.empty(nd); cv = np.empty((nd, nd), order="F")
        self._check(self.lib.gpb200_cond_mvn(self._h, ng, nd, _ptr(mean_a), _ptr(sigma), N, _ptr(xg), _ptr(cm),
                                             _ptr(cv), nd), "cond_mvn")
        return cm, cv

    # -- f-4 ---------------------------------------------------------------------------------------
    def normal_fill(self, seed, n, offset=0):
        out = np.empty(int(n))
        self._check(self.lib.gpb200_normal_fill(self._h, int(seed), int(offset), int(n), _ptr(out)), "normal_fill")
        return out

    def mvrnorm(self, ndraws, mu, Sigma, seed, jitter=0.0):
        """MASS::mvrnorm(ndraws, mu, Sigma): (ndraws, m) array (a vector when ndraws == 1, like R)."""
        S = _f(Sigma)
        m = S.shape[0]
        mu_a = None if mu is None else np.ascontiguousarray(mu, dtype=np.float64)
        out = np.empty((ndraws, m), order="F")
        self._check(self.lib.gpb200_mvrnorm(self._h, int(ndraws), m, _ptr(mu_a), _ptr(S), max(m, 1), float(jitter),
                                            int(seed), _ptr(out), max(ndraws, 1)), "mvrnorm")
        return out[0].copy() if ndraws == 1 else np.ascontiguousarray(out)

    def posterior_draws_batched(self, t, y, theta, order=1, s=None, jitter=1e-8, seed=None, z=None):
        """One posterior draw of f^(order) on s (on t when s is None) per hyper-parameter row theta[b] =
        (alpha, rho, sigma), given y observed on t (include/gpb200.h: gpb200_posterior_draws_batched).
        t: (n,) or (B, n); s: (m,) or (B, m); y: (n,) or (B, n); z: (B, m) normals, else the device
        stream of `seed` (0 when None).  Returns draws (B, m), mu (B, m), info (B,)."""
        th = np.ascontiguousarray(theta, dtype=np.float64)
        if th.ndim != 2 or th.shape[1] != 3:
            raise ValueError("theta must be (B, 3) = (alpha, rho, sigma) per row")
        B = th.shape[0]
        t = np.ascontiguousarray(t, dtype=np.float64); y = np.ascontiguousarray(y, dtype=np.float64)
        if t.ndim not in (1, 2) or y.ndim not in (1, 2):
            raise ValueError("t and y must be (n,) or (B, n)")
        n = t.shape[-1]
        if y.shape[-1] != n or (t.ndim == 2 and t.shape[0] != B) or (y.ndim == 2 and y.shape[0] != B):
            raise ValueError("t and y must be (n,) or (B, n) with the same n")
        s_a = None if s is None else np.ascontiguousarray(s, dtype=np.float64)
        if s_a is not None and (s_a.ndim not in (1, 2) or (s_a.ndim == 2 and s_a.shape[0] != B)):
            raise ValueError("s must be (m,) or (B, m)")
        m = n if s_a is None else s_a.shape[-1]
        z_a = None
        if z is not None:
            z_a = np.ascontiguousarray(z, dtype=np.float64)
            if z_a.shape != (B, m):
                raise ValueError("z must be (B, m)")
        draws = np.empty((B, m)); mu = np.empty((B, m)); info = np.zeros(B, dtype=np.int32)
        self._check(self.lib.gpb200_posterior_draws_batched(
            self._h, n, m, int(order), B, _ptr(t), n if t.ndim == 2 else 0, _ptr(s_a),
            m if s_a is not None and s_a.ndim == 2 else 0, _ptr(y), n if y.ndim == 2 else 0, _ptr(th), float(jitter),
            _ptr(z_a), int(seed or 0), _ptr(draws), _ptr(mu), _ptr(info)), "posterior_draws_batched")
        return draws, mu, info

    def posterior_draws_batched_device(self, n, m, order, B, t, t_stride, s, s_stride, y, y_stride, theta, jitter, z, seed,
                                       draws, mu, info):
        """Device-pointer variant: every array argument is a torch CUDA tensor (float64 / int32) or None; the
        handle must be in device-pointer mode.  Asynchronous on the handle's stream."""
        assert self.device_pointers
        self._check(self.lib.gpb200_posterior_draws_batched(self._h, n, m, order, B, _ptr(t), t_stride, _ptr(s), s_stride,
                                                            _ptr(y), y_stride, _ptr(theta), jitter, _ptr(z), int(seed),
                                                            _ptr(draws), _ptr(mu), _ptr(info)), "posterior_draws_batched")


_default = {}


def default_handle(device: int = 0) -> Handle:
    if device not in _default:
        _default[device] = Handle(device)
    return _default[device]
