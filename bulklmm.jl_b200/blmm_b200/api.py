"""Host-side mirror of BulkLMM.jl's public API for the multi-trait genome-scan path, on top of the
C-ABI of libblmm_b200.so.

Julia is not installed in the build image, so this Python layer stands where the Julia shim
(bulklmm.jl_b200/julia/BulkLMMB200.jl) stands in production: same function names, keyword
arguments, defaults, result fields and error strings as the reference

    bulkscan / bulkscan_null_grid / bulkscan_alt_grid / bulkscan_null   src/bulkscan.jl:81-526
    scan(...; permutation_test=true, nperms, rndseed)                   src/scan.jl:94-271, 485-557
    calcKinship                                                         src/kinship.jl:4-14
    transform_rotation                                                  src/transform_helpers.jl:1-54
    get_thresholds                               src/analysis_helpers/single_trait_analysis.jl:13-23

All compute happens in the CUDA library; what is done here is argument plumbing (intercept column,
observation-weight pre-scaling, column-major staging).  Matrices are n x m (traits), n x p
(markers), results p x m, exactly as in Julia.
"""
from __future__ import annotations

import ctypes as C
from types import SimpleNamespace
from typing import Optional, Sequence

import os

import numpy as np

from . import _lib as L


class BlmmError(Exception):
    """Mirrors Julia `error(msg)`: `.msg` is the reference's string, `.code` the BLMM_E_* status."""

    def __init__(self, code: int, msg: str):
        super().__init__(msg)
        self.code = code
        self.msg = msg


def _f(a) -> np.ndarray:
    """float64, column-major (Julia layout)."""
    return np.asfortranarray(np.asarray(a, dtype=np.float64))


def _ptr(a: Optional[np.ndarray]):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class Engine:
    """One context = one GPU (blmm_create), or, with `devices=[...]`, several GPUs of one box behind one
    context (blmm_create_multi: traits / permutation columns sharded inside the library).  Not thread-safe:
    one call in flight per engine."""

    def __init__(self, device: int = 0, devices: Optional[Sequence[int]] = None):
        self.lib = L.load()
        h = C.c_void_p()
        if devices is not None:
            devs = (C.c_int * len(devices))(*[int(d) for d in devices])
            st = self.lib.blmm_create_multi(C.byref(h), devs, len(devices))
            device = int(devices[0]) if len(devices) else 0
        else:
            st = self.lib.blmm_create(C.byref(h), int(device))
        if st != L.OK:
            raise BlmmError(st, "blmm_create failed: no usable sm_100 (B200) device" if st == L.E_NO_DEVICE
                            else f"blmm_create failed with status {st}")
        self.h = h
        self.device = device

    @property
    def device_count(self) -> int:
        return int(self.lib.blmm_device_count(self.h))

    def last_gather_ms(self) -> float:
        return float(self.lib.blmm_last_gather_ms(self.h))

    def close(self):
        if getattr(self, "h", None):
            self.lib.blmm_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- plumbing ----------------------------------------------------------------------------
    def _check(self, st: int):
        if st != L.OK:
            raise BlmmError(st, self.lib.blmm_last_error(self.h).decode())

    def sync(self):
        self._check(self.lib.blmm_sync(self.h))

    @property
    def stream(self) -> int:
        return int(self.lib.blmm_stream(self.h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.blmm_launch_count(self.h))

    def set_profiling(self, on: bool):
        self.lib.blmm_set_profiling(self.h, int(on))

    def last_scan_ms(self) -> float:
        return float(self.lib.blmm_last_scan_ms(self.h))

    @staticmethod
    def make_opts(method=L.METHOD_NULL_GRID, reml=False, prior_variance=1.0, prior_sample_size=0.0,
                  h2_grid=None, optim_interval=1, h2_panel_mode=L.H2PANEL_REFERENCE, mem_space=L.MEM_HOST,
                  ld_out=0, chisq_df=0, log10p_out=None):
        o = L.Opts()
        o.method = method
        o.reml = int(bool(reml))
        o.prior_variance = float(prior_variance)
        o.prior_sample_size = float(prior_sample_size)
        keep = None
        if h2_grid is not None:
            keep = np.ascontiguousarray(np.asarray(h2_grid, dtype=np.float64))
            o.h2_grid = keep.ctypes.data_as(L.c_double_p)
            o.ngrid = keep.shape[0]
        o.optim_interval = int(optim_interval)
        o.h2_panel_mode = h2_panel_mode
        o.mem_space = mem_space
        o.ld_out = ld_out
        o.chisq_df = int(chisq_df)
        o.log10p_out = log10p_out
        return o, keep

    @staticmethod
    def make_problem(n, p, m, c, Y, G, Covar, U, lam, obs_weights=None):
        """Raw-pointer problem (ints are addresses: host numpy `.ctypes.data` or device `data_ptr()`)."""
        pr = L.Problem()
        pr.n, pr.p, pr.m, pr.c = n, p, m, c
        pr.Y, pr.G, pr.Covar, pr.U, pr.lam = Y, G, Covar, U, lam
        pr.obs_weights = obs_weights
        return pr

    def _host_problem(self, Y, G, Covar, U, lam, weights=None):
        n = Covar.shape[0]
        m = 0 if Y is None else Y.shape[1]
        p = 0 if G is None else G.shape[1]
        # raw pointers cross the ABI next: every array must have the n rows the library will read
        if (U.ndim != 2 or U.shape != (n, n) or lam.shape != (n,) or (Y is not None and Y.shape[0] != n)
                or (G is not None and G.shape[0] != n) or (weights is not None and weights.shape != (n,))):
            raise BlmmError(L.E_DIM, "Dimension mismatch.")
        pr = self.make_problem(n, p, m, Covar.shape[1],
                               None if Y is None else Y.ctypes.data, None if G is None else G.ctypes.data,
                               Covar.ctypes.data, U.ctypes.data, lam.ctypes.data,
                               None if weights is None else weights.ctypes.data)
        return pr

    # -- setup ---------------------------------------------------------------------------------
    def calc_kinship(self, G) -> np.ndarray:
        G = _f(G)
        n, p = G.shape
        K = np.empty((n, n), order="F")
        self._check(self.lib.blmm_kinship(self.h, n, p, _ptr(G), _ptr(K), L.MEM_HOST))
        return K

    def weight_kinship(self, K, weights) -> np.ndarray:
        """W*K*W (src/bulkscan.jl:239)."""
        K, w = _f(K), np.ascontiguousarray(weights, dtype=np.float64)
        n = K.shape[0]
        if K.shape[1] != n or w.shape != (n,):
            raise BlmmError(L.E_DIM, "Dimension mismatch.")
        out = np.empty((n, n), order="F")
        self._check(self.lib.blmm_weight_kinship(self.h, n, _ptr(K), _ptr(w), _ptr(out), L.MEM_HOST))
        return out

    def lod2log10p(self, lod, df: int = 1) -> np.ndarray:
        """src/util.jl:199-206 elementwise on the device."""
        a = _f(np.atleast_2d(np.asarray(lod, dtype=np.float64).T).T) if np.ndim(lod) < 2 else _f(lod)
        out = np.empty_like(a, order="F")
        self._check(self.lib.blmm_lod2log10p(self.h, _ptr(a), a.shape[0], a.shape[1], 0, 0, int(df), _ptr(out),
                                             L.MEM_HOST))
        return out.reshape(np.shape(lod))

    def thresholds(self, max_lod, signif_level) -> np.ndarray:
        """Type-7 quantiles of the per-permutation maximum LODs at 1 - signif_level (device sort)."""
        mx = np.ascontiguousarray(max_lod, dtype=np.float64)
        sl = np.ascontiguousarray(signif_level, dtype=np.float64)
        thr = np.empty(sl.shape[0])
        self._check(self.lib.blmm_thresholds(self.h, _ptr(mx), mx.shape[0], _ptr(sl), sl.shape[0], _ptr(thr),
                                             L.MEM_HOST))
        return thr

    def decompose(self, K, decomp_scheme: str = "eigen"):
        """(U, lambda): columns of U are eigenvectors (Ut = U.T).  Returns also #eigenvalues < -1e-7."""
        if decomp_scheme not in ("eigen", "svd"):
            raise BlmmError(L.E_INVALID, "Please choose either `eigen` or `svd` for decomposition of the kinship matrix.")
        K = _f(K)
        n = K.shape[0]
        if K.shape[1] != n:
            raise BlmmError(L.E_DIM, "Dimension mismatch.")
        U = np.empty((n, n), order="F")
        lam = np.empty(n)
        nneg = C.c_int(0)
        self._check(self.lib.blmm_decompose(self.h, n, _ptr(K), L.DECOMP_EIGEN if decomp_scheme == "eigen" else L.DECOMP_SVD,
                                            _ptr(U), _ptr(lam), C.byref(nneg), L.MEM_HOST))
        return U, lam, int(nneg.value)

    def rotate(self, Y, X, U, lam):
        """(Ut*Y, Ut*X) for a given decomposition."""
        Y, X, U = _f(Y), _f(X), _f(U)
        n = Y.shape[0]
        pr = self.make_problem(n, 0, Y.shape[1], X.shape[1], Y.ctypes.data, None, X.ctypes.data, U.ctypes.data,
                               np.ascontiguousarray(lam).ctypes.data)
        Y0 = np.empty_like(Y, order="F")
        X0 = np.empty_like(X, order="F")
        self._check(self.lib.blmm_rotate(self.h, C.byref(pr), _ptr(Y0), _ptr(X0), L.MEM_HOST))
        return Y0, X0

    # -- the hot path (raw pointers: device-resident buffers, asynchronous until sync()) --------
    def bulkscan_raw(self, pr, opts, L_ptr: int, h2_ptr: Optional[int]):
        self._check(self.lib.blmm_bulkscan(self.h, C.byref(pr), C.byref(opts), C.c_void_p(L_ptr),
                                           C.c_void_p(h2_ptr) if h2_ptr else None))

    def bulkscan_peaks_raw(self, pr, opts, lod_ptr: int, marker_ptr: Optional[int], h2_ptr: Optional[int]):
        """blmm_bulkscan_peaks with raw pointers (m doubles, m int64 markers, m doubles)."""
        vp = lambda a: C.c_void_p(a) if a else None
        self._check(self.lib.blmm_bulkscan_peaks(self.h, C.byref(pr), C.byref(opts), vp(lod_ptr), vp(marker_ptr),
                                                 vp(h2_ptr)))

    def scan_perms_raw(self, pr, opts, perm_ptr: int, nperms: int, lod_ptr: int, Lperms_ptr: Optional[int],
                       max_ptr: Optional[int], s2_ptr: Optional[int], h2_ptr: Optional[int]):
        vp = lambda a: C.c_void_p(a) if a else None
        self._check(self.lib.blmm_scan_perms(self.h, C.byref(pr), C.byref(opts), vp(perm_ptr), nperms, vp(lod_ptr),
                                             vp(Lperms_ptr), vp(max_ptr), vp(s2_ptr), vp(h2_ptr)))

    # -- the hot path (host buffers) -----------------------------------------------------------
    def bulkscan_host(self, Y, G, Covar, U, lam, method, h2_grid, reml, prior_variance, prior_sample_size,
                      optim_interval=1, h2_panel_mode=L.H2PANEL_REFERENCE, want_h2=True, weights=None,
                      chisq_df=0):
        """Returns (L, h2) or, with chisq_df > 0, (L, h2, log10p)."""
        Y, G, Covar, U = _f(Y), _f(G), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        p, m = G.shape[1], Y.shape[1]
        pr = self._host_problem(Y, G, Covar, U, lam, weights)
        P = np.empty((p, m), order="F") if chisq_df else None
        o, keep = self.make_opts(method=method, reml=reml, prior_variance=prior_variance,
                                 prior_sample_size=prior_sample_size, h2_grid=h2_grid,
                                 optim_interval=optim_interval, h2_panel_mode=h2_panel_mode, chisq_df=chisq_df,
                                 log10p_out=None if P is None else P.ctypes.data)
        Lout = np.empty((p, m), order="F")
        if method == L.METHOD_ALT_GRID:
            H = np.empty((p, m), order="F") if want_h2 else None
        else:
            H = np.empty(m) if want_h2 else None
        self._check(self.lib.blmm_bulkscan(self.h, C.byref(pr), C.byref(o), _ptr(Lout), _ptr(H)))
        return (Lout, H, P) if chisq_df else (Lout, H)

    def bulkscan_peaks_host(self, Y, G, Covar, U, lam, method, h2_grid, reml, prior_variance, prior_sample_size,
                            optim_interval=1, h2_panel_mode=L.H2PANEL_REFERENCE, weights=None, chisq_df=0):
        """Per-trait peaks of the bulk scan: (lod, marker (0-based int64), h2) or, with chisq_df > 0,
        (lod, marker, h2, log10p), each of length m; no p x m matrix is formed."""
        Y, G, Covar, U = _f(Y), _f(G), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        m = Y.shape[1]
        pr = self._host_problem(Y, G, Covar, U, lam, weights)
        P = np.empty(m) if chisq_df else None
        o, keep = self.make_opts(method=method, reml=reml, prior_variance=prior_variance,
                                 prior_sample_size=prior_sample_size, h2_grid=h2_grid,
                                 optim_interval=optim_interval, h2_panel_mode=h2_panel_mode, chisq_df=chisq_df,
                                 log10p_out=None if P is None else P.ctypes.data)
        lod, marker, H = np.empty(m), np.empty(m, dtype=np.int64), np.empty(m)
        self._check(self.lib.blmm_bulkscan_peaks(self.h, C.byref(pr), C.byref(o), _ptr(lod), _ptr(marker), _ptr(H)))
        return (lod, marker, H, P) if chisq_df else (lod, marker, H)

    def grid_loglik(self, Y, Covar, U, lam, h2_grid, reml=False, prior_variance=1.0, prior_sample_size=0.0):
        Y, Covar, U = _f(Y), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        pr = self._host_problem(Y, None, Covar, U, lam)
        o, keep = self.make_opts(reml=reml, prior_variance=prior_variance, prior_sample_size=prior_sample_size,
                                 h2_grid=h2_grid)
        ell = np.empty((len(keep), Y.shape[1]), order="F")
        self._check(self.lib.blmm_grid_loglik(self.h, C.byref(pr), C.byref(o), _ptr(ell)))
        return ell

    def fit_h2(self, Y, Covar, U, lam, reml=False, prior_variance=0.0, prior_sample_size=0.0, optim_interval=1):
        Y, Covar, U = _f(Y), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        m = Y.shape[1]
        pr = self._host_problem(Y, None, Covar, U, lam)
        o, _ = self.make_opts(reml=reml, prior_variance=prior_variance, prior_sample_size=prior_sample_size,
                              optim_interval=optim_interval)
        h2, s2, ell = np.empty(m), np.empty(m), np.empty(m)
        self._check(self.lib.blmm_fit_h2(self.h, C.byref(pr), C.byref(o), _ptr(h2), _ptr(s2), _ptr(ell)))
        return h2, s2, ell

    def scan_null_host(self, Y, G, Covar, U, lam, reml=False, prior_variance=0.0, prior_sample_size=0.0,
                       optim_interval=1, weights=None):
        """blmm_scan_null: per-trait fitlmm + single-trait null scan for every column of Y."""
        Y, G, Covar, U = _f(Y), _f(G), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        p, m = G.shape[1], Y.shape[1]
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        pr = self._host_problem(Y, G, Covar, U, lam, weights)
        o, _ = self.make_opts(method=L.METHOD_NULL_EXACT, reml=reml, prior_variance=prior_variance,
                              prior_sample_size=prior_sample_size, optim_interval=optim_interval)
        lod = np.empty((p, m), order="F")
        s2, h2 = np.empty(m), np.empty(m)
        self._check(self.lib.blmm_scan_null(self.h, C.byref(pr), C.byref(o), _ptr(lod), _ptr(s2), _ptr(h2)))
        return lod, s2, h2

    def scan_alt_host(self, y, G, Covar, U, lam, reml=False, prior_variance=0.0, prior_sample_size=0.0,
                      optim_interval=1, weights=None):
        """blmm_scan_alt: per-marker variance components (src/scan.jl:397-453)."""
        y, G, Covar, U = _f(y), _f(G), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        p = G.shape[1]
        pr = self._host_problem(y, G, Covar, U, lam, weights)
        o, _ = self.make_opts(method=L.METHOD_NULL_EXACT, reml=reml, prior_variance=prior_variance,
                              prior_sample_size=prior_sample_size, optim_interval=optim_interval)
        lod, h2e, s2, h2 = np.empty(p), np.empty(p), np.empty(1), np.empty(1)
        self._check(self.lib.blmm_scan_alt(self.h, C.byref(pr), C.byref(o), _ptr(lod), _ptr(h2e), _ptr(s2), _ptr(h2)))
        return lod, h2e, float(s2[0]), float(h2[0])

    def scan_perms_host(self, y, G, Covar, U, lam, perm_idx, reml=False, prior_variance=0.0,
                        prior_sample_size=0.0, optim_interval=1, want_L=True, want_max=True, weights=None):
        y, G, Covar, U = _f(y), _f(G), _f(Covar), _f(U)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        perm_idx = np.asfortranarray(np.asarray(perm_idx, dtype=np.int32))
        n, p = G.shape
        if perm_idx.ndim != 2 or (perm_idx.shape[1] > 0 and perm_idx.shape[0] != n):
            raise BlmmError(L.E_DIM, "Dimension mismatch.")
        nperms = perm_idx.shape[1]
        weights = None if weights is None else np.ascontiguousarray(weights, dtype=np.float64)
        pr = self._host_problem(y, G, Covar, U, lam, weights)
        o, _ = self.make_opts(reml=reml, prior_variance=prior_variance, prior_sample_size=prior_sample_size,
                              optim_interval=optim_interval)
        lod = np.empty(p)
        Lp = np.empty((p, nperms), order="F") if want_L else None
        mx = np.empty(nperms) if want_max else None
        s2, h2 = np.empty(1), np.empty(1)
        self._check(self.lib.blmm_scan_perms(self.h, C.byref(pr), C.byref(o), _ptr(perm_idx), nperms, _ptr(lod),
                                             _ptr(Lp), _ptr(mx), _ptr(s2), _ptr(h2)))
        return SimpleNamespace(sigma2_e=float(s2[0]), h2_null=float(h2[0]), lod=lod, L_perms=Lp, max_lod=mx)


_default_engine: Optional[Engine] = None


def default_engine() -> Engine:
    global _default_engine
    if _default_engine is None:
        _default_engine = Engine(0)
    return _default_engine


# ---------------------------------------------------------------------------------------------
# Reference-shaped functions
# ---------------------------------------------------------------------------------------------
def calcKinship(geno, engine: Optional[Engine] = None) -> np.ndarray:
    """src/kinship.jl:4-14."""
    return (engine or default_engine()).calc_kinship(geno)


def transform_rotation(y, g, K, addIntercept: bool = True, decomp_scheme: str = "eigen",
                       engine: Optional[Engine] = None):
    """src/transform_helpers.jl:1-54 -> (Ut*y, Ut*X, lambda)."""
    eng = engine or default_engine()
    y, g = _f(y), _f(g)
    n = y.shape[0]
    if g.shape[0] != n or np.asarray(K).shape[0] != n:
        raise BlmmError(L.E_DIM, "Dimension mismatch.")
    X = np.hstack([np.ones((n, 1)), g]) if addIntercept else g
    U, lam, _ = eng.decompose(K, decomp_scheme)
    Y0, X0 = eng.rotate(y, X, U, lam)
    return Y0, X0, lam


def _prep(Y, G, Covar, K, weights, addIntercept, eng):
    """The argument plumbing shared by the scan entry points: default intercept-only covariates
    (3-argument forms, src/bulkscan.jl:94-109) and the intercept column.  Observation weights
    (src/bulkscan.jl:231-250, 351-370, 457-476) are NOT applied here: they cross the ABI
    (blmm_problem.obs_weights) and Y, G, Covar are row-scaled on the device; only the n x n kinship is
    turned into W*K*W up front (blmm_weight_kinship) because it feeds the decomposition."""
    Y = np.asarray(Y, dtype=np.float64)
    if Y.ndim == 1:
        Y = Y.reshape(-1, 1)
    G = np.asarray(G, dtype=np.float64)
    K = np.asarray(K, dtype=np.float64)
    n = Y.shape[0]
    if G.shape[0] != n or K.shape[0] != n or K.shape[1] != n:
        raise BlmmError(L.E_DIM, "Dimension mismatch.")
    if Covar is None:
        C0 = np.ones((n, 1))
    else:
        Covar = np.asarray(Covar, dtype=np.float64).reshape(n, -1)
        C0 = np.hstack([np.ones((n, 1)), Covar]) if addIntercept else Covar
    if weights is not None:
        weights = np.ascontiguousarray(weights, dtype=np.float64)
        if weights.shape != (n,):
            raise BlmmError(L.E_DIM, "Dimension mismatch.")
        K = eng.weight_kinship(K, weights)
    return Y, G, C0, K, weights


_METHODS = {"null-grid": L.METHOD_NULL_GRID, "alt-grid": L.METHOD_ALT_GRID, "null-exact": L.METHOD_NULL_EXACT}


def bulkscan(Y, G, K, Covar=None, method: str = "null-grid", h2_grid=None, nb: int = 1, nt_blas: int = 1,
             addIntercept: bool = True, weights=None, prior_variance: float = 1.0,
             prior_sample_size: float = 0.0, reml: bool = False, optim_interval: int = 1,
             decomp_scheme: str = "eigen", output_pvals: bool = False, chisq_df: int = 1,
             h2_panel_mode: str = "reference", decomposition=None, engine: Optional[Engine] = None):
    """src/bulkscan.jl:81-162.  `nb` / `nt_blas` are accepted and ignored (CPU threading knobs).
    `decomposition=(U, lambda)` skips the kinship eigendecomposition (blmm_decompose)."""
    eng = engine or default_engine()
    if method not in _METHODS:
        raise BlmmError(L.E_INVALID, "unknown method: choose null-exact, null-grid or alt-grid")
    if h2_grid is None:
        h2_grid = np.arange(10) / 10.0  # collect(0.0:0.1:0.9), src/bulkscan.jl:82
    Y, G, C0, K, weights = _prep(Y, G, Covar, K, weights, addIntercept, eng)
    if decomposition is None:
        U, lam, _ = eng.decompose(K, decomp_scheme)
    else:
        U, lam = decomposition
    mode = L.H2PANEL_ARGMAX if h2_panel_mode == "argmax" else L.H2PANEL_REFERENCE
    res = eng.bulkscan_host(Y, G, C0, U, lam, _METHODS[method], h2_grid, reml, prior_variance,
                            prior_sample_size, optim_interval=optim_interval, h2_panel_mode=mode, weights=weights,
                            chisq_df=chisq_df if output_pvals else 0)
    Lmat, H = res[0], res[1]
    out = SimpleNamespace(L=Lmat)
    if method == "alt-grid":
        out.h2_panel = H
    else:
        out.h2_null_list = H
    if output_pvals:
        out.log10Pvals_mat = res[2]  # fused on the device before the copy-back (blmm_opts.chisq_df)
        out.Chisq_df = chisq_df
    return out


def bulkscan_peaks(Y, G, K, Covar=None, method: str = "null-grid", h2_grid=None, nb: int = 1, nt_blas: int = 1,
                   addIntercept: bool = True, weights=None, prior_variance: float = 1.0,
                   prior_sample_size: float = 0.0, reml: bool = False, optim_interval: int = 1,
                   decomp_scheme: str = "eigen", output_pvals: bool = False, chisq_df: int = 1,
                   h2_panel_mode: str = "reference", decomposition=None, engine: Optional[Engine] = None):
    """The per-trait peaks of `bulkscan` with the same keywords, without forming the p x m LOD matrix:
    `lod[j]` = L[marker[j], j] at the first maximum of column j (NaN ranks highest, as Julia's findmax), `marker`
    0-based, `h2[j]` = h2_panel[marker[j], j] (alt-grid) or h2_null_list[j]; `log10Pvals` with output_pvals."""
    eng = engine or default_engine()
    if method not in _METHODS:
        raise BlmmError(L.E_INVALID, "unknown method: choose null-exact, null-grid or alt-grid")
    if h2_grid is None:
        h2_grid = np.arange(10) / 10.0
    Y, G, C0, K, weights = _prep(Y, G, Covar, K, weights, addIntercept, eng)
    if decomposition is None:
        U, lam, _ = eng.decompose(K, decomp_scheme)
    else:
        U, lam = decomposition
    mode = L.H2PANEL_ARGMAX if h2_panel_mode == "argmax" else L.H2PANEL_REFERENCE
    res = eng.bulkscan_peaks_host(Y, G, C0, U, lam, _METHODS[method], h2_grid, reml, prior_variance,
                                  prior_sample_size, optim_interval=optim_interval, h2_panel_mode=mode,
                                  weights=weights, chisq_df=chisq_df if output_pvals else 0)
    out = SimpleNamespace(lod=res[0], marker=res[1], h2=res[2])
    if output_pvals:
        out.log10Pvals = res[3]
    return out


def bulkscan_null_grid(Y, G, K, grid_list, Covar=None, **kw):
    """src/bulkscan.jl:321-385 -> (L, h2_null_list)."""
    return bulkscan(Y, G, K, Covar=Covar, method="null-grid", h2_grid=grid_list, **kw)


def bulkscan_alt_grid(Y, G, K, hsq_list, Covar=None, **kw):
    """src/bulkscan.jl:428-526 -> (L, h2_panel)."""
    return bulkscan(Y, G, K, Covar=Covar, method="alt-grid", h2_grid=hsq_list, **kw)


def bulkscan_null(Y, G, K, Covar=None, **kw):
    """src/bulkscan.jl:188-314 -> (L, h2_null_list)."""
    return bulkscan(Y, G, K, Covar=Covar, method="null-exact", **kw)


def scan(y, g, K, covar=None, weights=None, prior_variance: float = 0.0, prior_sample_size: float = 0.0,
         addIntercept: bool = True, reml: bool = False, assumption: str = "null", method: str = "qr",
         optim_interval: int = 1, permutation_test: bool = False, nperms: int = 1024, rndseed: int = 0,
         perm_idx=None, decomp_scheme: str = "eigen", decomposition=None, engine: Optional[Engine] = None,
         output_pvals: bool = False, chisq_df: int = 1, profileLL: bool = False, markerID: int = 0, h2_grid=None):
    """src/scan.jl:94-271 with permutation_test=true -> scan_perms_lite (src/scan.jl:485-557).

    The shuffles are drawn on the host and cross the ABI as indices (`perm_idx`, n x nperms,
    0-based).  In production the Julia shim draws them from MersenneTwister(rndseed) exactly as
    the reference does; here numpy's generator seeded with `rndseed` stands in: `rndseed` is therefore NOT
    reference-compatible in this mirror (same distribution, different stream) — pass `perm_idx` to reproduce a
    Julia run.  `output_pvals` / `chisq_df` add `log10pvals` (src/scan.jl:353-358, 447-452; for permutations the
    intended result instead of the reference's UndefVarError, SURVEY B2, with df = 1 as scan_perms_lite's default);
    `profileLL` / `markerID` (1-based, as in Julia) / `h2_grid` return (results, profile) as src/scan.jl:249-266."""
    res = _scan(y, g, K, covar, weights, prior_variance, prior_sample_size, addIntercept, reml, assumption, method,
                optim_interval, permutation_test, nperms, rndseed, perm_idx, decomp_scheme, decomposition, engine)
    eng = engine or default_engine()
    if output_pvals:
        df = 1 if permutation_test else chisq_df
        res.log10pvals = eng.lod2log10p(res.lod, df)
        if permutation_test:
            res.log10Pvals_perms = eng.lod2log10p(res.L_perms, df)
    if profileLL:
        # profile_LL, src/analysis_helpers/single_trait_analysis.jl:46-73: null and marker-model log-likelihoods on
        # h2_grid, no intercept added at this point (the reference rotates with addIntercept = false)
        yv = np.asarray(y, dtype=np.float64).reshape(-1, 1)
        n = yv.shape[0]
        gv = np.asarray(g, dtype=np.float64)
        if not (1 <= markerID <= gv.shape[1]):
            raise BlmmError(L.E_INVALID, "markerID out of range")
        cv = np.ones((n, 1)) if covar is None else np.asarray(covar, dtype=np.float64).reshape(n, -1)
        Kv = np.asarray(K, dtype=np.float64)
        if weights is not None:
            w = np.asarray(weights, dtype=np.float64)
            cv = w[:, None] * (np.hstack([np.ones((n, 1)), cv]) if (addIntercept and covar is not None) else cv)
            yv, gcol, Kv = w[:, None] * yv, w[:, None] * gv[:, markerID - 1:markerID], eng.weight_kinship(Kv, w)
        else:
            gcol = gv[:, markerID - 1:markerID]
        U, lam, _ = eng.decompose(Kv, decomp_scheme) if decomposition is None or weights is not None else (*decomposition, 0)
        grid = np.asarray(h2_grid, dtype=np.float64)
        kw = dict(reml=reml, prior_variance=prior_variance, prior_sample_size=prior_sample_size)
        prof = SimpleNamespace(ll_list_null=eng.grid_loglik(yv, cv, U, lam, grid, **kw)[:, 0],
                               ll_list_alt=eng.grid_loglik(yv, np.hstack([cv, gcol]), U, lam, grid, **kw)[:, 0])
        return res, prof
    return res


def _scan(y, g, K, covar, weights, prior_variance, prior_sample_size, addIntercept, reml, assumption, method,
          optim_interval, permutation_test, nperms, rndseed, perm_idx, decomp_scheme, decomposition, engine):
    eng = engine or default_engine()
    y = np.asarray(y, dtype=np.float64)
    if y.ndim == 1:
        y = y.reshape(-1, 1)
    if covar is None and not addIntercept:
        raise BlmmError(L.E_INVALID, "Intercept has to be added when no other covariate is given.")
    if assumption not in ("null", "alt"):
        raise BlmmError(L.E_INVALID, "Assumption keyword is not supported. Please enter null or alt.")
    if assumption == "alt" and permutation_test:
        raise BlmmError(L.E_INVALID, "Permutation test option currently is not supported for the alternative assumption.")
    if y.shape[1] != 1:
        raise BlmmError(L.E_ONE_TRAIT, "Can only handle one trait.")
    y, g, C0, K, weights = _prep(y, g, covar, K, weights, addIntercept, eng)
    n = y.shape[0]
    if assumption == "alt":
        # scan_alt, src/scan.jl:397-453
        if decomposition is None:
            U, lam, _ = eng.decompose(K, decomp_scheme)
        else:
            U, lam = decomposition
        lod, h2e, s2, h2 = eng.scan_alt_host(y, g, C0, U, lam, reml=reml, prior_variance=prior_variance,
                                             prior_sample_size=prior_sample_size, optim_interval=optim_interval,
                                             weights=weights)
        return SimpleNamespace(sigma2_e=s2, h2_null=h2, h2_each_marker=h2e, lod=lod)
    if not permutation_test:
        # scan_null, src/scan.jl:310-360
        if decomposition is None:
            U, lam, _ = eng.decompose(K, decomp_scheme)
        else:
            U, lam = decomposition
        lod, s2, h2 = eng.scan_null_host(y, g, C0, U, lam, reml=reml, prior_variance=prior_variance,
                                         prior_sample_size=prior_sample_size, optim_interval=optim_interval,
                                         weights=weights)
        return SimpleNamespace(sigma2_e=float(s2[0]), h2_null=float(h2[0]), lod=lod[:, 0].copy())
    if perm_idx is None:
        from .synth import make_perm_indices
        perm_idx = make_perm_indices(n, nperms, rndseed)
    if decomposition is None:
        U, lam, _ = eng.decompose(K, decomp_scheme)
    else:
        U, lam = decomposition
    r = eng.scan_perms_host(y, g, C0, U, lam, perm_idx, reml=reml, prior_variance=prior_variance,
                            prior_sample_size=prior_sample_size, optim_interval=optim_interval, weights=weights)
    return r


def get_thresholds(L_perms: np.ndarray, signif_level: Sequence[float], engine: Optional[Engine] = None):
    """src/analysis_helpers/single_trait_analysis.jl:13-23 (Julia `quantile` = type 7).  Given the full
    L_perms matrix as in the reference; the column maxima are taken here, the quantiles on the device."""
    return thresholds_from_max(np.max(np.asarray(L_perms), axis=0), signif_level, engine=engine)


def thresholds_from_max(max_lod: np.ndarray, signif_level: Sequence[float], engine: Optional[Engine] = None):
    """get_thresholds from the per-permutation maxima the fused kernel returns (no L_perms needed):
    blmm_thresholds sorts them on the device and interpolates the type-7 quantiles."""
    eng = engine or default_engine()
    sl = np.asarray(signif_level, dtype=np.float64)
    return SimpleNamespace(probs=1.0 - sl, thrs=eng.thresholds(max_lod, sl))


def lod2log10p(lod, df: int = 1, engine: Optional[Engine] = None):
    """src/util.jl:199-206 on the device (blmm_lod2log10p)."""
    return (engine or default_engine()).lod2log10p(lod, df)


# ---- data ingest (src/readData.jl) ------------------------------------------------------------------
class DeviceMatrix:
    """A column-major Float64 matrix in device memory owned by the library (blmm_read_csv with device >= 0):
    `.ptr` goes straight into Engine.make_problem for BLMM_MEM_DEVICE calls."""

    def __init__(self, ptr: int, rows: int, cols: int, device: int):
        self.ptr, self.shape, self.device = ptr, (rows, cols), device

    def free(self):
        if self.ptr:
            L.load().blmm_free_matrix(self.ptr, self.device)
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def read_csv_matrix(path: str, skip_rows: int = 1, first_col: int = 0, col_step: int = 1, drop_last_cols: int = 0,
                    delim: str = ",", device: Optional[int] = None):
    """blmm_read_csv: numpy array (Fortran order) or, with `device=<gpu index>`, a DeviceMatrix."""
    lib = L.load()
    rows, cols, data = C.c_int64(0), C.c_int64(0), C.c_void_p(0)
    dev = -1 if device is None else int(device)
    st = lib.blmm_read_csv(os.fsencode(path), delim.encode()[:1], skip_rows, first_col, col_step, drop_last_cols, dev,
                           C.byref(rows), C.byref(cols), C.byref(data))
    if st != 0:
        raise BlmmError(st, lib.blmm_io_last_error().decode())
    if dev >= 0:
        return DeviceMatrix(data.value, rows.value, cols.value, dev)
    try:
        n = rows.value * cols.value
        arr = np.ctypeslib.as_array(C.cast(data, C.POINTER(C.c_double)), shape=(max(n, 1),))[:n].copy()
    finally:
        lib.blmm_free_matrix(data, -1)
    return arr.reshape((rows.value, cols.value), order="F")


def readBXDpheno(file: str, device: Optional[int] = None):
    """src/readData.jl:159-161: skip the header line, drop the first (id) and last (sex) columns."""
    return read_csv_matrix(file, skip_rows=1, first_col=1, col_step=1, drop_last_cols=1, device=device)


def readBXDgeno(file: str, skipstart: int = 1, device: Optional[int] = None):
    """src/readData.jl:163-165: `[:, 2:2:end]` of the data lines."""
    return read_csv_matrix(file, skip_rows=skipstart, first_col=1, col_step=2, device=device)


def readGenoProb_ExcludeComplements(file: str, device: Optional[int] = None):
    """src/readData.jl:85-96: header of marker names, first column ids, then the odd probability columns."""
    return read_csv_matrix(file, skip_rows=1, first_col=1, col_step=2, device=device)
