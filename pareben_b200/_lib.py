"""ctypes binding to libpareben.so (the C-ABI declared in include/pareben.h).

The shared library is built in-tree by `__graft_entry__.build()` (nvcc, sm_100a).  There is
no CPU fallback: if the library is missing, or no CUDA device is present, calls raise.
"""
from __future__ import annotations

import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("PAREBEN_LIB") or os.path.join(_HERE, "libpareben.so")

GAUSSIAN, BINOMIAL = 0, 1
FIT_BASIS_CAP, FIT_NOT_PD, FIT_NONFINITE, FIT_ITER_MAX, FIT_LIST_CAP = 1, 2, 4, 8, 16
MODE_AUTO, MODE_CACHED, MODE_STREAMING = 0, 1, 2

_dp = ctypes.POINTER(ctypes.c_double)
_ip = ctypes.POINTER(ctypes.c_int)
_vp = ctypes.c_void_p

# every symbol include/pareben.h declares: (restype, argtypes)
SIGNATURES = {
    "pareben_problem_create": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, _dp, ctypes.c_int, ctypes.c_int, _dp, _ip,
                                              ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "pareben_problem_create_multi": (ctypes.c_int, [ctypes.POINTER(_vp), ctypes.c_int, _dp, ctypes.c_int, ctypes.c_int, _dp,
                                                    ctypes.c_int, _ip, ctypes.c_int, ctypes.c_int, ctypes.c_int]),
    "pareben_problem_destroy": (None, [_vp]),
    "pareben_release_cache": (None, []),
    "pareben_run_fits": (ctypes.c_int, [_vp, ctypes.c_int, _ip, _dp, _dp, _dp, _ip, _ip, _ip]),
    "pareben_cv_grid": (ctypes.c_int, [_dp, ctypes.c_int, ctypes.c_int, _dp, _ip, ctypes.c_int, _dp, _dp, ctypes.c_int,
                                       ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _dp, _ip,
                                       _ip]),
    "pareben_problem_cv_grid": (ctypes.c_int, [_vp, _dp, _dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _dp, _ip, _ip]),
    "pareben_run_fits_multi": (ctypes.c_int, [_vp, ctypes.c_int, _ip, _ip, _dp, _dp, _dp, _ip, _ip, _ip]),
    "pareben_cv_grid_multi": (ctypes.c_int, [_dp, ctypes.c_int, ctypes.c_int, _dp, ctypes.c_int, _ip, ctypes.c_int, _dp, _dp,
                                             ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_int, _dp, _ip, _ip]),
    "pareben_problem_cv_grid_multi": (ctypes.c_int, [_vp, _dp, _dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, _dp, _ip, _ip]),
    "elasticNetLinearNeMainEff": (None, [_dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip, _ip, _dp]),
    "elasticNetLinearNeEpisEff": (None, [_dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip, _ip, _dp]),
    "ElasticNetBinaryNEmainEff": (None, [_dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip, _ip, _ip]),
    "ElasticNetBinaryNEfull": (None, [_dp, _dp, _dp, _dp, _dp, _dp, _dp, _dp, _ip, _ip, _ip, _ip]),
    "pareben_shard_plan": (ctypes.c_int, [_dp, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_int, _ip, _ip]),
    "pareben_fit": (ctypes.c_int, [_vp, ctypes.c_double, ctypes.c_double, _dp, _dp, _dp, _dp, _ip]),
    "pareben_max_effects": (ctypes.c_int, [_vp, _ip]),
    "pareben_fit_batch": (ctypes.c_int, [_vp, ctypes.c_int, _ip, _ip, _dp, _dp, ctypes.c_int, _ip, _ip, _dp, _dp, _dp, _ip, _dp]),
    "pareben_lambda_max": (ctypes.c_int, [_vp, _dp]),
    "pareben_lambda_max_multi": (ctypes.c_int, [_vp, _dp]),
    "pareben_sl_filter": (ctypes.c_int, [_vp, ctypes.c_double, ctypes.c_double, ctypes.c_int, _ip, _dp, _ip]),
    "pareben_last_counters": (ctypes.c_int, [_vp, _dp, _dp, _ip]),
    "pareben_last_gram_info": (ctypes.c_int, [_vp, _ip, _dp, _dp]),
    "pareben_last_contraction_info": (ctypes.c_int, [_vp, _ip, _dp]),
    "pareben_set_mode": (ctypes.c_int, [ctypes.c_int]),
    "pareben_is_streaming": (ctypes.c_int, [_vp]),
    "pareben_last_stream_counters": (ctypes.c_int, [_vp, _dp, _dp, _ip, _ip]),
    "pareben_measure_fp64_peak": (ctypes.c_int, [ctypes.c_int, ctypes.c_int, _dp]),
    "pareben_device_count": (ctypes.c_int, []),
    "pareben_last_error": (ctypes.c_char_p, []),
    "pareben_version": (ctypes.c_int, []),
}

_lib = None


class ParebenError(RuntimeError):
    pass


def load():
    """Load libpareben.so and bind every declared symbol; raises if the extension is not built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ParebenError(f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                               "(the CUDA extension is the only implementation; there is no CPU path)")
        lib = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc: int):
    if rc != 0:
        raise ParebenError(f"libpareben error {rc}: {load().pareben_last_error().decode()}")


def _d(a):
    return a.ctypes.data_as(_dp)


def _i(a):
    return a.ctypes.data_as(_ip)


def device_count() -> int:
    return load().pareben_device_count()


def release_cache() -> None:
    """Give the library's idle device buffers back to the driver (pareben_release_cache)."""
    load().pareben_release_cache()


def set_mode(mode: int) -> None:
    """pareben_set_mode: 0 automatic, 1 cached kernel, 2 streaming kernels (read when a problem is created)."""
    _check(load().pareben_set_mode(int(mode)))


def default_device() -> int:
    """Device used when the caller does not name one: LOCAL_RANK under a one-process-per-GPU launcher
    (torchrun), else 0 -- so that ranks started with default arguments do not all land on cuda:0."""
    try:
        return int(os.environ.get("LOCAL_RANK", "0"))
    except ValueError:
        return 0


def _targets_matrix(Targets, n: int) -> np.ndarray:
    """An n x T response matrix as the column-major doubles pareben_*_multi take; every shape is checked here."""
    Y = np.asarray(Targets, dtype=np.float64)
    if Y.ndim != 2 or Y.shape[0] != n:
        raise ValueError(f"Targets must be an n x T matrix with n = nrow(BASIS) = {n}; got shape {Y.shape}")
    if Y.shape[1] < 1:
        raise ValueError("Targets must hold at least one response (T >= 1)")
    return np.asfortranarray(Y)


class Problem:
    """One CrossValidate problem resident on a GPU (pareben_problem_create).  A 2-D Target of shape (n, T) makes a problem
    with T responses sharing the design (pareben_problem_create_multi); a 1-D Target is the single-response problem."""

    def __init__(self, BASIS, Target, fold_id=None, n_folds: int = 0, epis: bool = False, prior: str = "gaussian",
                 device: int | None = None):
        lib = load()
        device = default_device() if device is None else int(device)
        self._X = np.asfortranarray(np.asarray(BASIS, dtype=np.float64))
        n, k = self._X.shape
        multi = np.ndim(Target) == 2
        if multi:
            self._y = _targets_matrix(Target, n)
            self.n_targets = self._y.shape[1]
        else:
            self._y = np.ascontiguousarray(np.asarray(Target, dtype=np.float64).ravel())
            self.n_targets = 1
            if self._y.size != n:
                raise ValueError("Target length must equal nrow(BASIS)")
        self.n, self.k, self.n_folds, self.epis = n, k, int(n_folds), bool(epis)
        self.prior = GAUSSIAN if prior == "gaussian" else BINOMIAL
        fid = None
        if n_folds > 0:
            fid = np.ascontiguousarray(np.asarray(fold_id, dtype=np.int32).ravel())
            if fid.size != n:
                raise ValueError("fold_id length must equal nrow(BASIS)")
        self._h = _vp()
        if multi:
            _check(lib.pareben_problem_create_multi(ctypes.byref(self._h), device, _d(self._X), n, k, _d(self._y), self.n_targets,
                                                    _i(fid) if fid is not None else None, self.n_folds, int(self.epis), self.prior))
        else:
            _check(lib.pareben_problem_create(ctypes.byref(self._h), device, _d(self._X), n, k, _d(self._y),
                                              _i(fid) if fid is not None else None, self.n_folds, int(self.epis), self.prior))

    def close(self):
        if getattr(self, "_h", None):
            load().pareben_problem_destroy(self._h)
            self._h = None

    __del__ = close

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    def run_fits(self, fold, alpha, lam, target=None):
        """(fold_err, status, n_selected, n_iter) of independent fits; target: response index of each fit (None: response 0)."""
        fold = np.ascontiguousarray(fold, dtype=np.int32)
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        m = fold.size
        if alpha.size != m or lam.size != m:
            raise ValueError("fold, alpha and lambda must have equal length")
        err = np.empty(m); st = np.empty(m, np.int32); ns = np.empty(m, np.int32); it = np.empty(m, np.int32)
        if target is None:
            _check(load().pareben_run_fits(self._h, m, _i(fold), _d(alpha), _d(lam), _d(err), _i(st), _i(ns), _i(it)))
        else:
            target = np.ascontiguousarray(target, dtype=np.int32)
            if target.size != m:
                raise ValueError("target must have one entry per fit")
            _check(load().pareben_run_fits_multi(self._h, m, _i(target), _i(fold), _d(alpha), _d(lam), _d(err), _i(st), _i(ns), _i(it)))
        return err, st, ns, it

    def cv_grid(self, alpha, lam, shard: int = 0, n_shards: int = 1):
        """The grid call on a problem that is already resident (BuildGrid's lambda_max and the fits share one
        upload): same table layout and the same shard assignment as pareben_cv_grid; entries of other shards stay 0."""
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        if alpha.size != lam.size or self.n_folds < 1:
            raise ValueError("alpha and lambda must have equal length and the problem must have folds")
        nf, total = self.n_folds, alpha.size * self.n_folds
        err = np.zeros(total); st = np.zeros(total, np.int32); ns = np.zeros(total, np.int32)
        _check(load().pareben_problem_cv_grid(self._h, _d(alpha), _d(lam), alpha.size, int(shard), int(n_shards), _d(err), _i(st), _i(ns)))
        return err.reshape(alpha.size, nf), st.reshape(alpha.size, nf), ns.reshape(alpha.size, nf)

    def cv_grid_multi(self, alpha, lam, shard: int = 0, n_shards: int = 1):
        """pareben_problem_cv_grid_multi: alpha and lam are (T, n_grid), one grid per response; returns three
        (T, n_grid, n_folds) tables.  Entries of other shards stay 0."""
        alpha = np.ascontiguousarray(alpha, dtype=np.float64)
        lam = np.ascontiguousarray(lam, dtype=np.float64)
        T = self.n_targets
        if alpha.shape != lam.shape or alpha.ndim != 2 or alpha.shape[0] != T or alpha.shape[1] < 1 or self.n_folds < 1:
            raise ValueError(f"alpha and lambda must both be ({T}, n_grid) arrays and the problem must have folds")
        n_grid, nf = alpha.shape[1], self.n_folds
        total = T * n_grid * nf
        err = np.zeros(total); st = np.zeros(total, np.int32); ns = np.zeros(total, np.int32)
        _check(load().pareben_problem_cv_grid_multi(self._h, _d(alpha), _d(lam), n_grid, int(shard), int(n_shards), _d(err), _i(st), _i(ns)))
        return err.reshape(T, n_grid, nf), st.reshape(T, n_grid, nf), ns.reshape(T, n_grid, nf)

    def fit(self, alpha: float, lam: float):
        """Batch-of-1 final model: returns (beta_table, wald, intercept, extra, status)."""
        k = self.k
        if self.prior == GAUSSIAN:
            rows, cols = ((k + 1) * k // 2, 5) if self.epis else (k, 4)
        else:
            rows, cols = (2 * k, 4) if self.epis else (k, 4)
        beta = np.zeros(rows * cols)
        wald = np.zeros(1); icpt = np.zeros(2); extra = np.zeros(1); st = np.zeros(1, np.int32)
        _check(load().pareben_fit(self._h, float(alpha), float(lam), _d(beta), _d(wald), _d(icpt), _d(extra), _i(st)))
        return beta.reshape((rows, cols), order="F"), float(wald[0]), icpt, float(extra[0]), int(st[0])

    def max_effects(self) -> int:
        """pareben_max_effects: the most effects one fit of this problem can report."""
        out = ctypes.c_int(0)
        _check(load().pareben_max_effects(self._h, ctypes.byref(out)))
        return out.value

    def fit_batch(self, target, fold, alpha, lam):
        """pareben_fit_batch: the final models of len(target) fits in one launch (fit i: response target[i], fold[i]: 0 =
        all rows, f >= 1 = fold f's training rows, at (alpha[i], lam[i])).  Returns a dict of compact records:
        n_effects (m,), cand (m, max_effects) 1-based candidate ids in Used order, beta and var (m, max_effects),
        scalars (m, 4) = wald, intercept[0], intercept[1], residual variance | log-likelihood, status (m,), fold_err (m,)."""
        target = np.ascontiguousarray(target, dtype=np.int32).ravel()
        fold = np.ascontiguousarray(fold, dtype=np.int32).ravel()
        alpha = np.ascontiguousarray(alpha, dtype=np.float64).ravel()
        lam = np.ascontiguousarray(lam, dtype=np.float64).ravel()
        m = target.size
        if fold.size != m or alpha.size != m or lam.size != m:
            raise ValueError("target, fold, alpha and lambda must have equal length")
        me = self.max_effects()
        out = {"n_effects": np.zeros(m, np.int32), "cand": np.zeros((m, me), np.int32), "beta": np.zeros((m, me)),
               "var": np.zeros((m, me)), "scalars": np.zeros((m, 4)), "status": np.zeros(m, np.int32), "fold_err": np.zeros(m)}
        _check(load().pareben_fit_batch(self._h, m, _i(target), _i(fold), _d(alpha), _d(lam), me, _i(out["n_effects"]),
                                        _i(out["cand"]), _d(out["beta"]), _d(out["var"]), _d(out["scalars"]), _i(out["status"]),
                                        _d(out["fold_err"])))
        return out

    def lambda_max(self) -> float:
        out = np.zeros(1)
        _check(load().pareben_lambda_max(self._h, _d(out)))
        return float(out[0])

    def lambda_max_multi(self) -> np.ndarray:
        """pareben_lambda_max_multi: lambda_max of every response (length T), one pass over the candidates."""
        out = np.zeros(self.n_targets)
        _check(load().pareben_lambda_max_multi(self._h, _d(out)))
        return out

    def sl_filter(self, tau_main: float, tau_pair: float):
        """pareben_sl_filter: (candidate ids ascending, statistics) of the single-locus prefilter."""
        cap = 1 << 16
        while True:
            cand = np.empty(cap, np.int32); stat = np.empty(cap); cnt = ctypes.c_int(0)
            _check(load().pareben_sl_filter(self._h, float(tau_main), float(tau_pair), cap, _i(cand), _d(stat), ctypes.byref(cnt)))
            if cnt.value <= cap:
                return cand[:cnt.value].copy(), stat[:cnt.value].copy()
            cap = cnt.value

    @property
    def streaming(self) -> bool:
        return bool(load().pareben_is_streaming(self._h))

    def stream_counters(self):
        """(scan ms, scan flops, scan launches, rounds) of the last run_fits in streaming mode."""
        ms = np.zeros(1); fl = np.zeros(1); ln = np.zeros(1, np.int32); rd = np.zeros(1, np.int32)
        _check(load().pareben_last_stream_counters(self._h, _d(ms), _d(fl), _i(ln), _i(rd)))
        return float(ms[0]), float(fl[0]), int(ln[0]), int(rd[0])

    def counters(self):
        fl = np.zeros(1); ms = np.zeros(1); ln = np.zeros(1, np.int32)
        _check(load().pareben_last_counters(self._h, _d(fl), _d(ms), _i(ln)))
        return float(fl[0]), float(ms[0]), int(ln[0])

    def gram_info(self):
        """(in use, model flops the last run_fits did not execute, ms the last run_fits spent building the matrices):
        the Gram organisation of the Gaussian cached kernels (include/pareben.h, pareben_last_gram_info).  Binomial
        main-effect fits report the FullStats they skip at a fixed point of the posterior mode as not executed."""
        use = np.zeros(1, np.int32); av = np.zeros(1); ms = np.zeros(1)
        _check(load().pareben_last_gram_info(self._h, _i(use), _d(av), _d(ms)))
        return bool(use[0]), float(av[0]), float(ms[0])

    def contraction_info(self):
        """(binomial score contraction on the int8 tensor cores, contractions the last run_fits ran there)
        (include/pareben.h, pareben_last_contraction_info)."""
        tc = np.zeros(1, np.int32); n = np.zeros(1)
        _check(load().pareben_last_contraction_info(self._h, _i(tc), _d(n)))
        return bool(tc[0]), int(n[0])


def cv_grid(BASIS, Target, fold_id, n_folds, alpha, lam, epis=False, prior="gaussian", device=None,
            shard=0, n_shards=1, n_devices=1):
    """pareben_cv_grid: host buffers in, per-fit hold-out errors out (grid-major, fold-minor).
    n_devices GPUs starting at `device` share the call (0 = all visible).  Entries owned by other shards are left 0
    so that shards merge by summation."""
    X = np.asfortranarray(np.asarray(BASIS, dtype=np.float64))
    y = np.ascontiguousarray(np.asarray(Target, dtype=np.float64).ravel())
    fid = np.ascontiguousarray(np.asarray(fold_id, dtype=np.int32).ravel())
    alpha = np.ascontiguousarray(alpha, dtype=np.float64)
    lam = np.ascontiguousarray(lam, dtype=np.float64)
    if X.ndim != 2:
        raise ValueError("BASIS must be a matrix")
    n, k = X.shape
    n_folds = int(n_folds)
    # the C side only sees pointers: every length is checked here
    if y.size != n:
        raise ValueError("Target length must equal nrow(BASIS)")
    if fid.size != n:
        raise ValueError("fold_id length must equal nrow(BASIS)")
    if alpha.size != lam.size or alpha.size < 1:
        raise ValueError("alpha and lambda must be non-empty and of equal length")
    if n_folds < 1:
        raise ValueError("n_folds must be >= 1")
    device = default_device() if device is None else int(device)
    total = alpha.size * n_folds
    err = np.zeros(total); st = np.zeros(total, np.int32); ns = np.zeros(total, np.int32)
    _check(load().pareben_cv_grid(_d(X), n, k, _d(y), _i(fid), n_folds, _d(alpha), _d(lam), alpha.size, int(bool(epis)),
                                  GAUSSIAN if prior == "gaussian" else BINOMIAL, int(n_devices), device, shard, n_shards,
                                  _d(err), _i(st), _i(ns)))
    return err.reshape(alpha.size, n_folds), st.reshape(alpha.size, n_folds), ns.reshape(alpha.size, n_folds)


def cv_grid_multi(BASIS, Targets, fold_id, n_folds, alpha, lam, epis=False, prior="gaussian", device=None,
                  shard=0, n_shards=1, n_devices=1):
    """pareben_cv_grid_multi: T responses (Targets n x T) against one design in one call.  alpha and lam are (T, n_grid),
    each response's own grid; returns three (T, n_grid, n_folds) tables.  Entries owned by other shards are left 0."""
    X = np.asfortranarray(np.asarray(BASIS, dtype=np.float64))
    if X.ndim != 2:
        raise ValueError("BASIS must be a matrix")
    n, k = X.shape
    Y = _targets_matrix(Targets, n)
    T = Y.shape[1]
    fid = np.ascontiguousarray(np.asarray(fold_id, dtype=np.int32).ravel())
    alpha = np.ascontiguousarray(alpha, dtype=np.float64)
    lam = np.ascontiguousarray(lam, dtype=np.float64)
    n_folds = int(n_folds)
    if fid.size != n:
        raise ValueError("fold_id length must equal nrow(BASIS)")
    if alpha.shape != lam.shape or alpha.ndim != 2 or alpha.shape[0] != T or alpha.shape[1] < 1:
        raise ValueError(f"alpha and lambda must both be ({T}, n_grid) arrays")
    if n_folds < 1:
        raise ValueError("n_folds must be >= 1")
    device = default_device() if device is None else int(device)
    n_grid = alpha.shape[1]
    total = T * n_grid * n_folds
    err = np.zeros(total); st = np.zeros(total, np.int32); ns = np.zeros(total, np.int32)
    _check(load().pareben_cv_grid_multi(_d(X), n, k, _d(Y), T, _i(fid), n_folds, _d(alpha), _d(lam), n_grid, int(bool(epis)),
                                        GAUSSIAN if prior == "gaussian" else BINOMIAL, int(n_devices), device, shard, n_shards,
                                        _d(err), _i(st), _i(ns)))
    return err.reshape(T, n_grid, n_folds), st.reshape(T, n_grid, n_folds), ns.reshape(T, n_grid, n_folds)


def shard_plan(lam, n_folds: int, shard: int, n_shards: int) -> np.ndarray:
    """Fit numbers (grid-major, fold-minor) that `shard` of `n_shards` computes; host-only logic."""
    lam = np.ascontiguousarray(lam, dtype=np.float64)
    idx = np.empty(lam.size * n_folds, np.int32)
    cnt = ctypes.c_int(0)
    _check(load().pareben_shard_plan(_d(lam), lam.size, n_folds, shard, n_shards, _i(idx), ctypes.byref(cnt)))
    return idx[:cnt.value].copy()


def measure_fp64_peak(device: int = 0, which: int = 0) -> float:
    out = np.zeros(1)
    _check(load().pareben_measure_fp64_peak(device, which, _d(out)))
    return float(out[0])
