"""ctypes binding of include/inqcohort.h (cohort `outlier` rows and `assoc`, part of libinqcall.so). No CPU fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np

from .api import INQ_OK, InqError, load_library

ZSCORE, DBSCAN = 0, 1
INQ_ERR_NO_MODE, INQ_ERR_HITS_CAP = -15, -16
LINEAR, LOGISTIC, FIRTH = 0, 1, 2
PRED_SUM, PRED_MAX = 0, 1
ASSOC_OK, ASSOC_FEW_SAMPLES, ASSOC_SINGULAR, ASSOC_NO_CONVERGENCE, ASSOC_SEPARATION = 0, 1, 2, 3, 4
ASSOC_STATUS_NAMES = ["ok", "few_samples", "singular", "no_convergence", "separation"]
COX_EFRON, COX_BRESLOW = 0, 1
EXPORTS = ["inq_outlier", "inq_assoc", "inq_assoc_traits", "inq_assoc_cox", "inq_cohort_last_error"]

_BOUND = False


def _lib():
    global _BOUND
    L = load_library()
    if not _BOUND:
        L.inq_outlier.restype = C.c_int
        L.inq_outlier.argtypes = [C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_float,
                                  C.c_void_p, C.POINTER(C.c_uint64), C.c_void_p, C.c_uint64, C.POINTER(C.c_float)]
        L.inq_assoc.restype = C.c_int
        L.inq_assoc.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_uint32,
                                C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_void_p, C.POINTER(C.c_float)]
        L.inq_assoc_traits.restype = C.c_int
        L.inq_assoc_traits.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_uint32, C.c_void_p,
                                       C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        L.inq_assoc_cox.restype = C.c_int
        L.inq_assoc_cox.argtypes = [C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                    C.c_void_p, C.c_void_p, C.POINTER(C.c_float)]
        L.inq_cohort_last_error.restype = C.c_char_p
        L.inq_cohort_last_error.argtypes = []
        _BOUND = True
    return L


def outlier(matrix, minsize: int = 10, cutoff: float = 3.0, method: str = "zscore", device: int = 0):
    """Outliers of every row of a rows x cols f32 matrix (outlier.rs:41-71).
    -> (row_kept[rows] u8, rows_of_hits, cols_of_hits, kernel milliseconds); hits sorted by (row, col)."""
    m = np.ascontiguousarray(matrix, dtype=np.float32)
    rows, cols = m.shape
    meth = {"zscore": ZSCORE, "dbscan": DBSCAN}[method]
    kept = np.zeros(rows, np.uint8)
    n = C.c_uint64(0)
    ms = C.c_float(0)
    cap = max(1024, rows // 4)
    L = _lib()
    while True:
        hits = np.zeros(cap, np.uint64)
        rc = L.inq_outlier(device, meth, rows, cols, m.ctypes.data, int(minsize), float(cutoff), kept.ctypes.data,
                           C.byref(n), hits.ctypes.data, cap, C.byref(ms))
        if rc == INQ_ERR_HITS_CAP:
            cap = int(n.value)
            continue
        if rc != INQ_OK:
            raise InqError(rc, L.inq_cohort_last_error().decode())
        h = hits[:int(n.value)]
        return kept, (h >> np.uint64(32)).astype(np.int64), (h & np.uint64(0xFFFFFFFF)).astype(np.int64), float(ms.value)


def assoc(haps, y, cov=None, model: str = "linear", predictor: str = "sum", device: int = 0):
    """Per-row association of STR length with the trait y (include/inqcohort.h inq_assoc).
    haps: rows x 2*samples f64 (H1, H2 of each sample, NaN = no call); y: samples; cov: samples x n_cov or None.
    model: "linear", "logistic" or "firth" (Firth-penalized logistic, stat = penalized likelihood-ratio chi^2).
    -> dict of per-row arrays beta, se, stat, p (f64), n (u32), status (u8, ASSOC_*), n_iter (u8), and ms_kernel."""
    h = np.ascontiguousarray(haps, dtype=np.float64)
    rows, cols = h.shape
    if cols % 2:
        raise ValueError("haps needs two columns per sample")
    ns = cols // 2
    yy = np.ascontiguousarray(y, dtype=np.float64)
    if yy.shape != (ns,):
        raise ValueError("y needs one value per sample")
    c = np.zeros((ns, 0)) if cov is None else np.ascontiguousarray(np.asarray(cov, np.float64).reshape(ns, -1))
    out = {k: np.zeros(rows, np.float64) for k in ("beta", "se", "stat", "p")}
    out["n"] = np.zeros(rows, np.uint32)
    out["status"] = np.zeros(rows, np.uint8)
    out["n_iter"] = np.zeros(rows, np.uint8)
    ms = C.c_float(0)
    L = _lib()
    rc = L.inq_assoc(device, {"linear": LINEAR, "logistic": LOGISTIC, "firth": FIRTH}[model], {"sum": PRED_SUM, "max": PRED_MAX}[predictor],
                     rows, ns, h.ctypes.data, yy.ctypes.data, c.shape[1], c.ctypes.data if c.size else None,
                     out["beta"].ctypes.data, out["se"].ctypes.data, out["stat"].ctypes.data, out["p"].ctypes.data,
                     out["n"].ctypes.data, out["status"].ctypes.data, out["n_iter"].ctypes.data, C.byref(ms))
    if rc != INQ_OK:
        raise InqError(rc, L.inq_cohort_last_error().decode())
    out["ms_kernel"] = float(ms.value)
    return out


def assoc_traits(haps, Y, cov=None, model: str = "linear", predictor: str = "sum", device: int = 0):
    """Per-row association of STR length with each column of Y (include/inqcohort.h inq_assoc_traits).
    Y: samples x T, NaN = the sample is not used for that trait. Column t of every output equals what assoc gives for
    trait t alone over the samples where it is not NaN.
    -> dict of rows x T arrays beta, se, stat, p (f64), n (u32), status (u8), n_iter (u8), and ms_kernel."""
    h = np.ascontiguousarray(haps, dtype=np.float64)
    rows, cols = h.shape
    if cols % 2:
        raise ValueError("haps needs two columns per sample")
    ns = cols // 2
    yy = np.ascontiguousarray(Y, dtype=np.float64)
    if yy.ndim != 2 or yy.shape[0] != ns:
        raise ValueError("Y needs one row per sample")
    nt = yy.shape[1]
    c = np.zeros((ns, 0)) if cov is None else np.ascontiguousarray(np.asarray(cov, np.float64).reshape(ns, -1))
    out = {k: np.zeros((rows, nt), np.float64) for k in ("beta", "se", "stat", "p")}
    out["n"] = np.zeros((rows, nt), np.uint32)
    out["status"] = np.zeros((rows, nt), np.uint8)
    out["n_iter"] = np.zeros((rows, nt), np.uint8)
    ms = C.c_float(0)
    L = _lib()
    rc = L.inq_assoc_traits(device, {"linear": LINEAR, "logistic": LOGISTIC, "firth": FIRTH}[model], {"sum": PRED_SUM, "max": PRED_MAX}[predictor],
                            rows, ns, h.ctypes.data, nt, yy.ctypes.data, c.shape[1], c.ctypes.data if c.size else None,
                            out["beta"].ctypes.data, out["se"].ctypes.data, out["stat"].ctypes.data, out["p"].ctypes.data,
                            out["n"].ctypes.data, out["status"].ctypes.data, out["n_iter"].ctypes.data, C.byref(ms))
    if rc != INQ_OK:
        raise InqError(rc, L.inq_cohort_last_error().decode())
    out["ms_kernel"] = float(ms.value)
    return out


def assoc_cox(haps, time, event, cov=None, ties: str = "efron", predictor: str = "sum", device: int = 0):
    """Per-row Cox proportional-hazards regression of (time, event) on STR length (include/inqcohort.h inq_assoc_cox).
    haps: rows x 2*samples f64 (NaN = no call); time: samples (finite); event: samples, 1 = event, 0 = censored;
    cov: samples x n_cov or None. ties: "efron" or "breslow". stat is the Wald z.
    -> dict of per-row arrays beta, se, stat, p (f64), n (u32), status (u8, ASSOC_*), n_iter (u8), and ms_kernel."""
    h = np.ascontiguousarray(haps, dtype=np.float64)
    rows, cols = h.shape
    if cols % 2:
        raise ValueError("haps needs two columns per sample")
    ns = cols // 2
    t = np.ascontiguousarray(time, dtype=np.float64)
    e = np.asarray(event, dtype=np.float64)
    if t.shape != (ns,) or e.shape != (ns,):
        raise ValueError("time and event need one value per sample")
    ev = np.ascontiguousarray(np.where(e == 0, 0, np.where(e == 1, 1, 2)), dtype=np.uint8)    # 2: rejected by the ABI
    c = np.zeros((ns, 0)) if cov is None else np.ascontiguousarray(np.asarray(cov, np.float64).reshape(ns, -1))
    out = {k: np.zeros(rows, np.float64) for k in ("beta", "se", "stat", "p")}
    out["n"] = np.zeros(rows, np.uint32)
    out["status"] = np.zeros(rows, np.uint8)
    out["n_iter"] = np.zeros(rows, np.uint8)
    ms = C.c_float(0)
    L = _lib()
    rc = L.inq_assoc_cox(device, {"efron": COX_EFRON, "breslow": COX_BRESLOW}[ties], {"sum": PRED_SUM, "max": PRED_MAX}[predictor],
                         rows, ns, h.ctypes.data, t.ctypes.data, ev.ctypes.data, c.shape[1], c.ctypes.data if c.size else None,
                         out["beta"].ctypes.data, out["se"].ctypes.data, out["stat"].ctypes.data, out["p"].ctypes.data,
                         out["n"].ctypes.data, out["status"].ctypes.data, out["n_iter"].ctypes.data, C.byref(ms))
    if rc != INQ_OK:
        raise InqError(rc, L.inq_cohort_last_error().decode())
    out["ms_kernel"] = float(ms.value)
    return out
