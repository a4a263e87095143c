"""ctypes front-end of the masked-step oracle (holdout_oracle.c) and its independent NumPy twin.

TEST INFRASTRUCTURE ONLY.  The library is compiled on first use with the flags of oracle/Makefile into a per-user
temporary directory (keyed by the source and the host CPU), so the repository tree is never written.  OracleParams and
make_params are oracle/oracle.py's: the struct is the same.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np

from oracle.oracle import OracleParams, _cpu_tag, make_params  # noqa: F401  (re-exported)

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "holdout_oracle.c")
_CFLAGS = ["-O3", "-march=native", "-fPIC", "-fopenmp", "-ffp-contract=off", "-fno-fast-math", "-Wall", "-Wextra", "-std=c11"]


def build() -> str:
    """Compile libholdout_oracle.so (gcc + OpenMP, the flags of oracle/Makefile); returns its path."""
    with open(_SRC, "rb") as fh:
        key = hashlib.sha1(fh.read() + " ".join(_CFLAGS).encode() + _cpu_tag().encode()).hexdigest()[:16]
    d = os.path.join(tempfile.gettempdir(), f"bigclam_holdout_oracle-{os.getuid()}-{key}")
    path = os.path.join(d, "libholdout_oracle.so")
    if not os.path.exists(path):
        os.makedirs(d, exist_ok=True)
        cc = "/usr/bin/gcc" if os.access("/usr/bin/gcc", os.X_OK) else "gcc"
        tmp = f"{path}.{os.getpid()}"
        subprocess.run([cc, *_CFLAGS, "-shared", "-o", tmp, _SRC, "-lm"], check=True)
        os.replace(tmp, path)
    return path


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        L = C.CDLL(build())
        vp, i64, P = C.c_void_p, C.c_int64, C.POINTER(OracleParams)
        L.oracle_step_masked.argtypes = [i64, vp, vp, vp, vp, P, vp, vp, vp, vp, C.POINTER(i64), vp, vp, C.c_int32, vp, vp]
        L.oracle_step_masked.restype = C.c_double
        L.oracle_llh_masked.argtypes = [i64, vp, vp, vp, vp, P, vp, vp, vp]
        L.oracle_llh_masked.restype = C.c_double
        L.oracle_armijo_margins_masked.argtypes = [i64, vp, vp, vp, vp, P, vp, vp, vp, i64, vp, vp]
        L.oracle_armijo_margins_masked.restype = None
        L.oracle_run_masked.argtypes = [i64, vp, vp, vp, vp, P, vp, vp, C.c_double, i64, C.POINTER(C.c_double), vp, i64]
        L.oracle_run_masked.restype = C.c_int64
        L.oracle_holdout_llh.argtypes = [i64, vp, vp, vp, P, vp, C.POINTER(i64)]
        L.oracle_holdout_llh.restype = C.c_double
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def _lists(rowptr, col, ho_rowptr, ho_col, F, k):
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
    col = np.ascontiguousarray(col, dtype=np.int32)
    ho_rowptr = np.ascontiguousarray(ho_rowptr, dtype=np.int64)
    ho_col = np.ascontiguousarray(ho_col, dtype=np.int32)
    n = len(rowptr) - 1
    assert len(ho_rowptr) == n + 1 and len(ho_col) == ho_rowptr[-1]
    if F is not None:
        assert F.dtype == np.float64 and F.flags.c_contiguous and F.shape == (n, k), (F.shape, n, k)
    return n, rowptr, col, ho_rowptr, ho_col


@dataclass
class StepResult:
    F: np.ndarray
    sumF: np.ndarray
    llh: float
    n_updated: int
    accepted: np.ndarray
    trials: np.ndarray
    grad: np.ndarray | None
    llh_u: np.ndarray | None


def step(rowptr, col, ho_rowptr, ho_col, F, sumF, params: OracleParams, node_mask=None, early_exit=True, want_pre=False) -> StepResult:
    """One masked backtrackingLineSearchs call on (F, sumF); inputs are not modified."""
    n, rowptr, col, ho_rowptr, ho_col = _lists(rowptr, col, ho_rowptr, ho_col, F, params.k)
    k = params.k
    sumF2 = np.array(sumF, dtype=np.float64, copy=True)
    Fo = np.empty_like(F)
    acc = np.empty(n, dtype=np.int8)
    tr = np.empty(n, dtype=np.int8)
    grad = np.empty((n, k)) if want_pre else None
    llh_u = np.empty(n) if want_pre else None
    if node_mask is not None:
        node_mask = np.ascontiguousarray(node_mask, dtype=np.uint8)
    nupd = C.c_int64(0)
    v = lib().oracle_step_masked(n, _p(rowptr), _p(col), _p(ho_rowptr), _p(ho_col), C.byref(params), _p(F), _p(sumF2),
                                 _p(node_mask), _p(Fo), C.byref(nupd), _p(acc), _p(tr), 1 if early_exit else 0, _p(grad), _p(llh_u))
    return StepResult(Fo, sumF2, v, nupd.value, acc, tr, grad, llh_u)


def llh(rowptr, col, ho_rowptr, ho_col, F, sumF, params: OracleParams, per_node=False):
    n, rowptr, col, ho_rowptr, ho_col = _lists(rowptr, col, ho_rowptr, ho_col, F, params.k)
    sumF = np.ascontiguousarray(sumF, dtype=np.float64)
    pn = np.empty(n) if per_node else None
    v = lib().oracle_llh_masked(n, _p(rowptr), _p(col), _p(ho_rowptr), _p(ho_col), C.byref(params), _p(F), _p(sumF), _p(pn))
    return (v, pn) if per_node else v


def armijo_margins(rowptr, col, ho_rowptr, ho_col, F, sumF, params: OracleParams, nodes):
    n, rowptr, col, ho_rowptr, ho_col = _lists(rowptr, col, ho_rowptr, ho_col, F, params.k)
    nodes = np.ascontiguousarray(nodes, dtype=np.int64)
    m = np.empty((len(nodes), params.max_inter + 1))
    lu = np.empty(len(nodes))
    sumF = np.ascontiguousarray(sumF, dtype=np.float64)
    lib().oracle_armijo_margins_masked(n, _p(rowptr), _p(col), _p(ho_rowptr), _p(ho_col), C.byref(params), _p(F), _p(sumF),
                                       _p(nodes), len(nodes), _p(m), _p(lu))
    return m, lu


def run(rowptr, col, ho_rowptr, ho_col, F, sumF, params: OracleParams, rel_tol=1e-4, max_outer=0, trace_cap=4096):
    """SGDFindC on the masked objective.  Returns (F, sumF, llh, calls, trace)."""
    n, rowptr, col, ho_rowptr, ho_col = _lists(rowptr, col, ho_rowptr, ho_col, F, params.k)
    F2 = np.array(F, copy=True)
    s2 = np.array(sumF, dtype=np.float64, copy=True)
    trace = np.full(trace_cap, np.nan)
    out = C.c_double(0.0)
    calls = lib().oracle_run_masked(n, _p(rowptr), _p(col), _p(ho_rowptr), _p(ho_col), C.byref(params), _p(F2), _p(s2),
                                    rel_tol, max_outer, C.byref(out), _p(trace), trace_cap)
    return F2, s2, out.value, calls, trace[:min(calls, trace_cap)]


def holdout_llh(ho_rowptr, ho_col, ho_is_edge, F, params: OracleParams):
    """(L_HO, number of unordered pairs scored)."""
    ho_rowptr = np.ascontiguousarray(ho_rowptr, dtype=np.int64)
    ho_col = np.ascontiguousarray(ho_col, dtype=np.int32)
    ho_is_edge = np.ascontiguousarray(ho_is_edge, dtype=np.uint8)
    F = np.ascontiguousarray(F, dtype=np.float64)
    npairs = C.c_int64(0)
    v = lib().oracle_holdout_llh(len(ho_rowptr) - 1, _p(ho_rowptr), _p(ho_col), _p(ho_is_edge), C.byref(params), _p(F), C.byref(npairs))
    return v, npairs.value


# --------------------------------------------------------------------------------------------------------------------
# NumPy twin, written from the formulas (DESIGN.md (f) f-5), not from the C: vectorised per node, NumPy's summation
# order, so it agrees with the C restatement to reassociation noise.  Small graphs only.
MIN_P_, MAX_P_, MIN_F_, MAX_F_ = 0.0001, 0.9999, 0.0, 1000.0


def _terms(x):
    p = np.minimum(np.maximum(np.exp(-x), MIN_P_), MAX_P_)
    return np.log(1.0 - p) + x, p


def twin_llh(rowptr, col, ho_rowptr, ho_col, F, sumF):
    total = 0.0
    for u in range(len(rowptr) - 1):
        fu = F[u]
        nb, ho = col[rowptr[u]:rowptr[u + 1]], ho_col[ho_rowptr[u]:ho_rowptr[u + 1]]
        t, _ = _terms(F[nb] @ fu)
        total += t.sum() + (F[ho] @ fu).sum() - fu @ sumF + fu @ fu
    return total


def twin_step(rowptr, col, ho_rowptr, ho_col, F, sumF, alpha=0.05, beta=0.1, max_inter=15):
    """Returns (F_new, sumF_new, LLH, accepted index per node, -1 = kept)."""
    n = F.shape[0]
    steps = beta ** np.arange(max_inter + 1)
    F_new = F.copy()
    accepted = np.full(n, -1, dtype=np.int8)
    changed = np.zeros(n, dtype=bool)
    for u in range(n):
        nb, ho = col[rowptr[u]:rowptr[u + 1]], ho_col[ho_rowptr[u]:ho_rowptr[u + 1]]
        if len(nb) == 0:
            continue
        fu, FV, FH = F[u], F[nb], F[ho]
        t, p = _terms(FV @ fu)
        grad = (FV / (1.0 - p)[:, None]).sum(axis=0) + FH.sum(axis=0) - sumF + fu
        llh_u = t.sum() + (FH @ fu).sum() - fu @ sumF + fu @ fu
        for j, s in enumerate(steps):
            nf = np.minimum(np.maximum(fu + s * grad, MIN_F_), MAX_F_)
            tt, _ = _terms(FV @ nf)
            res = tt.sum() + (FH @ nf).sum() - nf @ (sumF - fu + nf) + nf @ nf
            if res >= llh_u + alpha * s * (grad @ grad):
                accepted[u] = j
                F_new[u] = nf
                changed[u] = True
                break
    sumF_new = sumF - (F[changed].sum(axis=0) - F_new[changed].sum(axis=0)) if changed.any() else sumF.copy()
    return F_new, sumF_new, twin_llh(rowptr, col, ho_rowptr, ho_col, F_new, sumF_new), accepted
