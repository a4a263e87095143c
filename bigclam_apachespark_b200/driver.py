"""Host-side mirror of the reference's spark-shell surface for the hot path.

The reference is three flat spark-shell scripts; the names below are the script-level
variables and functions a user of codes/bigclam4-7.scala (and the older v2/v3 scripts) edits
and calls.  Every method that computes goes through the C ABI (libbigclam_b200.so); nothing
here does arithmetic on F.

    script variable / function                     here
    numCore            bigclam4-7.scala:14         BigClam(numCore=...)  (Spark partitions -> unused on one GPU)
    minCom/maxCom/divCom :16-20                    BigClam(minCom, maxCom, divCom), Kset()
    alpha, beta, MaxInter :22-26                   BigClam(alpha, beta, MaxInter)
    GraphLoader.edgeListFile + collectNeighborIds :45,:50   BigClam.load_edge_list / read_edge_list
    conductanceLocalMin() / Sbc :58-75             BigClam.conductanceLocalMin()
    K = sc.broadcast(i); initNeighborComF(K) :249-250       BigClam.initNeighborComF(K)  (or set_K(K); set_F(F0))
    backtrackingLineSearchs(uset) :152             BigClam.backtrackingLineSearchs(uset=None)
    loglikelihood()    bigclamv3-7.scala:106       BigClam.loglikelihood()
    SGDFindC()         bigclam4-7.scala:225        BigClam.SGDFindC()
    MBSGD()            bigclamv3-7.scala:206 / Bigclamv2.scala:203   BigClam.MBSGD(version=3|2)
"""
from __future__ import annotations

import ctypes as C
import math

import numpy as np

from . import _lib
from ._lib import Graph, Params, check


def Kset(minCom: int, maxCom: int, divCom: int, int_division: bool = True) -> list[int]:
    """Geometric grid of K values, bigclam4-7.scala:116-133.

    `maxCom/minCom` is an Int division in the Scala (both are Int vars, :16-18); the pasted REPL
    value at :268 (minCom=50, maxCom=200, divCom=15) is only reproduced with that quirk, so it is
    the default.  int_division=False gives the real-valued ratio the thesis describes.
    """
    ratio = (maxCom // minCom) if int_division else (maxCom / minCom)
    conGap = math.exp(math.log(ratio) / divCom)
    ks = [int(minCom)]
    x = int(minCom)
    while True:
        xtemp = int(x * conGap)
        if xtemp == x:
            xtemp += 1
        x = xtemp
        if x >= maxCom:
            break
        ks.append(x)
    ks.append(int(maxCom))
    return ks


def read_edge_list(path: str, multiplicity: str = "dedup"):
    """GraphLoader.edgeListFile + collectNeighborIds(Either) (bigclam4-7.scala:45,50) via the C++ reader.

    Returns (rowptr int64[n+1], col int32[nnz], ids int64[n]).  multiplicity: "keep" = literal
    GraphX (one neighbour entry per edge line and endpoint), "dedup" = simple undirected graph.
    """
    lib = _lib.load()
    g = Graph()
    err = C.create_string_buffer(512)
    mult = {"keep": 0, "dedup": 1}[multiplicity]
    rc = lib.bigclam_graph_read_edgelist(path.encode(), mult, C.byref(g), err, len(err))
    if rc != _lib.OK:
        raise _lib.BigclamError(rc, err.value.decode())
    try:
        n, nnz = g.n, g.nnz
        rowptr = np.ctypeslib.as_array(g.rowptr, shape=(n + 1,)).copy()
        col = np.ctypeslib.as_array(g.col, shape=(max(nnz, 1),))[:nnz].copy()
        ids = np.ctypeslib.as_array(g.ids, shape=(max(n, 1),))[:n].copy()
    finally:
        lib.bigclam_graph_free(C.byref(g))
    return rowptr, col, ids


class BigClam:
    """One solver instance == the global state of one spark-shell session of the reference."""

    def __init__(self, numCore: int = 36, minCom: int = 1000, maxCom: int = 9000, divCom: int = 100,
                 alpha: float = 0.05, beta: float = 0.1, MaxInter: int = 15, device: int = -1,
                 time_kernels: bool = False, record_accepted: bool = False, verbose: bool = False,
                 sparse_rows: bool = False, numGPUs: int = 1, devices=None, exhaustive_linesearch: bool = False):
        self.numCore, self.minCom, self.maxCom, self.divCom = numCore, minCom, maxCom, divCom
        self.alpha, self.beta, self.MaxInter = alpha, beta, MaxInter
        self.MIN_P_, self.MAX_P_, self.MIN_F_, self.MAX_F_ = 0.0001, 0.9999, 0.0, 1000.0   # :40-43
        self.device = device
        self.flags = (_lib.F_TIME_KERNELS if time_kernels else 0) | (_lib.F_RECORD_ACCEPTED if record_accepted else 0)
        if sparse_rows:       # F as sparse rows on the device (the reference's BSV[Double]); K <= 256, one GPU
            self.flags |= _lib.F_SPARSE_ROWS
        if exhaustive_linesearch:     # evaluate every candidate of every node (no bounds), like the reference's cartesian (:172-181)
            self.flags |= _lib.F_LS_EXHAUSTIVE
        self.verbose = verbose
        self.K = None
        self.rowptr = self.col = self.ids = None
        self._ctx = None
        self._F0 = None
        # numGPUs > 1: all GPUs of the box behind one handle (bigclam_multi_*, sparse rows, fused NVLink collective) —
        # the role `numCore` plays in the script (:14); devices: CUDA ordinals, default 0 .. numGPUs-1
        self.numGPUs = int(numGPUs)
        self.devices = None if devices is None else [int(d) for d in devices]
        self._multi = None
        if self.numGPUs > 1:
            self.flags |= _lib.F_SPARSE_ROWS

    # ---- graph (collectNeighbor / Neightborbc, :50-51) ----
    def load_edge_list(self, path: str, multiplicity: str = "dedup"):
        self.set_graph(*read_edge_list(path, multiplicity))
        return self

    def set_graph(self, rowptr, col, ids=None):
        self._free()
        self.rowptr = np.ascontiguousarray(rowptr, dtype=np.int64)
        self.col = np.ascontiguousarray(col, dtype=np.int32)
        self.ids = ids
        self.Sbc = None
        return self

    @property
    def n(self) -> int:
        return len(self.rowptr) - 1

    # ---- K / F (K = sc.broadcast(i); initNeighborComF(K), :249-250) ----
    def set_K(self, K: int):
        if self.rowptr is None:
            raise ValueError("load a graph first")
        self._free()
        self.K = int(K)
        lib = _lib.load()
        p = Params()
        check(lib.bigclam_default_params(C.byref(p), self.K))
        p.max_inter, p.alpha, p.beta = self.MaxInter, self.alpha, self.beta
        p.min_p, p.max_p, p.min_f, p.max_f = self.MIN_P_, self.MAX_P_, self.MIN_F_, self.MAX_F_
        p.device, p.flags = self.device, self.flags
        ctx = C.c_void_p()
        if self.numGPUs > 1:
            devs = None
            if self.devices is not None:
                devs = (C.c_int32 * self.numGPUs)(*self.devices[:self.numGPUs])
            rc = lib.bigclam_multi_create(C.byref(ctx), self.n, self.rowptr.ctypes.data, self.col.ctypes.data, C.byref(p),
                                          self.numGPUs, devs)
            if rc != _lib.OK:
                raise _lib.BigclamError(rc, (lib.bigclam_multi_last_error(None) or b"").decode())
            self._multi = ctx
            return self
        check(lib.bigclam_create(C.byref(ctx), self.n, self.rowptr.ctypes.data, self.col.ctypes.data, C.byref(p)))
        self._ctx = ctx
        return self

    def _mcheck(self, rc):
        if rc != _lib.OK:
            raise _lib.BigclamError(rc, (_lib.load().bigclam_multi_last_error(self._multi) or b"").decode())

    def set_F_csr(self, indptr, indices, values, K=None, sumF=None):
        """F <- CSR rows (the reference's RDD[(Long, BSV[Double])], :97-104); sumF <- column sums unless given.
        With sparse_rows=True no dense n x K image is built anywhere."""
        indptr = np.ascontiguousarray(indptr, dtype=np.int64)
        indices = np.ascontiguousarray(indices, dtype=np.int32)
        values = np.ascontiguousarray(values, dtype=np.float64)
        if K is not None and (self._ctx is None or int(K) != self.K):
            self.set_K(int(K))
        if len(indptr) != self.n + 1 or len(indices) != indptr[-1] or len(values) != indptr[-1]:
            raise ValueError("CSR arrays do not describe n rows")
        if self._multi is not None:
            self._mcheck(_lib.load().bigclam_multi_set_F_csr(self._multi, indptr.ctypes.data, indices.ctypes.data, values.ctypes.data))
            if sumF is not None:
                sumF = np.ascontiguousarray(sumF, dtype=np.float64)
                self._mcheck(_lib.load().bigclam_multi_set_sumF(self._multi, sumF.ctypes.data))
            return self
        check(_lib.load().bigclam_set_F_csr(self._need(), indptr.ctypes.data, indices.ctypes.data, values.ctypes.data), self._ctx)
        if sumF is not None:
            sumF = np.ascontiguousarray(sumF, dtype=np.float64)
            check(_lib.load().bigclam_set_sumF(self._ctx, sumF.ctypes.data), self._ctx)
        return self

    def F_csr(self):
        """Current F as (indptr, indices, values): ascending indices inside a row, no stored zeros."""
        lib = _lib.load()
        nnz = C.c_int64()
        if self._multi is not None:
            self._mcheck(lib.bigclam_multi_get_F_nnz(self._multi, C.byref(nnz)))
        else:
            check(lib.bigclam_get_F_nnz(self._need(), C.byref(nnz)), self._ctx)
        indptr = np.empty(self.n + 1, dtype=np.int64)
        indices = np.empty(max(nnz.value, 1), dtype=np.int32)
        values = np.empty(max(nnz.value, 1), dtype=np.float64)
        if self._multi is not None:
            self._mcheck(lib.bigclam_multi_get_F_csr(self._multi, indptr.ctypes.data, indices.ctypes.data, values.ctypes.data))
        else:
            check(lib.bigclam_get_F_csr(self._ctx, indptr.ctypes.data, indices.ctypes.data, values.ctypes.data), self._ctx)
        return indptr, indices[:nnz.value], values[:nnz.value]

    def set_F(self, F, sumF=None):
        """F <- n x K (the result of initNeighborComF); sumF <- column sums unless given."""
        if hasattr(F, "tocsr"):                 # scipy.sparse matrix
            m = F.tocsr()
            return self.set_F_csr(m.indptr, m.indices, m.data, K=m.shape[1], sumF=sumF)
        F = np.ascontiguousarray(F, dtype=np.float64)
        if (self._ctx is None and self._multi is None) or F.shape[1] != self.K:
            self.set_K(F.shape[1])
        if F.shape != (self.n, self.K):
            raise ValueError(f"F must be {self.n} x {self.K}")
        if self._multi is not None:
            self._mcheck(_lib.load().bigclam_multi_set_F(self._multi, F.ctypes.data))
            if sumF is not None:
                sumF = np.ascontiguousarray(sumF, dtype=np.float64)
                self._mcheck(_lib.load().bigclam_multi_set_sumF(self._multi, sumF.ctypes.data))
            return self
        check(_lib.load().bigclam_set_F(self._ctx, F.ctypes.data), self._ctx)
        if sumF is not None:
            sumF = np.ascontiguousarray(sumF, dtype=np.float64)
            check(_lib.load().bigclam_set_sumF(self._ctx, sumF.ctypes.data), self._ctx)
        return self

    def replica_F(self, rank: int = 0) -> np.ndarray:
        """numGPUs > 1: the F replica of one rank (all replicas are identical after every call)."""
        out = np.empty((self.n, self.K), dtype=np.float64)
        self._mcheck(_lib.load().bigclam_multi_get_F(self._multi, int(rank), out.ctypes.data))
        return out

    def replica_sumF(self, rank: int = 0) -> np.ndarray:
        out = np.empty(self.K, dtype=np.float64)
        self._mcheck(_lib.load().bigclam_multi_get_sumF(self._multi, int(rank), out.ctypes.data))
        return out

    @property
    def F(self) -> np.ndarray:
        if self._multi is not None:
            return self.replica_F(0)
        out = np.empty((self.n, self.K), dtype=np.float64)
        check(_lib.load().bigclam_get_F(self._need(), out.ctypes.data), self._ctx)
        return out

    @property
    def sumF(self) -> np.ndarray:
        if self._multi is not None:
            return self.replica_sumF(0)
        out = np.empty(self.K, dtype=np.float64)
        check(_lib.load().bigclam_get_sumF(self._need(), out.ctypes.data), self._ctx)
        return out

    # ---- init of F (conductanceLocalMin + initNeighborComF, bigclam4-7.scala:58-108) ----
    def conductanceLocalMin(self, on_gpu=None):
        """Ranked seed candidates (dense vertex indices) and the conductance of every vertex.  on_gpu: True = the
        CUDA kernel (csrc/initf_gpu.cu), False = the host path, None = the GPU when there is one."""
        lib = _lib.load()
        cond = np.empty(self.n, dtype=np.float64)
        seeds = np.empty(self.n, dtype=np.int32)
        cnt = C.c_int64()
        if on_gpu is None:
            on_gpu = lib.bigclam_device_count() > 0
        if on_gpu:
            rc = lib.bigclam_conductance_seeds_gpu(self.n, self.rowptr.ctypes.data, self.col.ctypes.data, self.device,
                                                   cond.ctypes.data, seeds.ctypes.data, C.byref(cnt))
        else:
            rc = lib.bigclam_conductance_seeds(self.n, self.rowptr.ctypes.data, self.col.ctypes.data, cond.ctypes.data,
                                               seeds.ctypes.data, C.byref(cnt))
        if rc != _lib.OK:
            raise _lib.BigclamError(rc, "bigclam_conductance_seeds failed")
        self.Sbc = seeds[:cnt.value].copy()             # `Sbc` of the script (:75), reused for every K
        self.conductance = cond
        return self.Sbc

    def initNeighborComF(self, K: int, include_self: bool = False, pad_seed: int = 1234):
        """Builds F0 from the ranked seeds and loads it (sets F and sumF like the script, :105-107)."""
        if getattr(self, "Sbc", None) is None:
            self.conductanceLocalMin()
        F0 = np.empty((self.n, int(K)), dtype=np.float64)
        rc = _lib.load().bigclam_init_neighbor_com_F(self.n, self.rowptr.ctypes.data, self.col.ctypes.data, int(K),
                                                     self.Sbc.ctypes.data, len(self.Sbc), 1 if include_self else 0,
                                                     C.c_uint64(pad_seed), F0.ctypes.data)
        if rc != _lib.OK:
            raise _lib.BigclamError(rc, "bigclam_init_neighbor_com_F failed")
        self.set_F(F0)
        return F0

    # ---- the hot path ----
    def backtrackingLineSearchs(self, uset=None) -> float:
        """bigclam4-7.scala:152-223.  uset: None = all vertices (as the reference always passes),
        else an iterable of dense vertex indices."""
        mask_ptr = None
        if uset is not None:
            mask = np.zeros(self.n, dtype=np.uint8)
            mask[np.asarray(list(uset), dtype=np.int64)] = 1
            mask_ptr = mask.ctypes.data
        llh = C.c_double()
        nupd = C.c_int64()
        if self._multi is not None:
            self._mcheck(_lib.load().bigclam_multi_step(self._multi, mask_ptr, C.byref(llh), C.byref(nupd)))
        else:
            check(_lib.load().bigclam_step(self._need(), mask_ptr, C.byref(llh), C.byref(nupd)), self._ctx)
        self.last_n_updated = nupd.value
        return llh.value

    def loglikelihood(self) -> float:
        """bigclamv3-7.scala:106-120 / Bigclamv2.scala:187-200."""
        llh = C.c_double()
        if self._multi is not None:
            self._mcheck(_lib.load().bigclam_multi_loglikelihood(self._multi, C.byref(llh)))
        else:
            check(_lib.load().bigclam_loglikelihood(self._need(), C.byref(llh)), self._ctx)
        return llh.value

    def _run(self, variant: int, rel_tol: float, max_outer: int, trace_cap: int = 65536):
        trace = np.full(trace_cap, np.nan)
        llh = C.c_double()
        calls = C.c_int64()
        if self._multi is not None:
            self._mcheck(_lib.load().bigclam_multi_run(self._multi, variant, rel_tol, max_outer, C.byref(llh), C.byref(calls),
                                                       trace.ctypes.data, trace_cap))
        else:
            check(_lib.load().bigclam_run(self._need(), variant, rel_tol, max_outer, C.byref(llh), C.byref(calls),
                                          trace.ctypes.data, trace_cap), self._ctx)
        self.last_calls = calls.value
        self.last_trace = trace[:min(calls.value, trace_cap)]
        return llh.value

    def SGDFindC(self, rel_tol: float = 0.0001, max_outer: int = 0) -> float:
        """bigclam4-7.scala:225-243: one call for LLHold, then loop until |1 - new/old| < 1e-4;
        returns LLHold.  max_outer=0: no iteration cap, like the reference."""
        ret = self._run(4, rel_tol, max_outer)
        if self.verbose:
            for i, v in enumerate(self.last_trace[1:], start=1):
                print("-------Inter: " + str(i) + " LLH: " + repr(float(v)))          # :236
        return ret

    def MBSGD(self, version: int = 3, rel_tol: float = 0.0001, max_outer: int = 0) -> None:
        """bigclamv3-7.scala:206-222 (LLHold = 0.0) or Bigclamv2.scala:203-219 (LLHold = loglikelihood())."""
        if version not in (2, 3):
            raise ValueError("version must be 2 or 3")
        if self.verbose:
            print("LLH: " + repr(0.0 if version == 3 else self.loglikelihood()))       # v3 :208 / v2 :205
        self._run(version, rel_tol, max_outer)
        if self.verbose:
            for i, v in enumerate(self.last_trace, start=1):
                print(" Inter: " + str(i * self.n) + " LLH: " + repr(float(v)))         # v3 :216 (i += uset.size)

    def Kset(self) -> list[int]:
        return Kset(self.minCom, self.maxCom, self.divCom)

    def sweep_K(self, rel_gain: float = 0.001, max_outer: int = 0):
        """The K sweep at the bottom of the script (bigclam4-7.scala:244-266): for K in Kset, initNeighborComF(K),
        SGDFindC(); stop at the first K whose LLH gain over the previous K is below 0.1 % (`1 - new/old < 0.001`).
        As coded, LLHKold starts at 0.0 (the `== null` test is never true for a Double), so the first K never
        stops the sweep.  Returns (KforC, [(K, LLH), ...]); KforC is 0 when the sweep ran out of K values (:245)."""
        LLHKold, KforC, hist = 0.0, 0, []
        for i in self.Kset():
            self.initNeighborComF(i)
            LLHKnew = self.SGDFindC(max_outer=max_outer)
            if self.verbose:
                print(str(i) + " LLH: " + repr(LLHKnew))                                   # :258
            hist.append((i, LLHKnew))
            with np.errstate(divide="ignore", invalid="ignore"):
                gain = 1.0 - np.float64(LLHKnew) / np.float64(LLHKold)
            if gain < rel_gain:                                                          # :259
                KforC = i
                break
            LLHKold = LLHKnew
        return KforC, hist

    # ---- K by held-out likelihood (the thesis p.20; holdout.py, DESIGN.md (f) f-5) ----
    def set_holdout(self, ho_rowptr, ho_col, ho_is_edge):
        """Held-out pairs of the current context (sparse rows, one GPU): from now on the steps, SGDFindC and
        loglikelihood() use the masked objective, which leaves every held-out pair out.  Symmetric lists, disjoint from
        the neighbour lists; ho_is_edge = 1 for a held-out edge, 0 for a held-out non-edge (holdout.split_pairs makes
        them).  The lists belong to the context: set_K() or a new graph drops them."""
        if self._multi is not None:
            raise RuntimeError("held-out pairs are single-GPU only (numGPUs = 1)")
        rp = np.ascontiguousarray(ho_rowptr, dtype=np.int64)
        hc = np.ascontiguousarray(ho_col, dtype=np.int32)
        he = np.ascontiguousarray(ho_is_edge, dtype=np.uint8)
        if len(rp) != self.n + 1 or len(hc) != rp[-1] or len(he) != rp[-1]:
            raise ValueError("held-out CSR arrays do not describe n rows")
        check(_lib.load().bigclam_set_holdout(self._need(), rp.ctypes.data, hc.ctypes.data, he.ctypes.data), self._ctx)
        return self

    def clear_holdout(self):
        """Back to the unmasked objective (exactly as if no held-out pairs had been set)."""
        if self._ctx is not None:
            check(_lib.load().bigclam_set_holdout(self._ctx, None, None, None), self._ctx)
        return self

    def holdout_loglikelihood(self) -> float:
        """Log-likelihood of the held-out pairs under the current F: sum of log(1 - p) over held-out edges plus sum of
        log(p) over held-out non-edges, p = clamp(exp(-Fu.Fv)), each pair once.  Sets last_holdout_pairs."""
        llh = C.c_double()
        npairs = C.c_int64()
        check(_lib.load().bigclam_holdout_loglikelihood(self._need(), C.byref(llh), C.byref(npairs)), self._ctx)
        self.last_holdout_pairs = npairs.value
        return llh.value

    def select_K(self, Ks=None, ho_frac: float = 0.2, repeats: int = 3, seed: int = 0, max_outer: int = 0, refit: bool = True):
        """Chooses K by held-out likelihood.  For every K (default: Kset()) and repeat r the graph is split with seed
        seed + r (holdout.split_pairs: ho_frac of the edges and as many non-edges); on the TRAINING graph
        conductanceLocalMin(), initNeighborComF(K), set_holdout and SGDFindC(max_outer) run, then the held-out pairs are
        scored.  K_best has the highest mean over the repeats (ties: the smaller K).  Returns (K_best, rows), rows =
        [(K, mean, [value per repeat], [SGDFindC calls per repeat]), ...].  Sparse rows are used whatever the constructor
        flags.  With refit the solver is left on the full graph at K_best, fitted by SGDFindC(max_outer) with the
        constructor's flags and ready for communities.extract; otherwise it is left on the full graph with no context."""
        from .holdout import split_pairs
        if self.numGPUs > 1:
            raise ValueError("select_K runs on one GPU (numGPUs = 1)")
        if self.rowptr is None:
            raise ValueError("load a graph first")
        if repeats < 1:
            raise ValueError("repeats must be >= 1")
        Ks = [int(k) for k in (self.Kset() if Ks is None else Ks)]
        full = (self.rowptr, self.col, self.ids)
        flags = self.flags
        splits = [split_pairs(full[0], full[1], ho_frac, seed + r) for r in range(repeats)]
        seeds = [None] * repeats
        rows = []
        try:
            self.flags = flags | _lib.F_SPARSE_ROWS
            for K in Ks:
                vals, calls = [], []
                for r, sp in enumerate(splits):
                    self.set_graph(sp.rowptr, sp.col, full[2])
                    if seeds[r] is None:
                        seeds[r] = self.conductanceLocalMin()
                    self.Sbc = seeds[r]
                    self.initNeighborComF(K)
                    self.set_holdout(sp.ho_rowptr, sp.ho_col, sp.ho_is_edge)
                    self.SGDFindC(max_outer=max_outer)
                    vals.append(self.holdout_loglikelihood())
                    calls.append(self.last_calls)
                    if self.verbose:
                        print(str(K) + " repeat " + str(r) + " held-out LLH: " + repr(vals[-1]))
                rows.append((K, float(np.mean(vals)), vals, calls))
        finally:
            self.flags = flags
            self.set_graph(*full)
        K_best = max(rows, key=lambda row: (row[1], -row[0]))[0]
        if refit:
            self.conductanceLocalMin()
            self.initNeighborComF(K_best)
            self.SGDFindC(max_outer=max_outer)
        return K_best, rows

    # ---- diagnostics ----
    def accepted(self) -> np.ndarray:
        out = np.empty(self.n, dtype=np.int8)
        check(_lib.load().bigclam_get_accepted(self._need(), out.ctypes.data), self._ctx)
        return out

    def kernel_time(self):
        ms = C.c_double()
        nstep = C.c_int64()
        nall = C.c_int64()
        if self._multi is not None:          # slowest rank's sum of step-kernel times
            self._mcheck(_lib.load().bigclam_multi_get_kernel_time(self._multi, C.byref(ms), C.byref(nstep)))
            return ms.value, nstep.value, nstep.value
        check(_lib.load().bigclam_get_kernel_time(self._need(), C.byref(ms), C.byref(nstep), C.byref(nall)), self._ctx)
        return ms.value, nstep.value, nall.value

    def retile(self):
        """Sparse rows: re-cut the tiles of small nodes for the rows' current size / the observed fallback rate
        (bigclam_run does this between its batches of 8 calls)."""
        if self._multi is None:
            check(_lib.load().bigclam_retile(self._need()), self._ctx)

    def tile_stats(self):
        """Sparse rows + time_kernels: dict(tiles_done, tiles_fallback, n_tiles, n_general_nodes, n_split_hubs)."""
        if self._multi is not None:
            raise RuntimeError("tile_stats() reads one context; with numGPUs > 1 use ls_stats() (summed over the ranks)")
        v = [C.c_int64() for _ in range(5)]
        check(_lib.load().bigclam_get_tile_stats(self._need(), *[C.byref(x) for x in v]), self._ctx)
        return dict(zip(("tiles_done", "tiles_fallback", "n_tiles", "n_general_nodes", "n_split_hubs"), (x.value for x in v)))

    def ls_stats(self):
        """Sparse rows: dict(nodes_asked, nodes_searched) of the tile path since the previous read — how many of the
        nodes that asked for a line search had a candidate the bounds could not exclude."""
        a, b = C.c_int64(), C.c_int64()
        if self._multi is not None:          # summed over the ranks (every rank counts the nodes it owns)
            self._mcheck(_lib.load().bigclam_multi_get_ls_stats(self._multi, C.byref(a), C.byref(b)))
            return {"nodes_asked": a.value, "nodes_searched": b.value}
        check(_lib.load().bigclam_get_ls_stats(self._need(), C.byref(a), C.byref(b)), self._ctx)
        return {"nodes_asked": a.value, "nodes_searched": b.value}

    def set_stream(self, cuda_stream: int):
        check(_lib.load().bigclam_set_stream(self._need(), C.c_void_p(cuda_stream)), self._ctx)

    def device_state(self):
        f, fn, sf = C.c_void_p(), C.c_void_p(), C.c_void_p()
        ld = C.c_int64()
        check(_lib.load().bigclam_device_state(self._need(), C.byref(f), C.byref(fn), C.byref(sf), C.byref(ld)), self._ctx)
        return f.value, fn.value, sf.value, ld.value

    def _need(self):
        if self._ctx is None:
            raise RuntimeError("no context: call set_K()/set_F() after loading a graph")
        return self._ctx

    def _free(self):
        if self._ctx is not None:
            _lib.load().bigclam_destroy(self._ctx)
            self._ctx = None
        if getattr(self, "_multi", None) is not None:
            _lib.load().bigclam_multi_destroy(self._multi)
            self._multi = None

    def close(self):
        self._free()

    def __del__(self):
        try:
            self._free()
        except Exception:
            pass
